#!/usr/bin/env python
"""Generates tests/golden/lz4/vectors.json: for every input of test_oracle_codec._corpus, the length and SHA-256 of what the LZ4 C library
(liblz4, LZ4_compress_default: the block compressor lz4-java's LZ4Compressor matches) produced for it. The corpus is regenerated from its
seed by the test, so the digests pin the oracle's LZ4 bytes to the library without the library installed. Run where liblz4 is installed;
the JSON is committed."""
import ctypes as C, hashlib, json, os, random, sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from test_oracle_codec import _corpus, _liblz4

L = _liblz4()
L.LZ4_versionString.restype = C.c_char_p; L.LZ4_compressBound.argtypes = [C.c_int]; L.LZ4_compressBound.restype = C.c_int
out = {"library": "liblz4 %s, LZ4_compress_default" % L.LZ4_versionString().decode(), "vectors": []}
for s in _corpus(random.Random(0xCA55)):
    cap = L.LZ4_compressBound(len(s)); buf = C.create_string_buffer(cap + 1)
    n = L.LZ4_compress_default(s, buf, len(s), cap); assert n > 0 or not s
    out["vectors"].append({"n": len(s), "compressed_len": n, "sha256": hashlib.sha256(buf.raw[:n]).hexdigest()})
dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "lz4", "vectors.json")
json.dump(out, open(dst, "w"), indent=0)
print("wrote %d vectors, %d bytes" % (len(out["vectors"]), os.path.getsize(dst)))
