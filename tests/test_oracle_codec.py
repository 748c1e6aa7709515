"""Pins the CPU oracle's codecs against (1) the reference's golden SSTables, (2) zlib, (3) liblz4 (stored digests, and liblz4.so.1 live).
SURVEY §8c: compressed bytes are pinned only by the golden files; CRC32 by Data.db inline checksums + Digest.crc32."""
import ctypes as C, hashlib, json, os, random, struct, zlib, pytest
import oracle_lib as O
from sstable_files import read_compression_info, split_chunks, find_tables

def _liblz4():
    for n in ("liblz4.so.1", "liblz4.so"):
        try:
            L = C.CDLL(n)
            L.LZ4_compress_default.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int]; L.LZ4_compress_default.restype = C.c_int
            return L
        except OSError:
            pass
    return None

def test_golden_chunks_crc_and_lz4(golden_dir):
    tables = find_tables(golden_dir)
    assert len(tables) >= 60
    nchunks = 0
    for base in tables:
        info = read_compression_info(base + "CompressionInfo.db")
        assert info["compressor"] == "LZ4Compressor"
        data = open(base + "Data.db", "rb").read()
        # Digest.crc32 = decimal CRC32 of the whole Data.db (chunks and inline CRCs): ChecksumWriter.java:62-104
        assert int(open(base + "Digest.crc32").read()) == O.crc32(data) == zlib.crc32(data)
        total = 0
        for comp, crc, ulen in split_chunks(data, info):
            assert O.crc32(comp) == crc                      # per-chunk CRC32 over the bytes as written
            (plen,) = struct.unpack_from("<I", comp, 0)      # LZ4Compressor 4-byte LE length prefix
            assert plen == ulen
            raw = O.chunk_decompress(O.COMP_LZ4, comp, ulen)
            assert len(raw) == ulen
            assert O.chunk_compress(O.COMP_LZ4, raw) == comp   # bit-exact recompression of what a real release wrote
            total += ulen; nchunks += 1
        assert total == info["data_length"]
    assert nchunks >= 280

def _corpus(rng):
    out = [b"", b"a", b"abcdefghijkl", b"abcdefghijklm", b"a" * 13, b"\x00" * 16384, bytes(range(256)) * 64]
    for n in (1, 5, 12, 13, 14, 64, 100, 1000, 4096, 16383, 16384, 16385, 40000, 65536, 65546):
        out.append(bytes(rng.getrandbits(8) for _ in range(n)))                        # incompressible
        out.append(bytes(rng.choice(b"abcd") for _ in range(n)))                       # tiny alphabet
        words = [bytes(rng.getrandbits(8) for _ in range(rng.randint(3, 24))) for _ in range(40)]
        s = b"".join(rng.choice(words) for _ in range(n // 8 + 1))[:n]; out.append(s)   # dictionary-like
        mixed = bytearray()
        while len(mixed) < n:
            if rng.random() < 0.5: mixed += bytes(rng.getrandbits(8) for _ in range(rng.randint(1, 300)))
            else: mixed += bytes([rng.getrandbits(8)]) * rng.randint(1, 700)
        out.append(bytes(mixed[:n]))
        # sstable-like: 8-byte BE counters + small vints
        rows = bytearray(); x = rng.getrandbits(40)
        while len(rows) < n:
            x += rng.randint(1, 1000); rows += b"\x24" + struct.pack(">q", x) + bytes([rng.randint(0, 20), 4, rng.randint(0, 255)]) + struct.pack(">q", rng.getrandbits(20))
        out.append(bytes(rows[:n]))
    return out

def test_lz4_matches_system_liblz4():
    # liblz4's output for the corpus is pinned by tests/golden/lz4/vectors.json (tests/golden/tools/make_lz4_vectors.py); where the library
    # is installed, its live output is compared as well
    want = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lz4", "vectors.json")))["vectors"]
    corpus = _corpus(random.Random(0xCA55))
    assert len(want) == len(corpus)
    L = _liblz4()
    for s, w in zip(corpus, want):
        c = O.lz4_compress(s)
        assert (len(s), len(c), hashlib.sha256(c).hexdigest()) == (w["n"], w["compressed_len"], w["sha256"])
        assert O.lz4_decompress(c, len(s)) == s
        if L is not None:
            cap = O.lib().orc_lz4_compress_bound(len(s)); buf = C.create_string_buffer(cap + 1)
            n = L.LZ4_compress_default(s, buf, len(s), cap)
            assert c == buf.raw[:n], len(s)

def test_lz4_rejects_malformed():
    s = bytes(random.Random(1).getrandbits(8) for _ in range(500)) + b"x" * 500
    c = O.lz4_compress(s)
    with pytest.raises(ValueError): O.lz4_decompress(c[:-3], len(s))
    with pytest.raises(ValueError): O.lz4_decompress(c, len(s) - 1)
    with pytest.raises(ValueError): O.lz4_decompress(b"\x10\x41\x05\x00", 50)   # offset beyond start

def test_crc32_matches_zlib_and_combine():
    rng = random.Random(7)
    for n in (0, 1, 3, 7, 8, 9, 63, 64, 1000, 16388, 70000):
        a = bytes(rng.getrandbits(8) for _ in range(n)); b = bytes(rng.getrandbits(8) for _ in range(n // 2 + 1))
        assert O.crc32(a) == zlib.crc32(a)
        assert O.crc32(b, O.crc32(a)) == zlib.crc32(a + b)
        assert O.lib().orc_crc32_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(a + b)

def test_vint_boundaries():
    # T/utils/vint/VIntCodingTest.java: size boundaries at 7*n bits; 9-byte form is 0xFF + 8 raw bytes
    L = O.lib()
    for bits in range(0, 64):
        for v in ((1 << bits) - 1, 1 << bits, (1 << bits) + 1):
            v &= (1 << 64) - 1
            enc = O.vint(v)
            expect = 1 if v < 128 else min(9, (v.bit_length() + 6) // 7)
            assert len(enc) == L.orc_vint_size(v) == expect, (v, enc)
            out = C.c_uint64(); assert L.orc_vint_read(enc, len(enc), C.byref(out)) == len(enc) and out.value == v
    assert O.vint(0) == b"\x00" and O.vint(127) == b"\x7f" and O.vint(128) == b"\x80\x80" and O.vint(16383) == b"\xbf\xff"
    assert O.vint((1 << 64) - 1) == b"\xff" * 9
    assert O.vint(1 << 56) == b"\xff\x01" + b"\x00" * 7

def _ref_murmur3_x64_128(key: bytes, seed=0):
    """Independent pure-Python restatement of S/utils/MurmurHash.java:178-260 incl. the signed tail bytes."""
    M = (1 << 64) - 1
    rotl = lambda v, n: ((v << n) | (v >> (64 - n))) & M
    def fmix(k):
        k ^= k >> 33; k = k * 0xff51afd7ed558ccd & M; k ^= k >> 33; k = k * 0xc4ceb9fe1a85ec53 & M; k ^= k >> 33; return k
    c1, c2 = 0x87c37b91114253d5, 0x4cf5ad432745937f
    h1 = h2 = seed; n = len(key); nb = n >> 4
    for i in range(nb):
        k1 = int.from_bytes(key[16 * i:16 * i + 8], "little"); k2 = int.from_bytes(key[16 * i + 8:16 * i + 16], "little")
        k1 = k1 * c1 & M; k1 = rotl(k1, 31); k1 = k1 * c2 & M; h1 ^= k1
        h1 = rotl(h1, 27); h1 = (h1 + h2) & M; h1 = (h1 * 5 + 0x52dce729) & M
        k2 = k2 * c2 & M; k2 = rotl(k2, 33); k2 = k2 * c1 & M; h2 ^= k2
        h2 = rotl(h2, 31); h2 = (h2 + h1) & M; h2 = (h2 * 5 + 0x38495ab5) & M
    t = key[nb * 16:]; k1 = k2 = 0
    sb = lambda i: (t[i] - 256 if t[i] >= 128 else t[i]) & M
    r = n & 15
    for i in range(r - 1, 7, -1): k2 ^= (sb(i) << (8 * (i - 8))) & M
    if r > 8: k2 = k2 * c2 & M; k2 = rotl(k2, 33); k2 = k2 * c1 & M; h2 ^= k2
    for i in range(min(r, 8) - 1, -1, -1): k1 ^= (sb(i) << (8 * i)) & M
    if r > 0: k1 = k1 * c1 & M; k1 = rotl(k1, 31); k1 = k1 * c2 & M; h1 ^= k1
    h1 ^= n; h2 ^= n; h1 = (h1 + h2) & M; h2 = (h2 + h1) & M
    h1 = fmix(h1); h2 = fmix(h2); h1 = (h1 + h2) & M; h2 = (h2 + h1) & M
    return h1, h2

def test_murmur3_token():
    rng = random.Random(3)
    assert O.token(b"") == -(1 << 63)
    for n in list(range(0, 40)) + [100, 255]:
        for _ in range(4):
            k = bytes(rng.getrandbits(8) for _ in range(n))
            if not k: continue
            h1, _ = _ref_murmur3_x64_128(k)
            t = h1 - (1 << 64) if h1 >= (1 << 63) else h1
            if t == -(1 << 63): t = (1 << 63) - 1
            assert O.token(k) == t
    # golden order: Index.db of legacy_oa_simple lists keys in token order; pinned further in test_oracle_sstable.py

def test_snappy_roundtrip_format():
    # PARITY UNPINNED for compressed bytes (no snappy golden / lib); the raw format itself is checked by round trip.
    rng = random.Random(5)
    for s in _corpus(rng):
        c = O.chunk_compress(O.COMP_SNAPPY, s)
        assert O.chunk_decompress(O.COMP_SNAPPY, c, len(s)) == s
