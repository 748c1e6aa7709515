"""Cost of the per-file side band (Filter.db, Summary.db, first / last key, Statistics) of a leveled compaction on the GPU.

Builds bench.py's configs[2] inputs (32 Snappy SSTables x 160 MiB, 160 MiB outputs) and, in one process on one GPU, times b200c_compact
with and without the side band, alternating call by call, for device-resident and host buffers, with the stage clock of every call. Every
output file of one call of each kind is then checked against the CPU oracle: Data.db, Index.db, chunk offsets, digest, and for the side
band call Filter.db, Summary.db, first / last key and every b200c_sstable_stats field. Prints one JSON line (--out: also writes it).

    python tools/bench_lcs_metadata.py --steps 5 --out profiles/r3_lcs_metadata_cfg2.json
"""
import argparse, ctypes as C, json, os, statistics, subprocess, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
import bench

def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().split(", ")
        return {"name": out[0], "power_limit": out[1], "max_sm_clock": out[2]}
    except Exception as e:
        return {"error": str(e)}

class SideBand:
    """host buffers of the side band for nout output slots (HOST pointers whatever the data buffers are)"""
    def __init__(self, nout, words, summary_cap):
        import numpy as np
        from cassandra_b200 import native
        self.keys = [np.zeros(2 * 65535, dtype=np.uint8) for _ in range(nout)]
        self.filter = [np.zeros(8 + 8 * words, dtype=np.uint8) for _ in range(nout)]
        self.summary = [np.zeros(summary_cap, dtype=np.uint8) for _ in range(nout)]
        self.stats = [native.SSTableStats() for _ in range(nout)]
    def attach(self, res):
        for k in range(res.noutputs_cap):
            o = res.outputs[k]
            o.key_buf, o.key_cap = self.keys[k].ctypes.data, len(self.keys[k])
            o.filter, o.filter_cap = self.filter[k].ctypes.data, len(self.filter[k])
            o.summary, o.summary_cap = self.summary[k].ctypes.data, len(self.summary[k])
            o.stats = C.pointer(self.stats[k])
        return res
    def files(self, res):
        return [(bytes(self.keys[k][:res.outputs[k].first_key_len + res.outputs[k].last_key_len]), res.outputs[k].first_key_len,
                 bytes(self.filter[k][:res.outputs[k].filter_len]), bytes(self.summary[k][:res.outputs[k].summary_len]), bytes(self.stats[k]))
                for k in range(res.noutputs)]

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5); ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from cassandra_b200 import native
    from cassandra_b200.io.sstable import bloom_geometry
    wl = dict(bench.WORKLOADS["cfg2"])
    L = native.lib(); ctx = native.Context(0)
    t0 = time.time()
    tabs = bench.make_inputs(wl, bench.gpu_compressor(ctx, wl), max(1, len(os.sched_getaffinity(0))))
    u_in = sum(t.compression.data_length for t in tabs); c_in = sum(t.hold[0].numel() for t in tabs); i_in = sum(t.hold[1].numel() for t in tabs)
    bench.log("inputs ready in %.1fs: %.1f MiB uncompressed" % (time.time() - t0, u_in / 2**20))
    cid, _ = bench.comp_ids(wl)
    nout = int(2 * u_in // wl["lcs"]) + 4
    cap_d = L.b200c_compress_bound(cid, min(u_in, 3 * wl["lcs"]) + (64 << 20), 16384)
    cap_i = min(i_in, i_in * 3 * wl["lcs"] // max(1, u_in) + (64 << 20)) + (1 << 20)
    cap_c = min(u_in, 4 * wl["lcs"]) // 16384 + 16
    # Filter.db geometry as MaxSSTableSizeWriter sizes it: the input keys over the expected number of files, fp chance 0.01
    keys = sum(t.partitions for t in tabs); files = max(1, c_in // wl["lcs"])
    hc, words = bloom_geometry(max(1, keys // files), 0.01)
    def manifests(dev_in=None):
        plain = bench.build_manifest(tabs, wl, dev_in); meta = bench.build_manifest(tabs, wl, dev_in)
        meta.bloom_hash_count, meta.bloom_words, meta.min_index_interval = hc, words, 128
        return plain, meta
    m_host, m_host_meta = manifests()
    dev_in = [(t.hold[0].cuda(), t.hold[1].cuda(), t.hold[2].cuda(), t.summary.cuda()) for t in tabs]
    m_dev, m_dev_meta = manifests([(a.data_ptr(), b.data_ptr(), c.data_ptr(), d_.data_ptr()) for a, b, c, d_ in dev_in])
    bufs = {True: bench.OutBufs(nout, cap_d, cap_i, cap_c, device=True), False: bench.OutBufs(nout, cap_d, cap_i, cap_c, device=False)}
    side = SideBand(nout, words, cap_i // 16 + (1 << 20))

    def call(dev, with_meta):
        res = bufs[dev].result()
        if with_meta: side.attach(res)
        m = (m_dev_meta if with_meta else m_dev) if dev else (m_host_meta if with_meta else m_host)
        torch.cuda.synchronize(); t = time.perf_counter()
        ctx.check(L.b200c_compact(ctx.handle, C.byref(m), C.byref(res), 1 if dev else 0), res.corruption)
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, res.kernel_ms, ctx.last_stage_ms(), res

    legs = {}
    for dev in (True, False):
        for _ in range(args.warmup): call(dev, False); call(dev, True)
        rec = {False: [], True: []}
        for _ in range(args.steps):
            for with_meta in (False, True):                         # alternating: drift hits both arms alike
                ms, kms, stages, _ = call(dev, with_meta); rec[with_meta].append((ms, kms, stages))
        leg = {}
        for with_meta, rows in rec.items():
            ms = [r[0] for r in rows]
            leg["side_band" if with_meta else "plain"] = {
                "ms_per_step": [round(x, 2) for x in ms], "median_ms": round(statistics.median(ms), 2),
                "MB_s": round(u_in / 1e6 / (statistics.median(ms) / 1e3), 1), "kernel_ms_median": round(statistics.median(r[1] for r in rows), 2),
                "stage_ms_mean": [round(sum(r[2][i] for r in rows) / len(rows), 2) for i in range(len(rows[0][2]))]}
        leg["side_band_cost_ms"] = round(leg["side_band"]["median_ms"] - leg["plain"]["median_ms"], 2)
        legs["device_resident" if dev else "host_buffers"] = leg
        bench.log("%s: plain %.1f ms, side band %.1f ms" % ("device" if dev else "host", leg["plain"]["median_ms"], leg["side_band"]["median_ms"]))

    # ---- where the side band's time goes, file by file (B200C_LCS_META_SPLIT: one JSON line per file from the writer loop) ----------------
    import tempfile
    split = {}
    for dev in (True, False):
        fd, path = tempfile.mkstemp(suffix=".jsonl"); os.close(fd)
        os.environ["B200C_LCS_META_SPLIT"] = path
        try: call(dev, True)
        finally: del os.environ["B200C_LCS_META_SPLIT"]
        split["device_resident" if dev else "host_buffers"] = [json.loads(l) for l in open(path) if l.strip()]
        os.unlink(path)

    # ---- every file of one call of each kind against the CPU oracle --------------------------------------------------------------
    O = bench.oracle_api()
    _, _, _, r_plain = call(False, False); got_plain = bufs[False].files(r_plain)
    _, _, _, r_meta = call(False, True); got_meta = bufs[False].files(r_meta); got_side = side.files(r_meta)
    _, _, _, r_dev = call(True, True); got_dev = bufs[True].files(r_dev); got_dev_side = side.files(r_dev)
    res_o, files_o = bench.host_out_bufs_numpy(nout, cap_d, cap_i, cap_c)
    side_o = SideBand(nout, words, cap_i // 16 + (1 << 20)); side_o.attach(res_o)
    t = time.perf_counter(); bench.cpu_compact(O, m_host_meta, res_o, 1); oracle_s = time.perf_counter() - t
    want = files_o(); want_side = side_o.files(res_o)
    checks = {"data_plain": bench.same_files(got_plain, want), "data_side_band": bench.same_files(got_meta, want),
              "data_side_band_device": bench.same_files(got_dev, want),
              "side_band": None if got_side == want_side else "side band differs in file %d" % next(k for k in range(max(len(got_side), len(want_side))) if k >= len(got_side) or k >= len(want_side) or got_side[k] != want_side[k]),
              "side_band_device": None if got_dev_side == want_side else "device-resident side band differs"}
    line = {"workload": wl["name"], "card": card(), "steps": args.steps, "warmup": args.warmup, "u_in_bytes": u_in, "output_files": len(want),
            "bloom": {"hash_count": hc, "words": words}, "stage_names": ["K1", "K2", "K3", "K4 size", "K4 emit", "K5"],
            "legs": legs, "side_band_split_per_file": split, "oracle_s": round(oracle_s, 1), "checks": checks, "verified": all(v is None for v in checks.values())}
    print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f: json.dump(line, f, indent=1)
    ctx.close()
    return 0 if line["verified"] else 1

if __name__ == "__main__":
    sys.exit(main())
