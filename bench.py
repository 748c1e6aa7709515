#!/usr/bin/env python
"""bench.py — compaction MB/s (uncompressed in) + rows merged/s on N x B200 (BASELINE.json metric).

A step = one full compaction (b200c_compact: K1 decompress+CRC verify -> K2 index scan -> K3 partition merge -> K4 row merge /
purge / serialise -> K5 LZ4|Snappy + CRC32) of one batch of synthetic input SSTables.
  --workload cfg1  (default) BASELINE.json configs[1]: STCS, 16 SSTables x 1 GiB (uncompressed), LZ4, chunk 16 KiB, schema N, seed 0xCA550002
  --workload cfg2  configs[2]: LCS L0->L1, 32 overlapping SSTables x 160 MiB, Snappy, output switched every 160 MiB (multi-file)
  --workload cfg4  configs[4] shape at one-GPU scale: schema W (1000 clustering rows / partition, ~70 KB partitions), 8 x 1 GiB, LZ4
  N>1              ONE compaction sharded by token range: rank 0 picks N-1 splitters from Summary.db samples and broadcasts them (the only
                   collective on the data path); every rank compacts its (lo, hi] of the SAME inputs. "scaling": "strong".
  value            whole-job MB/s with the inputs (compressed Data.db, Index.db, chunk offsets) already resident in HBM.
  e2e              the same metric through the C ABI with HOST buffers: pinned host -> device copies of every input and the
                   device -> host read-back of Data.db/Index.db/offsets are inside the timed region. Same number of steps as `value`.
  roofline         the dominant kernel stage (CUDA-event time from the engine's own stream) against MEASURED_PEAKS.json hbm_gbs;
                   traffic = DRAM bytes per launch from the committed ncu capture of the same workload (profiles/r2_traffic.json).
  cpu_baseline     the CPU oracle (C++ restatement of the reference algorithm) on this box's host cores over the SAME inputs: one
                   compaction cut into token ranges, one oracle thread per range (oracle/parallel.cc) — the reference itself would run
                   this compaction on ONE thread; that figure is reported beside it. Bounded to ~20 s (a prefix of the ring if needed).
  verified         the output of the timed configuration — device-resident AND streamed through host buffers — compared byte for byte
                   (Data.db, Index.db, chunk offsets, Digest.crc32, counters) with the CPU oracle's output for the same inputs.
--impl reference   the CPU oracle with all host threads on the same workload, same metric/unit (+ its scaling curve over threads).
--dump-outputs DIR the output files of the last timed device-resident step as DIR/<name>.npy (see dump_outputs), so that two builds can be
                   compared output for output: the inputs are seeded, identical from run to run for the same arguments.
Input synthesis (synth/) never touches oracle/: the b200 arm compresses its inputs with the engine's own K5 kernels.
"""
import argparse, ctypes as C, json, os, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: nothing is cached next to the sources
NOW = 1700000000
METRIC = "compaction MB/s (uncompressed in)"
INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1

WORKLOADS = {
    "cfg1": dict(name="BASELINE.json configs[1]: STCS 16 SSTables x 1024 MiB, LZ4", schema="N", sstables=16, mib=1024.0, comp="lz4", p=0.5, lcs=0, seed=0xCA550002, bands=0, l0=0),
    "cfg2": dict(name="BASELINE.json configs[2]: LCS L0->L1 32 SSTables x 160 MiB, Snappy, 160 MiB outputs", schema="N", sstables=32, mib=160.0, comp="snappy", p=0.25,
                 lcs=160 << 20, seed=0xCA550003, bands=8, l0=4),
    "cfg4": dict(name="BASELINE.json configs[4] shape at 1-GPU scale: schema W (1000 rows/partition), 8 SSTables x 1024 MiB, LZ4", schema="W", sstables=8, mib=1024.0,
                 comp="lz4", p=0.5, lcs=0, seed=0xCA550005, bands=0, l0=0),
}

def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)

def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try: return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
        except Exception: pass
    return 6650.0, "fallback"

class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    def __init__(self, gpu):
        super().__init__(daemon=True); self.gpu = gpu; self.samples = []; self.reasons = set(); self._stop_ev = threading.Event(); self.max_mhz = None
    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                    if "Active" in v and "Not" not in v: self.reasons.add(name)
            except Exception:
                pass
            self._stop_ev.wait(0.2)
    def stop(self):
        self._stop_ev.set(); self.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}

def bind_to_gpu_numa(local_rank):
    """pinned staging buffers and the threads that fill them should live on the GPU's NUMA node (2-socket hosts: GPUs 0-3 / 4-7)"""
    try:
        import pynvml
        pynvml.nvmlInit(); h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]).read())
        if node < 0: return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-"); cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:
        return {"numa_node": None, "error": str(e)[:80]}

# ---------------------------------------------------------------------------------------------------------------------------
class Inputs:
    """synthetic input SSTables of one workload: data/index/offsets/summary as (pinned) torch tensors in .hold / .summary"""
    pass

def comp_ids(wl):
    from cassandra_b200 import native
    return (native.COMP_SNAPPY, "SnappyCompressor") if wl["comp"] == "snappy" else (native.COMP_LZ4, "LZ4Compressor")

def make_inputs(wl, compress, threads, pinned=True):
    """compress(stream ndarray) -> (uint8 ndarray image, uint64 ndarray chunk offsets). Returns SSTable objects (cassandra_b200.io.sstable)."""
    import numpy as np, torch, synth
    from cassandra_b200 import native
    from cassandra_b200.io.sstable import SSTable
    from cassandra_b200.io.compress import CompressionMetadata
    schema = 0 if wl["schema"] == "N" else 1
    per = int(wl["mib"] * 2**20); nsst = wl["sstables"]; rpp = wl.get("rpp", 1000)
    universe = synth.universe_for(schema, per, wl["p"], rpp)
    _, cname = comp_ids(wl)
    tabs = []
    for s in range(nsst):
        t0 = time.time()
        raw = synth.generate_raw(schema, s, nsst, wl["seed"], universe, wl["p"], rows_per_partition=rpp, threads=threads, band_count=wl["bands"], l0_count=wl["l0"])
        n = len(raw["stream"])
        image, offs = compress(raw["stream"])
        def pin(a):
            t = torch.from_numpy(np.ascontiguousarray(a))
            return t.pin_memory() if pinned else t
        d = pin(image); ix = pin(np.frombuffer(raw["index"], dtype=np.uint8)); of = pin(offs.view(np.int64)); sm = pin(raw["summary"].view(np.int64))
        meta = CompressionMetadata(cname, 16384, native.INT32_MAX, n, [])
        t = SSTable(None, None, meta, raw["stats"], raw["stats"], synth.SCHEMAS[schema]["clustering"], synth.SCHEMAS[schema]["columns"], generation=s)
        t.hold = (d, ix, of); t.summary = sm; t.nchunks = len(offs); t.partitions = raw["partitions"]; t.rows = raw["rows"]
        tabs.append(t)
        log("input %d/%d: %.1f MiB uncompressed -> %.1f MiB, %d partitions (%.1fs)" % (s + 1, nsst, n / 2**20, len(image) / 2**20, raw["partitions"], time.time() - t0))
        del raw
    return tabs

def gpu_compressor(ctx, wl):
    import numpy as np
    from cassandra_b200 import native
    L = native.lib(); cid, _ = comp_ids(wl)
    def compress(stream):
        n = len(stream); cap = L.b200c_compress_bound(cid, n, 16384); nch = L.b200c_chunk_count(n, 16384)
        out = np.empty(cap, dtype=np.uint8); offs = np.zeros(max(nch, 1), dtype=np.uint64); out_len = C.c_uint64(); dig = C.c_uint32()
        ctx.check(L.b200c_compress_chunks(ctx.handle, cid, stream.ctypes.data, n, 16384, native.INT32_MAX, out.ctypes.data, cap, C.byref(out_len), offs.ctypes.data, C.byref(dig), 0))
        return out[:out_len.value], offs[:nch]
    return compress

def oracle_compressor(wl):
    """reference arm only: inputs compressed by the CPU oracle's codec (one C call per stream, GIL released)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np, oracle_lib as O
    L = O.lib(); cid = O.COMP_SNAPPY if wl["comp"] == "snappy" else O.COMP_LZ4
    L.orc_compress_stream.restype = C.c_uint64
    L.orc_compress_stream.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
    def compress(stream):
        n = len(stream); nch = (n + 16383) // 16384
        out = np.empty(nch * (L.orc_chunk_max_compressed(cid, 16384) + 4) + 64, dtype=np.uint8); offs = np.zeros(max(nch, 1), dtype=np.uint64)
        # chunk-parallel: slices of 4096 chunks on a thread pool, offsets re-based afterwards
        from concurrent.futures import ThreadPoolExecutor
        step = 4096 * 16384; pieces = [(i, min(n, i + step)) for i in range(0, n, step)]
        def one(ab):
            a, b = ab; k = (b - a + 16383) // 16384
            o = np.empty(k * (L.orc_chunk_max_compressed(cid, 16384) + 4) + 64, dtype=np.uint8); of = np.zeros(max(k, 1), dtype=np.uint64)
            m = L.orc_compress_stream(cid, stream[a:b].ctypes.data, b - a, 16384, o.ctypes.data, of.ctypes.data)
            return o[:m], of[:k]
        with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex: parts = list(ex.map(one, pieces))
        pos = 0; k0 = 0
        for o, of in parts:
            out[pos:pos + len(o)] = o; offs[k0:k0 + len(of)] = of + np.uint64(pos); pos += len(o); k0 += len(of)
        return out[:pos], offs[:nch]
    return compress

def build_manifest(tabs, wl, device_copies=None, token_range=(INT64_MIN, INT64_MAX)):
    """b200c_manifest over the inputs; device_copies = list of (data_ptr, index_ptr, offs_ptr, summary_ptr) to use instead of the host tensors."""
    import synth
    from cassandra_b200 import native
    from cassandra_b200.io import sstable as sst
    from cassandra_b200.db.compaction import merged_encoding_stats
    cid, _ = comp_ids(wl)
    m = native.Manifest(); m.abi_version = native.ABI_VERSION; m.ninputs = len(tabs)
    arr = (native.Input * len(tabs))()
    for k, t in enumerate(tabs):
        d, ix, of = t.hold
        a = arr[k]
        if device_copies: a.data, a.index, a.chunk_offsets, a.summary_positions = device_copies[k]
        else: a.data, a.index, a.chunk_offsets, a.summary_positions = d.data_ptr(), ix.data_ptr(), of.data_ptr(), t.summary.data_ptr()
        a.nsummary = t.summary.numel()
        a.data_len = d.numel(); a.index_len = ix.numel(); a.nchunks = t.nchunks; a.data_length = t.compression.data_length
        a.compressor = cid; a.chunk_len = 16384; a.max_compressed_len = native.INT32_MAX
        a.ncolumns = len(t.regular_columns)
        for ci in range(a.ncolumns): a.column_map[ci] = ci
        a.header_stats.min_timestamp, a.header_stats.min_local_deletion_time, a.header_stats.min_ttl = t.header_stats
    m.inputs = arr
    sc = synth.SCHEMAS[0 if wl["schema"] == "N" else 1]
    m.nclustering = len(sc["clustering"])
    for k, ty in enumerate(sc["clustering"]): m.clustering[k].type, m.clustering[k].fixed_len = sst.type_class(ty)
    m.ncolumns = len(sc["columns"])
    for k, (_, ty) in enumerate(sc["columns"]): m.columns[k].type, m.columns[k].fixed_len = sst.type_class(ty)
    m.out_stats.min_timestamp, m.out_stats.min_local_deletion_time, m.out_stats.min_ttl = merged_encoding_stats(tabs)
    m.out_compressor = cid; m.out_chunk_len = 16384; m.out_max_compressed_len = native.INT32_MAX; m.column_index_size = 65536
    m.now_in_sec = NOW; m.gc_before = NOW - 864000; m.purge_max_timestamp = INT64_MAX
    m.token_lo, m.token_hi = token_range
    m.max_sstable_bytes = wl["lcs"]; m.partitioner = native.PARTITIONER_MURMUR3
    m._keep = arr
    return m

class OutBufs:
    """caller-provided output buffers for up to `nout` files, on the host (pinned) or on the device"""
    def __init__(self, nout, cap_d, cap_i, cap_c, device):
        import torch
        mk = (lambda n, dt: torch.empty(n, dtype=dt, device="cuda")) if device else (lambda n, dt: torch.empty(n, dtype=dt).pin_memory())
        self.bufs = [(mk(cap_d, torch.uint8), mk(cap_i, torch.uint8), mk(cap_c, torch.int64)) for _ in range(nout)]
        self.caps = (cap_d, cap_i, cap_c); self.nout = nout
    def result(self):
        from cassandra_b200 import native
        res = native.Result(); outs = (native.Output * self.nout)()
        for o, (d, ix, co) in zip(outs, self.bufs):
            o.data, o.data_cap, o.index, o.index_cap, o.chunk_offsets, o.chunk_cap = d.data_ptr(), self.caps[0], ix.data_ptr(), self.caps[1], co.data_ptr(), self.caps[2]
        res.noutputs_cap = self.nout; res.outputs = outs; res._keep = outs
        return res
    def files(self, res):
        """[(Data.db bytes ndarray, Index.db ndarray, offsets ndarray, digest, partitions, rows)] as host numpy arrays"""
        out = []
        for k in range(res.noutputs):
            o = res.outputs[k]; d, ix, co = self.bufs[k]
            out.append((d[:o.data_len].cpu().numpy(), ix[:o.index_len].cpu().numpy(), co[:o.nchunks].cpu().numpy().view("uint64"), int(o.digest), int(o.partitions), int(o.rows)))
        return out

# ---------------------------------------------------------------------------------------------------------------------------
def oracle_api():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    from cassandra_b200 import native
    L = O.lib()
    L.orc_compact_parallel.restype = C.c_int
    L.orc_compact_parallel.argtypes = [C.POINTER(native.Manifest), C.POINTER(native.Result), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_char_p, C.c_int]
    L.orc_compact.restype = C.c_int
    L.orc_compact.argtypes = [C.POINTER(native.Manifest), C.POINTER(native.Result), C.c_char_p, C.c_int]
    return L

def usable_cpus():
    """(threads worth starting, note): the CPUs this process may run on, capped by the container's CPU-time quota (cgroup cpu.max /
    cfs_quota): with a quota of q CPUs, more than q busy threads are only throttled — on the round-2 GPU box 128 logical CPUs were visible,
    the pod got 16 CPUs' worth of time, and 64 / 128 oracle threads ran SLOWER than 16 (profiles/r2_cpu_arm_scaling.txt)."""
    n = len(os.sched_getaffinity(0)); quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max": quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0: quota = q / per
        except Exception: pass
    if quota is not None and quota < n: return max(1, int(quota + 0.5)), {"visible_cpus": n, "cgroup_cpu_quota": round(quota, 2)}
    return n, {"visible_cpus": n, "cgroup_cpu_quota": quota}

def cpu_compact(L, m, res, threads, ranges=0, max_ranges=0):
    """one CPU-oracle compaction of manifest m into res. threads > 1 (single-output workloads): token-range parallel oracle.
    Returns (seconds, sample_token_hi, [merge, stitch, compress] ms)."""
    err = C.create_string_buffer(256); tm = (C.c_double * 6)(); hi = C.c_int64(INT64_MAX)
    t0 = time.perf_counter()
    if m.max_sstable_bytes or threads <= 1 and not max_ranges:
        rc = L.orc_compact(C.byref(m), C.byref(res), err, 256)
    else:
        rc = L.orc_compact_parallel(C.byref(m), C.byref(res), threads, ranges or max(threads * 8, 16), max_ranges, tm, C.byref(hi), err, 256)
    dt = time.perf_counter() - t0
    if rc != 0: raise RuntimeError("CPU oracle failed rc=%d: %s" % (rc, err.value.decode()))
    return dt, hi.value, [round(tm[k], 1) for k in range(6)]

def host_out_bufs_numpy(nout, cap_d, cap_i, cap_c):
    import numpy as np
    from cassandra_b200 import native
    bufs = [(np.empty(cap_d, dtype=np.uint8), np.empty(cap_i, dtype=np.uint8), np.zeros(cap_c, dtype=np.uint64)) for _ in range(nout)]
    res = native.Result(); outs = (native.Output * nout)()
    for o, (d, ix, co) in zip(outs, bufs):
        o.data, o.data_cap, o.index, o.index_cap, o.chunk_offsets, o.chunk_cap = d.ctypes.data, cap_d, ix.ctypes.data, cap_i, co.ctypes.data, cap_c
    res.noutputs_cap = nout; res.outputs = outs; res._keep = (outs, bufs)
    def files():
        return [(bufs[k][0][:res.outputs[k].data_len], bufs[k][1][:res.outputs[k].index_len], bufs[k][2][:res.outputs[k].nchunks], int(res.outputs[k].digest),
                 int(res.outputs[k].partitions), int(res.outputs[k].rows)) for k in range(res.noutputs)]
    return res, files

def same_files(a, b):
    import numpy as np
    if len(a) != len(b): return "file count %d vs %d" % (len(a), len(b))
    for k, (x, y) in enumerate(zip(a, b)):
        for name, u, v in (("Data.db", x[0], y[0]), ("Index.db", x[1], y[1]), ("chunk offsets", x[2], y[2])):
            if len(u) != len(v) or not np.array_equal(u, v): return "file %d: %s differs (%d vs %d bytes)" % (k, name, len(u), len(v))
        if x[3:] != y[3:]: return "file %d: digest/partitions/rows %s vs %s" % (k, x[3:], y[3:])
    return None

DUMP_SAMPLES = {"data": 2 << 20, "index": 1 << 20, "chunk_offsets": 1 << 19}    # elements per job, split over its output files: < 64 MB in all

def sample_positions(n, cap, seed):
    """sorted positions of a stratified sample of cap of n elements, fixed by seed (every position when n <= cap)"""
    import numpy as np
    if n <= cap: return np.arange(n, dtype=np.int64)
    stride = n // cap
    return np.arange(cap, dtype=np.int64) * stride + np.random.default_rng(seed).integers(0, stride, cap)

def dump_outputs(ob, res, ninputs):
    """What a caller of b200c_compact receives, as float arrays. For output file k: out<k>_data, out<k>_index, out<k>_chunk_offsets hold the
    Data.db bytes, Index.db bytes and chunk offsets at the positions in out<k>_<name>_pos (a fixed, seeded sample of large files). `files` has
    one row per output: data_len, index_len, nchunks, data_length, digest (CRC32 of all of Data.db), CRC32 of all of Index.db, CRC32 of all
    chunk offsets, partitions, rows. `counters`: bytes_read, bytes_in_range, bytes_written, total_source_rows, input_partitions, merged_row_counts."""
    import numpy as np, torch, zlib
    out, files = {}, []
    for k in range(res.noutputs):
        o = res.outputs[k]; d, ix, co = ob.bufs[k]
        for j, (name, t, dt) in enumerate((("data", d[:o.data_len], np.float32), ("index", ix[:o.index_len], np.float32), ("chunk_offsets", co[:o.nchunks], np.float64))):
            pos = sample_positions(t.numel(), DUMP_SAMPLES[name] // res.noutputs, seed=1000 * k + j)
            out["out%d_%s" % (k, name)] = t[torch.from_numpy(pos).to(t.device)].cpu().numpy().astype(dt)
            out["out%d_%s_pos" % (k, name)] = pos.astype(np.float64)
        files.append([o.data_len, o.index_len, o.nchunks, o.data_length, o.digest, zlib.crc32(ix[:o.index_len].cpu().numpy()),
                      zlib.crc32(co[:o.nchunks].cpu().numpy()), o.partitions, o.rows])
    out["files"] = np.array(files, dtype=np.float64).reshape(-1, 9)
    out["counters"] = np.array([res.bytes_read, res.bytes_in_range, res.bytes_written, res.total_source_rows, res.input_partitions] +
                               [int(x) for x in res.merged_row_counts[:ninputs]], dtype=np.float64)
    return out

def estimate_max_ranges(u_in, threads, ranges, budget_s, per_thread_mbs=110.0):
    est = u_in / 1e6 / (per_thread_mbs * max(1, threads) * 0.7)
    if est <= budget_s: return 0, est
    return max(1, int(ranges * budget_s / est)), est

# ---------------------------------------------------------------------------------------------------------------------------
def run_b200(args, wl):
    import numpy as np, torch
    import torch.distributed as dist
    from cassandra_b200 import native, parallel
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa(local)                                   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    L = native.lib()
    ctx = native.Context(local)
    # the run manifest (workload shape) is decided by rank 0 and broadcast once
    shape = parallel.broadcast_manifest(dict(wl=wl, steps=args.steps, warmup=args.warmup, now=NOW) if rank == 0 else None)
    wl = shape["wl"]
    threads = max(1, len(os.sched_getaffinity(0)) // max(1, min(world, 4)))
    t0 = time.time()
    tabs = make_inputs(wl, gpu_compressor(ctx, wl), threads)
    log("rank %d: inputs ready in %.1fs" % (rank, time.time() - t0))
    u_in = sum(t.compression.data_length for t in tabs); c_in = sum(t.hold[0].numel() for t in tabs); i_in = sum(t.hold[1].numel() for t in tabs)
    cid, _ = comp_ids(wl)

    # multi-GPU: ONE compaction, sharded by token range. Rank 0 picks world-1 splitters from the Summary.db samples of all inputs
    # (every 128th key; the host hashes them) so that the shards hold equal numbers of sampled partitions; one broadcast.
    token_range = (INT64_MIN, INT64_MAX)
    if world > 1:
        cuts = None
        if rank == 0:
            toks = sample_tokens(tabs, per_input=4096)
            cuts = parallel.weighted_token_ranges(toks, world)
        cuts = parallel.broadcast_manifest(cuts)
        token_range = tuple(cuts[rank])

    nout = 1 if not wl["lcs"] else int(2 * u_in // wl["lcs"]) + 4
    cap_d = L.b200c_compress_bound(cid, u_in if not wl["lcs"] else min(u_in, 3 * wl["lcs"]) + (64 << 20), 16384)
    cap_i = (i_in if not wl["lcs"] else min(i_in, i_in * 3 * wl["lcs"] // max(1, u_in) + (64 << 20))) + (1 << 20)
    cap_c = (u_in if not wl["lcs"] else min(u_in, 4 * wl["lcs"])) // 16384 + 16
    if world > 1: cap_d = cap_d // world * 2 + (64 << 20); cap_i = cap_i // world * 2 + (16 << 20); cap_c = cap_c // world * 2 + 1024
    m_host = build_manifest(tabs, wl, token_range=token_range)
    ho = OutBufs(nout, cap_d, cap_i, cap_c, device=False)
    dev_in = [(t.hold[0].cuda(), t.hold[1].cuda(), t.hold[2].cuda(), t.summary.cuda()) for t in tabs]
    m_dev = build_manifest(tabs, wl, [(a.data_ptr(), b.data_ptr(), c.data_ptr(), d_.data_ptr()) for a, b, c, d_ in dev_in], token_range=token_range)
    do = OutBufs(nout, cap_d, cap_i, cap_c, device=True)

    def step(dev):
        res = (do if dev else ho).result()
        ctx.check(L.b200c_compact(ctx.handle, C.byref(m_dev if dev else m_host), C.byref(res), 1 if dev else 0), res.corruption)
        return res

    def timed(dev, steps, sampler=None):
        torch.cuda.synchronize()
        if world > 1: dist.barrier()
        torch.cuda.synchronize()
        if sampler: sampler.start()
        launches0 = ctx.total_kernel_launches
        t = time.perf_counter(); kms = 0.0; stages = [0.0] * 6; last = None
        for _ in range(steps):
            last = step(dev); kms += last.kernel_ms
            for i, v in enumerate(ctx.last_stage_ms()): stages[i] += v
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        clocks = sampler.stop() if sampler else None
        return parallel.max_over_ranks(dt, device="cuda"), kms / steps, [s / steps for s in stages], last, ctx.total_kernel_launches - launches0, clocks

    for _ in range(args.warmup): step(True)
    dt, kms, stages, last, launches, clocks = timed(True, args.steps, ClockSampler(local))
    dump = dump_outputs(do, last, len(tabs)) if args.dump_outputs else None     # before any later leg reuses the device buffers
    sum_outs = lambda res, f: sum(int(getattr(res.outputs[k], f)) for k in range(res.noutputs))
    u_out, c_out, i_out = int(last.bytes_written), sum_outs(last, "data_len"), sum_outs(last, "index_len")
    rows = int(last.total_source_rows); parts_in = int(last.input_partitions); in_range = int(last.bytes_in_range)
    # whole-job numbers: the job is ONE compaction of u_in bytes; a rank's own share is bytes_in_range
    counters = parallel.all_gather_counters(dict(in_range=in_range, rows=rows, parts_in=parts_in, u_out=u_out, c_out=c_out, i_out=i_out))
    job_in = sum(cn["in_range"] for cn in counters); job_rows = sum(cn["rows"] for cn in counters)
    value = job_in * args.steps / dt / 1e6
    step(False)
    edt, ekms, estages, elast, _, _ = timed(False, args.steps)
    e2e = job_in * args.steps / edt / 1e6
    sweep = {}
    for rr in [x for x in args.e2e_ranges.split(",") if x]:
        os.environ["B200C_RANGES"] = rr
        step(False)
        sdt, _, sst_, _, _, _ = timed(False, max(1, min(args.steps, 3)))
        sweep[rr] = {"ms_per_step": round(sdt / max(1, min(args.steps, 3)) * 1e3, 2), "stage_ms": [round(x, 1) for x in sst_]}
        del os.environ["B200C_RANGES"]
    ab = None
    if args.ab_env:
        for kv in args.ab_env.split(","):
            k_, v_ = kv.split("=", 1); os.environ[k_] = v_
        step(True); step(False)
        adt, _, ast_, _, _, _ = timed(True, args.steps)
        bdt, _, bst_, _, _, _ = timed(False, max(1, min(args.steps, 3)))
        ab = {"env": args.ab_env, "value": round(job_in * args.steps / adt / 1e6, 1), "e2e": round(job_in * max(1, min(args.steps, 3)) / bdt / 1e6, 1),
              "stage_ms": [round(x, 1) for x in ast_], "e2e_stage_ms": [round(x, 1) for x in bst_]}
        for kv in args.ab_env.split(","): del os.environ[kv.split("=", 1)[0]]
    h2d = c_in + i_in + 8 * sum(t.nchunks for t in tabs) + 8 * sum(t.summary.numel() for t in tabs) if world == 1 else None
    d2h = sum_outs(elast, "data_len") + sum_outs(elast, "index_len") + 8 * sum_outs(elast, "nchunks")

    # roofline of the dominant stage, algorithmic bytes per SURVEY §8(d): every compressed byte read once, every uncompressed byte
    # produced once, merged stream written once and compressed once
    names = ["K1 decompress+verify", "K2 index scan", "K3 partition merge", "K4 merge+purge+serialise", "K4 gather+index", "K5 compress+crc+pack"]
    share = in_range / max(1, u_in)
    alg = [(c_in + u_in) * share, i_in + 26 * parts_in, 26 * parts_in + 20 * parts_in, in_range + u_out, 2 * u_out + i_out, u_out + c_out]
    dom = max(range(6), key=lambda i: stages[i])
    peak, which = peaks()
    b_alg = (c_in + i_in + u_in) * share + u_out + c_out + i_out
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath)).get(args.workload, {})
            traffic = tj.get(names[dom])
        except Exception: pass
    roof = {"bound": "hbm", "kernel": names[dom], "achieved": round(alg[dom] / (stages[dom] / 1e3) / 1e9, 2), "peak": peak, "unit": "GB/s",
            "frac": round(alg[dom] / (stages[dom] / 1e3) / 1e9 / peak, 5), "traffic": traffic, "traffic_source": "profiles/r2_traffic.json (ncu dram__bytes_read+write per step, same workload)" if traffic else None,
            "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)" if which == "measured" else which,
            "stage_ms": {n: round(s, 3) for n, s in zip(names, stages)},
            "stage_achieved_gbs": {n: (round(a_ / (s / 1e3) / 1e9, 1) if s > 0 else None) for n, a_, s in zip(names, alg, stages)},
            "kernel_ms_per_step": round(kms, 3),
            "pipeline_achieved_gbs": round(b_alg / (kms / 1e3) / 1e9, 2), "pipeline_frac": round(b_alg / (kms / 1e3) / 1e9 / peak, 5),
            "algorithmic_bytes_per_step": int(b_alg)}
    line = {"metric": METRIC, "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": wl["name"] + ", chunk 16 KiB, schema %s, seed %#x" % (wl["schema"], wl["seed"]),
                       "uncompressed_in_bytes": u_in, "l2": "inputs (%.1f GB/step) larger than L2" % ((c_in + u_in) / 1e9),
                       "parallelism": ("ONE compaction sharded by token range over %d GPUs: splitters from Summary.db samples, one broadcast, no data-path collective" % world) if world > 1 else "1 GPU",
                       "now_in_sec": NOW, "gc_grace": 864000, "numa": numa},
            "rows_merged_per_s": round(job_rows * args.steps / dt, 0), "input_partitions_per_step": sum(cn["parts_in"] for cn in counters),
            "merged_row_counts": [int(x) for x in last.merged_row_counts[:len(tabs)]],
            "bytes": {"u_in": u_in, "c_in": c_in, "index_in": i_in, "in_range_this_rank": in_range, "u_out": u_out, "c_out": c_out, "index_out": i_out, "outputs": int(last.noutputs)},
            "shards": [cn["in_range"] for cn in counters] if world > 1 else None,
            "e2e": {"value": round(e2e, 1), "unit": "MB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": round(edt / args.steps * 1e3, 2), "steps": args.steps,
                    "device_ms_per_step": round(ekms, 2), "stage_ms": {n: round(s_, 2) for n, s_ in zip(names, estages)}},
            "e2e_ranges_sweep": sweep or None, "ab": ab, "gpu_launches": int(launches), "index_slow_path_inputs": int(last.index_slow_path_inputs), "clocks": clocks, "roofline": roof}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_leg_and_verify(args, wl, line, tabs, m_host, (cap_d, cap_i, cap_c, nout), ctx, L, do, ho, last, elast, build_manifest, dev_in)
    if rank == 0:
        emit(line)
    if dump:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, ("rank%d_" % rank if world > 1 else "") + name + ".npy"), a)
        log("wrote %d arrays (%.1f MB) to %s" % (len(dump), sum(a.nbytes for a in dump.values()) / 1e6, args.dump_outputs))
    ctx.close()
    if world > 1: dist.destroy_process_group()

def sample_tokens(tabs, per_input=4096):
    """Murmur3 tokens of evenly spaced Summary.db samples (host side, b200c_token — splitter choice only)"""
    import numpy as np
    from cassandra_b200 import native
    L = native.lib(); toks = []
    for t in tabs:
        ix = t.hold[1].numpy(); sm = t.summary.numpy().view("uint64")
        for k in np.linspace(0, len(sm) - 1, min(per_input, len(sm))).astype(np.int64):
            off = int(sm[k]); kl = (int(ix[off]) << 8) | int(ix[off + 1])
            toks.append(L.b200c_token(native.PARTITIONER_MURMUR3, ix[off + 2:off + 2 + kl].ctypes.data, kl))
    return toks

def cpu_leg_and_verify(args, wl, line, tabs, m_host, caps, ctx, L, do, ho, last, elast, build_manifest, dev_in):
    """rank 0, N=1: time the CPU oracle on the same inputs (bounded), then use its output to verify the GPU's."""
    import numpy as np
    from cassandra_b200 import native
    cap_d, cap_i, cap_c, nout = caps
    OL = oracle_api()
    threads, cpu_note = usable_cpus(); u_in = sum(t.compression.data_length for t in tabs)
    ranges = max(64, threads * 4)
    if wl["lcs"]:
        max_ranges = 0; thr = 1                 # multi-file output: the single-threaded oracle (= one reference compaction task)
    else:
        max_ranges, est = estimate_max_ranges(u_in, threads, ranges, args.cpu_budget_s); thr = threads
    res, files = host_out_bufs_numpy(nout, cap_d, cap_i, cap_c)
    sec, hi, tm = cpu_compact(OL, m_host, res, thr, ranges, max_ranges)
    covered = int(res.bytes_in_range)
    cb = {"value": round(covered / sec / 1e6, 1), "unit": "MB/s", "cores": thr, "kind": "port",
          "sample": ("the whole workload" if hi == INT64_MAX else "token range (MIN, %d] of the same workload = %.1f %% of its bytes" % (hi, 100.0 * covered / u_in)) +
                    (", one compaction cut into %d token ranges, one oracle thread per range (oracle/parallel.cc)" % ranges if thr > 1 else ", single-threaded oracle (= one reference compaction task)"),
          "seconds": round(sec, 2), "phase_ms": [round(x, 1) for x in tm[:3]], "range_tasks_ms": {"wall_sum": tm[3], "thread_cpu_sum": tm[4], "longest": tm[5]}, "host": cpu_note, "rows_merged_per_s": round(int(res.total_source_rows) / sec, 0)}
    if thr > 1:                                  # what ONE reference compaction task achieves: a single thread, on a small prefix
        r1, _ = host_out_bufs_numpy(1, cap_d // 16 + (1 << 20), cap_i // 16 + (1 << 20), cap_c // 16 + 1024)
        s1, _, _ = cpu_compact(OL, m_host, r1, 1, ranges, max(1, ranges // 128))
        cb["one_thread"] = {"value": round(int(r1.bytes_in_range) / s1 / 1e6, 1), "unit": "MB/s", "seconds": round(s1, 2), "sample_bytes": int(r1.bytes_in_range)}
    line["cpu_baseline"] = cb
    # ---- verification ----------------------------------------------------------------------------------------------------------------
    want = files()
    if hi == INT64_MAX:
        got_dev, got_host, lastc, elastc = do.files(last), ho.files(elast), last, elast
    else:                                        # the CPU covered a prefix of the ring: compact exactly that token range on the GPU, both ways
        mh = build_manifest(tabs, wl, token_range=(INT64_MIN, hi))
        md = build_manifest(tabs, wl, [(a.data_ptr(), b.data_ptr(), c.data_ptr(), d_.data_ptr()) for a, b, c, d_ in dev_in], token_range=(INT64_MIN, hi))
        lastc = do.result(); ctx.check(L.b200c_compact(ctx.handle, C.byref(md), C.byref(lastc), 1), lastc.corruption)
        elastc = ho.result(); ctx.check(L.b200c_compact(ctx.handle, C.byref(mh), C.byref(elastc), 0), elastc.corruption)
        got_dev, got_host = do.files(lastc), ho.files(elastc)
    problems = []
    for label, got, r in (("device-resident", got_dev, lastc), ("host-streamed", got_host, elastc)):
        p = same_files(got, want)
        if p: problems.append(label + ": " + p)
        for k in ("bytes_in_range", "bytes_written", "total_source_rows", "input_partitions"):
            if int(getattr(r, k)) != int(getattr(res, k)): problems.append("%s: %s %d vs %d" % (label, k, int(getattr(r, k)), int(getattr(res, k))))
        if [int(x) for x in r.merged_row_counts[:len(tabs)]] != [int(x) for x in res.merged_row_counts[:len(tabs)]]: problems.append(label + ": merged_row_counts")
    import zlib
    line["verified"] = {"ok": not problems, "against": "CPU oracle (oracle/, pinned by the reference's golden SSTables)", "fraction_of_workload": round(covered / u_in, 4),
                        "compared": ["Data.db", "Index.db", "chunk offsets", "Digest.crc32", "partitions", "rows", "counters"], "paths": ["device-resident", "host-streamed"],
                        "data_db_bytes": int(sum(len(f[0]) for f in want)), "digest_is_crc32_of_data": bool(all(zlib.crc32(f[0].tobytes()) == f[3] for f in got_host[:1])),
                        "problems": problems or None}
    if problems: log("VERIFY FAILED:", problems)

# ---------------------------------------------------------------------------------------------------------------------------
def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0: return
    import numpy as np
    threads, cpu_note = usable_cpus()
    if args.ref_threads: threads = args.ref_threads
    t0 = time.time()
    tabs = make_inputs(wl, oracle_compressor(wl), threads, pinned=False)
    log("reference arm: inputs ready in %.1fs" % (time.time() - t0))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cassandra_b200 import native
    OL = oracle_api()
    u_in = sum(t.compression.data_length for t in tabs); i_in = sum(t.hold[1].numel() for t in tabs)
    m = build_manifest(tabs, wl)
    nout = 1 if not wl["lcs"] else int(2 * u_in // wl["lcs"]) + 4
    cap_d = u_in + (64 << 20) if not wl["lcs"] else 3 * wl["lcs"] + (64 << 20); cap_i = i_in + (16 << 20); cap_c = u_in // 16384 + 16
    ranges = max(64, threads * 4)
    if wl["lcs"]: thr, max_ranges = 1, 0
    else:
        thr = threads; max_ranges, _ = estimate_max_ranges(u_in, threads, ranges, args.cpu_budget_s)
    res, files = host_out_bufs_numpy(nout, cap_d, cap_i, cap_c)
    for _ in range(args.warmup): cpu_compact(OL, m, res, thr, ranges, max_ranges)
    total = 0.0; covered = 0; rows = 0; tms = [0.0] * 6; hi = INT64_MAX
    for _ in range(args.steps):
        sec, hi, tm = cpu_compact(OL, m, res, thr, ranges, max_ranges)
        total += sec; covered += int(res.bytes_in_range); rows += int(res.total_source_rows); tms = [a + b for a, b in zip(tms, tm)]
    value = covered / total / 1e6
    # scaling curve: constant work per thread (4 of 1024 token ranges each), so the points are comparable
    curve = {}
    if not wl["lcs"]:
        for t in sorted({1, 4, 16, 64, threads, cpu_note["visible_cpus"]}):          # beyond the quota: shows the throttling
            r1, _ = host_out_bufs_numpy(1, cap_d, cap_i, cap_c) if t * 4 >= 512 else host_out_bufs_numpy(1, cap_d // 4 + (8 << 20), cap_i // 4 + (8 << 20), cap_c // 4 + 1024)
            s1, _, _ = cpu_compact(OL, m, r1, t, 1024, min(1024, 4 * t))
            curve[str(t)] = {"MB/s": round(int(r1.bytes_in_range) / s1 / 1e6, 1), "seconds": round(s1, 2)}
        one = curve.get("1", {}).get("MB/s")
        for k, v in curve.items():
            if one: v["efficiency"] = round(v["MB/s"] / (one * int(k)), 3)
    cb = {"value": round(value, 1), "unit": "MB/s", "cores": thr, "kind": "port",
          "sample": ("the whole workload" if hi == INT64_MAX else "token range (MIN, %d] = %.1f %% of the workload's bytes per step" % (hi, 100.0 * covered / args.steps / u_in)) +
                    (", ONE compaction cut into %d token ranges, one oracle thread per range" % ranges if thr > 1 else ", single-threaded oracle"),
          "phase_ms": [round(x / args.steps, 1) for x in tms[:3]], "range_tasks_ms": {"wall_sum": round(tms[3] / args.steps, 1), "thread_cpu_sum": round(tms[4] / args.steps, 1), "longest": round(tms[5] / args.steps, 1)},
          "scaling": curve or None, "host_threads": threads, "host": cpu_note}
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(total / args.steps * 1e3, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": wl["name"] + ", chunk 16 KiB, schema %s, seed %#x" % (wl["schema"], wl["seed"]), "uncompressed_in_bytes": u_in,
                       "reference_arm": "C++ restatement of the reference algorithm (oracle/; the JVM cannot run in this image: no JDK), same inputs as the b200 arm, "
                                        "as many threads as the container's CPU quota allows (cpu_baseline.host) via token-range parallelism; the reference itself runs one such compaction on ONE thread (cpu_baseline.scaling['1'])"},
            "rows_merged_per_s": round(rows / total, 0), "cpu_baseline": cb,
            "e2e": {"value": round(value, 1), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)

_REAL_STDOUT = None
def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n"); out.flush()

def main():
    # the contract is ONE JSON line on stdout: libraries (NCCL prints its version banner there) are diverted to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg1", choices=sorted(WORKLOADS))
    ap.add_argument("--sstables", type=int, default=0, help="override the workload's input count (development)")
    ap.add_argument("--sstable-mib", type=float, default=0.0, help="override the workload's input size (development; the line then says so)")
    ap.add_argument("--rows-per-partition", type=int, default=1000)
    ap.add_argument("--e2e-ranges", default="", help="development aid: also time the e2e path with B200C_RANGES forced to each of these comma-separated values")
    ap.add_argument("--ab-env", default="", help="development aid: NAME=VALUE[,NAME=VALUE]; after the normal measurement, time both legs again with these set")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="bound of one CPU-oracle compaction (cpu_baseline leg and reference arm)")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg AND the verification (development)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the last timed step's output files (a fixed sample of large ones) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1: ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference": ap.error("--dump-outputs writes what the b200 arm computed")
    wl = dict(WORKLOADS[args.workload]); wl["rpp"] = args.rows_per_partition
    if args.sstables or args.sstable_mib:
        if args.sstables: wl["sstables"] = args.sstables
        if args.sstable_mib: wl["mib"] = args.sstable_mib
        wl["name"] = "NOT the named config (scaled for development): %d x %g MiB; " % (wl["sstables"], wl["mib"]) + wl["name"]
    if args.warmup < 3 and args.impl == "b200": log("warning: fewer than 3 warm-up steps")
    if args.impl == "reference": run_reference(args, wl)
    else: run_b200(args, wl)

if __name__ == "__main__":
    main()
