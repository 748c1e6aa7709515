"""The side band of a leveled (multi-file) compaction on the GPU: for every output file that MaxSSTableSizeWriter starts, Filter.db, Summary.db,
first / last key and every b200c_sstable_stats field must equal the CPU oracle's, next to the file's Data.db, Index.db, chunk offsets and
digest. The oracle's per-file values are pinned independently by test_oracle_lcs_metadata.py."""
import ctypes as C, os, subprocess, sys, textwrap, pytest
import numpy as np
import oracle_lib as O
from synth_util import synth_tables
from cassandra_b200.db.compaction import CompactionTask, CompactionController, GpuEngine

NOW = 1700000000
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT64_MAX = (1 << 63) - 1

@pytest.fixture(scope="module")
def ctx():
    from cassandra_b200 import native
    c = native.Context(0)
    yield c
    c.close()

def same_file(g, w):
    assert g.data == w.data and g.index == w.index and g.digest == w.digest
    assert g.compression.chunk_offsets == w.compression.chunk_offsets and g.compression.data_length == w.compression.data_length
    assert (g.partitions, g.rows) == (w.partitions, w.rows)
    assert g.filter == w.filter and g.summary == w.summary and (g.first_key, g.last_key) == (w.first_key, w.last_key)
    for k in w.stats: assert g.stats[k] == w.stats[k], k

def lcs_both(ctx, tables, controller, engine=None, min_files=3, **kw):
    for g, t in enumerate(tables): t.generation = g
    kw.setdefault("with_metadata", True)
    want = CompactionTask(tables, controller, **kw).execute(O.OracleEngine(), max_outputs=64)
    got = CompactionTask(tables, controller, **kw).execute(engine or GpuEngine(ctx), max_outputs=64)
    assert len(want.outputs) >= min_files and len(got.outputs) == len(want.outputs)
    for g, w in zip(got.outputs, want.outputs): same_file(g, w)
    for k in ("bytes_read", "bytes_written", "total_source_rows", "merged_row_counts"): assert got.stats[k] == want.stats[k], k
    return got, want

@pytest.mark.gpu
@pytest.mark.parametrize("limit,n,universe", [(200_000, 6, 30000), (1 << 20, 8, 60000), (50_000, 3, 8000)])
def test_lcs_side_band_matches_oracle(ctx, limit, n, universe):
    tabs = synth_tables(0, n, 0x1C5 + n, universe)
    got, _ = lcs_both(ctx, tabs, CompactionController(NOW), max_sstable_bytes=limit, min_index_interval=16)
    assert all(o.stats["total_tombstones"] > 0 for o in got.outputs)
    lcs_both(ctx, tabs, CompactionController(0, 0), max_sstable_bytes=limit)                  # nothing purged, default sampling

@pytest.mark.gpu
def test_lcs_side_band_wide_partitions(ctx):
    tabs = synth_tables(1, 3, 0x1C9, 120, rows_per_partition=1000, column_index_size=4096)
    lcs_both(ctx, tabs, CompactionController(NOW), min_files=2, max_sstable_bytes=1 << 20, column_index_size=4096)

@pytest.mark.gpu
def test_lcs_side_band_static_complex_counter_tables(ctx):
    from static_tables import static_tables
    from complex_tables import complex_tables
    from counter_tables import counter_tables
    lcs_both(ctx, static_tables(8, ntables=6, nkeys=2000, cis=2048), CompactionController(NOW, 864000), column_index_size=2048, max_sstable_bytes=60000)
    lcs_both(ctx, complex_tables(9, ntables=6, nkeys=2500), CompactionController(NOW, 864000), max_sstable_bytes=60000)
    lcs_both(ctx, complex_tables(4, ntables=40, nkeys=60), CompactionController(NOW, 864000), min_files=2, max_sstable_bytes=8000)    # fan-in above 16
    lcs_both(ctx, counter_tables(9, ntables=6, nkeys=2500), CompactionController(NOW, 864000), max_sstable_bytes=30000)

@pytest.mark.gpu
def test_lcs_side_band_config2_shape(ctx):
    """BASELINE.json configs[2] at reduced scale: 32 Snappy inputs (4 L0 tables over the whole ring + 28 L1 tables in 8 token bands)"""
    tabs = synth_tables(0, 32, 0xCA550003, 40000, p=0.25, comp=O.COMP_SNAPPY, band_count=8, l0_count=4)
    lcs_both(ctx, tabs, CompactionController(NOW), max_sstable_bytes=160 * 1024)

@pytest.mark.gpu
def test_lcs_side_band_device_resident_buffers(ctx):
    from test_gpu_compaction import DeviceEngine
    tabs = synth_tables(0, 5, 0xD38, 30000)
    lcs_both(ctx, tabs, CompactionController(NOW), engine=DeviceEngine(ctx), max_sstable_bytes=100_000, min_index_interval=16)

@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"B200C_K4_WIDE_WARP": "256"}, {"B200C_K4_STAGED": "1"}])
def test_lcs_side_band_k4_variants(ctx, env, monkeypatch):
    for k, v in env.items(): monkeypatch.setenv(k, v)
    lcs_both(ctx, synth_tables(0, 20, 0x1CA, 20000), CompactionController(NOW), max_sstable_bytes=100_000)        # fan-in up to 20: every class
    lcs_both(ctx, synth_tables(1, 3, 0x1CB, 60, rows_per_partition=300, column_index_size=4096), CompactionController(NOW),
             min_files=2, max_sstable_bytes=1 << 18, column_index_size=4096)

@pytest.mark.gpu
def test_lcs_unbounded_limit_equals_single_output(ctx):
    """max_sstable_bytes = Long.MAX_VALUE (a level-0 user-defined task): one file through the multi-file path, the same side band as a
    single-output call"""
    tabs = synth_tables(0, 4, 0x1CC, 20000)
    got, _ = lcs_both(ctx, tabs, CompactionController(NOW), min_files=1, max_sstable_bytes=INT64_MAX, min_index_interval=16)
    one = CompactionTask(tabs, CompactionController(NOW), with_metadata=True, min_index_interval=16).execute(GpuEngine(ctx))
    assert len(got.outputs) == len(one.outputs) == 1
    same_file(got.outputs[0], one.outputs[0])

def raw_call(ctx, tabs, limit, nout, cap_of):
    """b200c_compact with hand-made output slots; cap_of(file, component) -> capacity of that component"""
    from cassandra_b200 import native
    task = CompactionTask(tabs, CompactionController(NOW), max_sstable_bytes=limit, with_metadata=True); m = task.build_manifest()
    res = native.Result(); outs = (native.Output * nout)(); keep = []
    for f in range(nout):
        o = outs[f]
        for name, n in (("data", 8 << 20), ("index", 1 << 20), ("key_buf", cap_of(f, "key")), ("filter", cap_of(f, "filter")), ("summary", cap_of(f, "summary"))):
            b = np.zeros(max(n, 1), dtype=np.uint8); keep.append(b); setattr(o, name, b.ctypes.data)
        co = np.zeros(1 << 12, dtype=np.uint64); keep.append(co)
        o.data_cap, o.index_cap, o.chunk_offsets, o.chunk_cap = 8 << 20, 1 << 20, co.ctypes.data, 1 << 12
        o.key_cap, o.filter_cap, o.summary_cap = cap_of(f, "key"), cap_of(f, "filter"), cap_of(f, "summary")
        st = native.SSTableStats(); keep.append(st); o.stats = C.pointer(st)
    res.noutputs_cap = nout; res.outputs = outs
    rc = native.lib().b200c_compact(ctx.handle, C.byref(m), C.byref(res), 0)
    return rc, res, outs

@pytest.mark.gpu
def test_lcs_side_band_buffers_too_small(ctx):
    from cassandra_b200 import native
    tabs = synth_tables(0, 3, 0x1C8, 8000)
    want = CompactionTask(tabs, CompactionController(NOW), max_sstable_bytes=50_000, with_metadata=True).execute(O.OracleEngine(), max_outputs=64).outputs
    assert len(want) >= 3
    big = lambda f, c: 1 << 20
    rc, res, outs = raw_call(ctx, tabs, 50_000, 64, big)
    assert rc == native.OK and res.noutputs == len(want)
    for comp, attr in (("filter", "filter_len"), ("summary", "summary_len")):
        rc, res, outs = raw_call(ctx, tabs, 50_000, 64, lambda f, c: 16 if (f, c) == (1, comp) else 1 << 20)
        assert rc == native.ETOOSMALL
        need = len(getattr(want[1], comp))
        assert getattr(outs[1], attr) == need > 16                    # the required size of the second file is reported in its slot
        assert getattr(outs[0], attr) == len(getattr(want[0], comp)) and getattr(outs[2], attr) == len(getattr(want[2], comp))
        # the slot that did not fit still reports every other length and gets its statistics
        assert (outs[1].filter_len, outs[1].summary_len) == (len(want[1].filter), len(want[1].summary))
        assert outs[1].stats.contents.total_rows == want[1].stats["total_rows"] > 0
    rc, res, outs = raw_call(ctx, tabs, 50_000, 2, big)             # fewer output slots than files
    assert rc == native.ETOOSMALL

@pytest.mark.gpu
def test_two_pass_mode_still_refuses_the_side_band():
    code = textwrap.dedent('''
        import sys; sys.path.insert(0, "tests"); sys.path.insert(0, ".")
        from synth_util import synth_tables
        from cassandra_b200 import native
        from cassandra_b200.db.compaction import CompactionTask, CompactionController, GpuEngine
        tabs = synth_tables(0, 3, 0x1C7, 8000)
        with native.Context(0) as ctx:
            for limit in (0, 50_000):
                try: CompactionTask(tabs, CompactionController(1700000000), max_sstable_bytes=limit, with_metadata=True).execute(GpuEngine(ctx), max_outputs=64)
                except native.UnsupportedError: continue
                raise SystemExit("side band accepted under B200C_K4_TWO_PASS, limit %d" % limit)
        print("ok")
    ''')
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, B200C_K4_TWO_PASS="1"), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-1000:] + r.stderr[-2000:]

def test_java_shim_has_the_leveled_hooks():
    d = os.path.join(ROOT, "java", "org", "apache", "cassandra", "db", "compaction")
    lcs = open(os.path.join(d, "GpuLeveledCompactionStrategy.java")).read()
    assert "extends LeveledCompactionStrategy" in lcs and "GpuCompactionTask" in lcs
    task = open(os.path.join(d, "GpuCompactionTask.java")).read()
    assert "putLong(M_MAX_SSTABLE_BYTES, maxSSTableBytes)" in task and "putLong(M_MAX_SSTABLE_BYTES, 0L)" not in task
    assert "int level, long maxSSTableBytes" in task                     # the leveled constructor
    assert "new MaxSSTableSizeWriter(" in task                          # the stock path of a leveled task (EUNSUPPORTED fallback) keeps the file limit
