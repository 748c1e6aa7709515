"""Pins the CPU oracle's side band per output file of a leveled (multi-file) compaction: Filter.db, Summary.db, first / last key and the
MetadataCollector reductions of every file that MaxSSTableSizeWriter starts (S/db/compaction/writers/MaxSSTableSizeWriter.java:76-79).
Nothing here trusts the oracle's Meta: Filter.db and Summary.db are rebuilt from the file's own Index.db, and the statistics of the files
are combined and compared with the same compaction written as one file (partition records do not depend on where a file starts)."""
import bisect, math, struct, pytest
import oracle_lib as O
from synth_util import synth_tables
from test_golden_murmur3 import bloom_bytes
from cassandra_b200.io.sstable import _vint
from cassandra_b200.db.compaction import CompactionTask, CompactionController

NOW = 1700000000
ADDITIVE = ("total_rows", "total_columns_set", "total_cells", "total_tombstones")

def index_entries(ix, with_positions=False):
    """(Index.db offset, key[, Data.db position]) of every entry: u16 keyLen | key | vint position | vint32 payload size | payload
    (RowIndexEntry.serialize)"""
    o = 0; out = []
    while o < len(ix):
        kl = (ix[o] << 8) | ix[o + 1]; key = bytes(ix[o + 2:o + 2 + kl]); p = o + 2 + kl
        dpos, p = _vint(ix, p); ps, p = _vint(ix, p)
        out.append((o, key, dpos) if with_positions else (o, key)); o = p + ps
    return out

def histogram_offsets(n):
    """EstimatedHistogram.newOffsets(n, false): 1, then round(last * 1.2), at least last + 1 (Math.round: half up)"""
    r = [1]
    while len(r) < n:
        nxt = int(math.floor(r[-1] * 1.2 + 0.5)); r.append(nxt if nxt != r[-1] else nxt + 1)
    return r

def size_histogram(o):
    """estimatedPartitionSize of one file from its own files: partition sizes are the gaps between the Data.db positions in Index.db"""
    pos = [p for _, _, p in index_entries(o.index, True)] + [o.compression.data_length]
    offs = histogram_offsets(155); hist = [0] * 156
    for a, b in zip(pos, pos[1:]): hist[bisect.bisect_left(offs, b - a)] += 1
    return hist

def summary_bytes(entries, interval):
    """IndexSummaryBuilder at full sampling (every interval-th key, with its Index.db position as a native long) + IndexSummarySerializer
    + first / last key, rebuilt from the entries alone"""
    samples = [k + struct.pack("<q", pos) for i, (pos, k) in enumerate(entries) if i % interval == 0]
    n = len(samples); body = b"".join(samples)
    offs, acc = [], 0
    for s in samples: offs.append(acc + 4 * n); acc += len(s)
    first, last = entries[0][1], entries[-1][1]
    return (struct.pack(">iiqii", interval, n, 4 * n + len(body), 128, (len(entries) + interval - 1) // interval)
            + b"".join(struct.pack("<I", v) for v in offs) + body
            + struct.pack(">i", len(first)) + first + struct.pack(">i", len(last)) + last)

def run(tabs, controller, limit, **kw):
    return CompactionTask(tabs, controller, max_sstable_bytes=limit, with_metadata=True, **kw).execute(O.OracleEngine(), max_outputs=64)

def check_files_against_single(tabs, controller, limit, interval, **kw):
    multi = run(tabs, controller, limit, min_index_interval=interval, **kw)
    single = run(tabs, controller, 0, min_index_interval=interval, **kw)
    assert len(multi.outputs) >= 3 and len(single.outputs) == 1
    one = single.outputs[0]
    # every file on its own: Filter.db and Summary.db from its Index.db
    for o in multi.outputs:
        ent = index_entries(o.index)
        assert len(ent) == o.partitions > 0
        hc, words = struct.unpack_from(">ii", o.filter, 0)
        assert o.filter[8:] == bloom_bytes([k for _, k in ent], hc, words)
        assert (hc, words) == struct.unpack_from(">ii", one.filter, 0)          # the same geometry for every file
        assert (o.first_key, o.last_key) == (ent[0][1], ent[-1][1])
        assert o.summary == summary_bytes(ent, interval)
        st = o.stats
        assert sum(st["partition_size_hist"]) == o.partitions == sum(st["cells_per_partition_hist"])
        assert st["partition_size_hist"] == size_histogram(o)                     # per file, from the file itself: no partition in the wrong file
    # the files together = the compaction written as one file
    s1 = one.stats; sts = [o.stats for o in multi.outputs]
    assert sum(o.partitions for o in multi.outputs) == one.partitions and sum(o.rows for o in multi.outputs) == one.rows
    for k in ADDITIVE: assert sum(s[k] for s in sts) == s1[k], k
    for k in ("partition_size_hist", "cells_per_partition_hist"): assert [sum(v) for v in zip(*(s[k] for s in sts))] == s1[k], k
    # tombstone drop times: a list that overflowed holds the smallest points only, so it is complete up to its last point
    cut = min([s["tombstone_drop_times"][-1][0] for s in sts + [s1] if s["tdrop_overflow"]] or [1 << 63])
    td = {}
    for s in sts:
        for p, c in s["tombstone_drop_times"]:
            if p <= cut: td[p] = td.get(p, 0) + c
    assert sorted(td.items()) == [(p, c) for p, c in s1["tombstone_drop_times"] if p <= cut] and len(td) > 16
    for k in ("min_timestamp", "min_local_deletion_time", "min_ttl"): assert min(s[k] for s in sts) == s1[k], k
    for k in ("max_timestamp", "max_local_deletion_time", "max_ttl"): assert max(s[k] for s in sts) == s1[k], k
    for k in ("has_partition_level_deletions", "has_legacy_counter_shards"): assert max(s[k] for s in sts) == s1[k], k
    assert bytes(max(v) for v in zip(*(s["hll_registers"] for s in sts))) == s1["hll_registers"]
    assert (multi.outputs[0].first_key, multi.outputs[-1].last_key) == (one.first_key, one.last_key)
    return multi, single

@pytest.mark.parametrize("interval", [16, 128])
def test_narrow_partitions_per_file_side_band(interval):
    tabs = synth_tables(0, 4, 0x1C5A, 8000)
    multi, single = check_files_against_single(tabs, CompactionController(NOW), 50_000, interval)
    st = single.outputs[0].stats
    assert st["total_tombstones"] > 0 and st["max_ttl"] > 0 and st["tombstone_drop_times"]      # the shapes the side band must carry
    check_files_against_single(tabs, CompactionController(0, 0), 50_000, interval)              # nothing purged: other tombstone / TTL paths

@pytest.mark.parametrize("interval", [16, 128])
def test_wide_partitions_per_file_side_band(interval):
    tabs = synth_tables(1, 3, 0x1C5B, 60, rows_per_partition=300, column_index_size=4096)
    check_files_against_single(tabs, CompactionController(NOW), 1 << 18, interval, column_index_size=4096)
