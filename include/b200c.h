/*
 * b200c.h — C ABI of libb200compact.so: the B200-native (sm_100a) SSTable compaction engine.
 *
 * This is the drop-in boundary a JNI (or JNA) shim in org.apache.cassandra.{db.compaction, io.compress} binds.
 * Plain pointers and sizes only. All host pointers are caller-owned (ideally pinned / registered DirectByteBuffers,
 * see b200c_host_register); results are written into caller-provided buffers. The library is re-entrant: one
 * b200c_ctx per calling thread (one per CompactionExecutor thread), each with its own CUDA stream and workspace.
 * No callbacks into the caller. No CPU fallback: without a CUDA device every entry point fails with B200C_ECUDA.
 *
 * Reference interfaces replaced (S/ = src/java/org/apache/cassandra/ in apache/cassandra @ 7446529e):
 *   b200c_compact              <- CompactionTask.runMayThrow hot loop              S/db/compaction/CompactionTask.java:184-236
 *                                 (CompactionIterator S/db/compaction/CompactionIterator.java:122-160 over ISSTableScanner
 *                                  S/io/sstable/ISSTableScanner.java:34-41, into CompactionAwareWriter.append
 *                                  S/db/compaction/writers/CompactionAwareWriter.java:138-142)
 *   b200c_compress_chunks      <- CompressedSequentialWriter.flushData             S/io/compress/CompressedSequentialWriter.java:140-206
 *                                 + ChecksumWriter.appendDirect                    S/io/util/ChecksumWriter.java:62-89
 *                                 + CompressionMetadata.Writer.addOffset           S/io/compress/CompressionMetadata.java:366-375
 *   b200c_decompress_chunks    <- CompressedChunkReader.readChunk                  S/io/util/CompressedChunkReader.java:103-173
 *   b200c_compress / _uncompress <- ICompressor.compress / uncompress              S/io/compress/ICompressor.java:28-86
 *                                 (LZ4Compressor S/io/compress/LZ4Compressor.java:113-190, SnappyCompressor.java:77-105)
 *   b200c_poll / b200c_cancel  <- CompactionInfo.Holder progress + isStopRequested S/db/compaction/CompactionIterator.java:167-176,709-742
 */
#ifndef B200C_H
#define B200C_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200C_ABI_VERSION 2

/* return codes (0 = success). The shim maps them to the reference's exceptions:
 * ECORRUPT -> CorruptSSTableException + markSuspect, ECANCELLED -> CompactionInterruptedException,
 * EUNSUPPORTED -> fall back to scheduling a stock CompactionTask (decision of the Java strategy, not of this library). */
enum {
    B200C_OK = 0,
    B200C_EINVAL = -1,        /* bad argument */
    B200C_ECUDA = -2,         /* CUDA error / no device; b200c_last_error has the text */
    B200C_ECORRUPT = -3,      /* checksum mismatch or malformed input; see b200c_corruption */
    B200C_ECANCELLED = -4,
    B200C_EUNSUPPORTED = -5,  /* schema/feature outside the supported envelope (multi-cell static columns, non-frozen UDTs, shadowable deletions, a counter context the reference never writes inside a merge ...) */
    B200C_ENOMEM = -6,        /* device or host workspace exhausted */
    B200C_ETOOSMALL = -7      /* a caller-provided output buffer is too small; required sizes are reported */
};

/* SNAPPY: raw snappy as snappy-java 1.1.10.4 / Google snappy 1.1.x writes it (hash table of at most 2^14 entries). SNAPPY15: the same format
 * written by Google snappy >= 1.2.0 (hash table of at most 2^15 entries: different, equally valid bytes; what newer snappy-java bundles, and the
 * generation tests/golden/snappy pins against the real library). Decompression is identical for both. */
enum { B200C_COMP_NONE = 0, B200C_COMP_LZ4 = 1, B200C_COMP_SNAPPY = 2, B200C_COMP_SNAPPY15 = 3 };
/* IPartitioner of the table (ValidationMetadata.partitioner, S/io/sstable/metadata/ValidationMetadata.java): decides the partition
 * order every input must already be in and the output is written in (DecoratedKey.compareTo, S/db/DecoratedKey.java:79-91).
 *   MURMUR3       S/dht/Murmur3Partitioner.java:256-296 — signed 64-bit token, ties by unsigned key bytes
 *   BYTE_ORDERED  S/dht/ByteOrderedPartitioner.java — the token IS the key: unsigned lexicographic key order. token_lo / token_hi
 *                 must span the whole ring (sub-ranges of a byte-ordered ring are not expressible as int64 and are refused).
 * Anything else (RandomPartitioner, LocalPartitioner, OrderPreservingPartitioner) -> B200C_EUNSUPPORTED. An input whose Index.db is
 * not in the stated order is B200C_ECORRUPT whatever its size. */
enum { B200C_PARTITIONER_MURMUR3 = 0, B200C_PARTITIONER_BYTE_ORDERED = 1 };

typedef struct b200c_ctx b200c_ctx;

typedef struct b200c_corruption {
    int32_t  input;           /* index of the input sstable (0 for the codec entry points) */
    int32_t  kind;            /* 1 = chunk CRC mismatch, 2 = malformed compressed chunk, 3 = malformed Index.db, 4 = malformed Data.db */
    uint64_t chunk;           /* chunk index */
    uint64_t offset;          /* byte offset in the component file */
} b200c_corruption;

/* ---- lifecycle ------------------------------------------------------------------------------------------------ */
int          b200c_abi_version(void);
int          b200c_device_count(void);
/* device: CUDA ordinal. workspace_bytes: initial device workspace (0 = grow on demand). NULL on failure. */
b200c_ctx*   b200c_create(int device, size_t workspace_bytes);
void         b200c_destroy(b200c_ctx*);
const char*  b200c_last_error(b200c_ctx*);
/* pin/unpin caller memory (DirectByteBuffer addresses) so cudaMemcpyAsync runs at PCIe speed */
int          b200c_host_register(void* p, size_t n);
int          b200c_host_unregister(void* p);
/* device memory helpers for callers that keep buffers resident in HBM (bench `value`, GPU-side pipelines) */
int          b200c_dev_alloc(b200c_ctx*, size_t n, void** dptr);
int          b200c_dev_free(b200c_ctx*, void* dptr);
int          b200c_memcpy_h2d(b200c_ctx*, void* dst_dev, const void* src_host, size_t n);
int          b200c_memcpy_d2h(b200c_ctx*, void* dst_host, const void* src_dev, size_t n);
int          b200c_sync(b200c_ctx*);
/* elapsed device time (ms, CUDA events on the ctx stream) of the kernels of the last call, and how many launched */
double       b200c_last_kernel_ms(b200c_ctx*);
uint64_t     b200c_last_kernel_launches(b200c_ctx*);
uint64_t     b200c_total_kernel_launches(b200c_ctx*);
/* device time (ms) of the stages of the last b200c_compact: [0] K1 decompress+verify, [1] K2 index scan, [2] K3 partition merge,
 * [3] K4 size pass, [4] K4 emit pass, [5] K5 compress+CRC+pack. Returns the number of entries written (<= n). */
int          b200c_last_stage_ms(b200c_ctx*, double* out, int n);

/* ---- chunk codec: the CompressedSequentialWriter / CompressedChunkReader data plane, batched ---------------------
 * b200c_compress_chunks: `in[0..n)` is an uncompressed Data stream. Chunk i = bytes [i*chunk_len, min((i+1)*chunk_len, n)).
 * Writes the Data.db image to `out`: for every chunk the compressor output (LZ4: 4-byte LE length + block) followed by the
 * 4-byte big-endian CRC32 of the bytes as written; chunk_offsets[i] = file offset of chunk i (CompressionInfo.db payload);
 * *digest = CRC32 of the whole image (Digest.crc32). If compressed_len >= max_compressed_len the chunk is stored raw
 * (padded with zeroes up to max_compressed_len when shorter) exactly as flushData does; pass INT32_MAX for the default
 * min_compress_ratio = 0. `out_cap` must be >= b200c_compress_bound(...). `flags` bit0: in/out/chunk_offsets are DEVICE pointers.
 * DEVICE pointers (B200C_FLAG_DEVICE_PTRS, here and in every other entry point): the kernels read whole aligned 16-byte words, so
 * every caller-owned device buffer must be 16-byte aligned and keep >= B200C_DEVICE_SLACK readable (for outputs: writable) bytes
 * behind its last used byte. b200c_dev_alloc adds that slack itself; plain cudaMalloc'ed buffers must be sized accordingly. */
#define B200C_DEVICE_SLACK 256
uint64_t     b200c_compress_bound(int compressor, uint64_t n, int chunk_len);
uint64_t     b200c_chunk_count(uint64_t n, int chunk_len);
int          b200c_compress_chunks(b200c_ctx*, int compressor, const uint8_t* in, uint64_t n, int chunk_len,
                                   int max_compressed_len, uint8_t* out, uint64_t out_cap, uint64_t* out_len,
                                   uint64_t* chunk_offsets, uint32_t* digest, int flags);
/* b200c_decompress_chunks: inverse. `data` is a Data.db image, `chunk_offsets[nchunks]` from CompressionInfo.db,
 * `data_length` the uncompressed length. Verifies every chunk CRC when verify_crc != 0 (crc_check_chance = 1.0).
 * On B200C_ECORRUPT *where (optional) describes the first bad chunk. flags bit0: data/chunk_offsets/out are DEVICE pointers. */
int          b200c_decompress_chunks(b200c_ctx*, int compressor, const uint8_t* data, uint64_t data_len,
                                     const uint64_t* chunk_offsets, uint64_t nchunks, int chunk_len, int max_compressed_len,
                                     uint64_t data_length, uint8_t* out, int verify_crc, b200c_corruption* where, int flags);
#define B200C_FLAG_DEVICE_PTRS 1

/* ICompressor single-buffer contract (degenerate one-chunk batch; PCIe-latency bound — the batched calls are the fast path).
 * Return the number of bytes written to `out`, or a negative error code. */
int          b200c_initial_compressed_buffer_length(int compressor, int chunk_len);
int          b200c_compress(b200c_ctx*, int compressor, const uint8_t* in, int n, uint8_t* out, int out_cap);
int          b200c_uncompress(b200c_ctx*, int compressor, const uint8_t* in, int n, uint8_t* out, int out_cap);

/* ---- compaction ---------------------------------------------------------------------------------------------- */

/* comparison / layout class of a CQL type, as AbstractType exposes it (S/db/marshal/AbstractType.java:66-82,212-215,490,535-552) */
enum {
    B200C_TYPE_BYTES = 0,     /* variable length, unsigned lexicographic compare (text, ascii, blob, varchar) */
    B200C_TYPE_FIXED_SIGNED = 1, /* fixed length big-endian two's complement, signed compare (bigint 8, int 4, smallint 2, tinyint 1, timestamp 8) */
    B200C_TYPE_FIXED_BYTES = 2,  /* fixed length, unsigned lexicographic compare (boolean 1, and any fixed type used only as a value) */
    B200C_TYPE_VAR_SIGNED = 3,   /* variable length payload holding a fixed-width signed int: empty value sorts first (LongType with empty) */
    B200C_TYPE_TIMEUUID = 4,     /* 16 bytes, TimeUUIDType.compareCustom (S/db/marshal/TimeUUIDType.java): timestamp fields first — cell paths of lists only */
    B200C_TYPE_COUNTER = 5       /* CounterColumnType: variable length counter context (S/db/context/CounterContext.java:40-76); live cells of the same
                                    row are MERGED shard by shard (Cells.resolveCounter S/db/rows/Cells.java:121-162) instead of picked. Regular
                                    and static simple columns. */
};
/* A multi-cell (complex) column — non-frozen map / set / list — stores one cell per element, each with a CELL PATH (the map key, the set
 * element, the list's timeuuid), and an optional complex deletion (S/db/rows/ComplexColumnData.java, UnfilteredSerializer.java:271-280,
 * Cell.java:268-305). Same struct, no layout change: `type` carries the class of the cell VALUES in bits 0-7 and, for a complex column,
 * 1 + the class of the cell PATHS in bits 8-15 (0 = simple column); `fixed_len` the values' fixed length in bits 0-15 and the paths'
 * in bits 16-31. In a SerializationHeader the simple columns come first, then the complex ones, each group in name order
 * (ColumnMetadata.comparisonOrder): column_map must follow that order. Complex static columns and non-frozen UDTs are refused. */
#define B200C_COLUMN_COMPLEX(value_type, path_type) ((value_type) | (((path_type) + 1) << 8))
#define B200C_COLUMN_FIXED(value_len, path_len)     ((value_len) | ((path_len) << 16))
enum { B200C_MAX_COMPLEX_COLUMNS = 8 };

typedef struct b200c_column {
    int32_t  type;            /* B200C_TYPE_* (complex columns: B200C_COLUMN_COMPLEX) */
    int32_t  fixed_len;       /* value length in bytes if fixed, else 0 (AbstractType.valueLengthIfFixed); complex columns: B200C_COLUMN_FIXED */
} b200c_column;

typedef struct b200c_encoding_stats {   /* S/db/rows/EncodingStats.java: base values the deltas in the files are against */
    int64_t  min_timestamp;
    int64_t  min_local_deletion_time;   /* widened; as EncodingStats.minLocalDeletionTime */
    int32_t  min_ttl;
    int32_t  _pad;
} b200c_encoding_stats;

#define B200C_MAX_CLUSTERING 8
#define B200C_MAX_COLUMNS    64
#define B200C_MAX_INPUTS     64      /* fan-in of one call (one or two sources per lane of the merge warp) */
#define B200C_MAX_STATIC_COLUMNS 16

typedef struct b200c_input {
    const uint8_t*  data;               /* Data.db image (compressed chunks + inline CRCs) */
    uint64_t        data_len;
    const uint8_t*  index;              /* Index.db image */
    uint64_t        index_len;
    const uint64_t* chunk_offsets;      /* CompressionInfo.db chunk offsets */
    uint64_t        nchunks;
    uint64_t        data_length;        /* uncompressed length (CompressionInfo.db dataLength) */
    int32_t         compressor;         /* B200C_COMP_* */
    int32_t         chunk_len;
    int32_t         max_compressed_len; /* INT32_MAX when min_compress_ratio = 0 */
    int32_t         ncolumns;           /* regular columns in this sstable's SerializationHeader, in header order */
    int32_t         column_map[B200C_MAX_COLUMNS]; /* header column i -> index in manifest.columns (output header) */
    b200c_encoding_stats header_stats;  /* SerializationHeader.Component stats used to DEcode this input */
    int32_t         _pad;
    int32_t         level;              /* informational (LCS level) */
    /* Summary.db (IndexSummary, S/io/sstable/indexsummary/IndexSummary.java:190-193 getPosition): Index.db offsets of the sampled
       entries, ascending, the first one 0. They are what BigTableScanner seeks with (S/io/sstable/format/big/BigTableScanner.java:
       105-132); here they seed the parallel Index.db walk, whose result is still proven against the sequential parse. Optional
       (NULL / 0): without them the walk has to speculate on entry starts with the help of Data.db, and host-buffer compactions
       cannot overlap their Data.db copies with the kernels (no token-range streaming). */
    const uint64_t* summary_positions;
    uint64_t        nsummary;
    /* static columns in this sstable's SerializationHeader (header.hasStatic() <=> nstatic_columns > 0: every partition then carries a
       static row right after its partition deletion, S/io/sstable/format/SortedTablePartitionWriter.java:97-126), header order */
    int32_t         nstatic_columns;
    int32_t         static_column_map[B200C_MAX_STATIC_COLUMNS]; /* header static column i -> index in manifest.static_columns */
    int32_t         _pad2;
} b200c_input;

typedef struct b200c_manifest {
    uint32_t        abi_version;        /* B200C_ABI_VERSION */
    int32_t         ninputs;
    const b200c_input* inputs;
    /* schema: partition key is opaque bytes ordered by (Murmur3 token, unsigned bytes) — S/db/DecoratedKey.java:79-91 */
    int32_t         nclustering;
    b200c_column    clustering[B200C_MAX_CLUSTERING];
    int32_t         ncolumns;           /* regular simple columns of the OUTPUT header (union of inputs), header order */
    b200c_column    columns[B200C_MAX_COLUMNS];
    int32_t         nstatic_columns;    /* static simple columns of the OUTPUT header (0: the table has none and no static rows are written) */
    /* output encoding: SerializationHeader.make (S/db/SerializationHeader.java:77-100) = min over inputs' StatsMetadata */
    b200c_encoding_stats out_stats;
    int32_t         out_compressor;
    int32_t         out_chunk_len;
    int32_t         out_max_compressed_len;
    int32_t         column_index_size;  /* bytes; 65536 default for big format (BigFormatPartitionWriter.java:49,73) */
    /* determinism inputs (SURVEY §5): */
    int64_t         now_in_sec;         /* CompactionTask.java:183 */
    int64_t         gc_before;          /* CompactionManager.java:2001-2006 */
    int64_t         purge_max_timestamp;/* getPurgeEvaluator threshold: tombstones purgeable iff timestamp < this. INT64_MAX = no overlaps */
    int32_t         tombstone_option;   /* must be 0 (NONE) */
    int32_t         enforce_strict_liveness; /* must be 0 */
    /* token range (lo, hi] handled by this call; lo = INT64_MIN and hi = INT64_MAX for the whole ring */
    int64_t         token_lo;
    int64_t         token_hi;
    /* LCS: switch output file when on-disk bytes exceed this (MaxSSTableSizeWriter.java:76-79); 0 = single output. A multi-file call
       returns one b200c_output per file, each with its own side band (Filter.db, Summary.db, first / last key, b200c_sstable_stats) as
       that file's writer would have gathered it; INT64_MAX (a level-0 user-defined LCS task) = one file through the same path */
    uint64_t        max_sstable_bytes;
    int32_t         partitioner;        /* B200C_PARTITIONER_* */
    /* optional purge table (CompactionController.getPurgeEvaluator is per partition key, S/db/compaction/CompactionController.java:
       247-286: the minimum timestamp over the overlapping sstables that may contain the key). The host buckets the ring: partitions
       with token <= purge_range_hi[k] (first such k, the array ascending) use purge_range_max_ts[k] instead of purge_max_timestamp;
       tokens above the last bound use purge_max_timestamp. npurge_ranges = 0: one threshold for the whole call. HOST pointers always. */
    int32_t         npurge_ranges;
    const int64_t*  purge_range_hi;
    const int64_t*  purge_range_max_ts;
    /* Filter.db geometry, decided by the host as FilterFactory.getFilter(estimatedKeys, fpChance) does (S/utils/FilterFactory.java:
       60-75, BloomCalculations): K hash functions over bloom_words 64-bit words, per output file. 0 words = no filter (fpChance 1.0).
       The same geometry applies to every file of a multi-file call: MaxSSTableSizeWriter sizes each writer's filter for
       sstableKeyCount() = estimatedTotalKeys / estimatedSSTables, the same for all of them (CompactionAwareWriter.java:230-250). */
    int32_t         bloom_hash_count;
    int32_t         min_index_interval; /* Summary.db sampling (128 default, S/schema/TableParams.java); 0 = 128 */
    uint64_t        bloom_words;
    b200c_column    static_columns[B200C_MAX_STATIC_COLUMNS];
} b200c_manifest;

/* What MetadataCollector gathers while an output is written (S/io/sstable/metadata/MetadataCollector.java:107-147,208-270; called
 * from SortedTableWriter.startPartition/addRow/addRangeTomstoneMarker/endPartition, S/io/sstable/format/SortedTableWriter.java:
 * 183-258, and Rows.collectStats S/db/rows/Rows.java:102-113): the per-cell / per-row / per-partition reductions the Java side
 * needs to finish Statistics.db (StatsMetadata + CompactionMetadata) WITHOUT re-reading the output. Trackers that saw no value
 * hold MetadataCollector's defaults (timestamps: INT64_MIN / INT64_MAX; local deletion times: INT64_MAX both; TTLs: 0 both). */
#define B200C_PSIZE_BUCKETS 156     /* EstimatedHistogram(155): 155 bucket offsets + overflow (MetadataCollector.defaultPartitionSizeHistogram :68-72) */
#define B200C_CELLS_BUCKETS 119     /* EstimatedHistogram(118) (defaultCellPerPartitionCountHistogram :62-66) */
#define B200C_HLL_P 13              /* HyperLogLogPlus(13, 25), MetadataCollector.java:139-145 */
#define B200C_TDROP_CAP 512
typedef struct b200c_sstable_stats {
    int64_t  min_timestamp, max_timestamp;                        /* timestampTracker */
    int64_t  min_local_deletion_time, max_local_deletion_time;    /* localDeletionTimeTracker */
    int32_t  min_ttl, max_ttl;                                    /* ttlTracker */
    uint64_t total_rows, total_columns_set;                       /* updateColumnSetPerRow */
    uint64_t total_cells;                                         /* sum of currentPartitionCells */
    uint64_t total_tombstones;                                    /* updateTombstoneCount over the whole file */
    int32_t  has_partition_level_deletions;
    int32_t  tdrop_overflow;                                      /* more than B200C_TDROP_CAP distinct rounded drop times: tdrop_* hold the first CAP */
    uint64_t partition_size_hist[B200C_PSIZE_BUCKETS];            /* estimatedPartitionSize.add(rowSize) per partition */
    uint64_t cells_per_partition_hist[B200C_CELLS_BUCKETS];       /* estimatedCellPerPartitionCount */
    /* estimatedTombstoneDropTime input: exact multiset of local deletion times rounded UP to TOMBSTONE_HISTOGRAM_TTL_ROUND_SECONDS
       (60 s, StreamingTombstoneHistogramBuilder.update), ascending; the shim replays them into the stock builder */
    uint32_t ntdrop;
    uint32_t has_legacy_counter_shards;                           /* updateHasLegacyCounterShards :352-355: a written counter cell holds a local or remote shard */
    int64_t  tdrop_point[B200C_TDROP_CAP];
    uint64_t tdrop_count[B200C_TDROP_CAP];
    /* HyperLogLog++ dense registers (p = 13: 8192 six-bit registers, one per byte here) over MurmurHash.hash2_64(key, seed 0)
       (MetadataCollector.addKey :160-166): register[h >>> 51] = max(1 + numberOfLeadingZeros((h << 13) | (1 << 12))) */
    uint8_t  hll_registers[1 << B200C_HLL_P];
} b200c_sstable_stats;

typedef struct b200c_output {           /* one output sstable (one per file of a multi-file call, each with its own side band); caller provides the buffers */
    uint8_t*  data;        uint64_t data_cap;     uint64_t data_len;      /* Data.db image */
    uint8_t*  index;       uint64_t index_cap;    uint64_t index_len;     /* Index.db image */
    uint64_t* chunk_offsets; uint64_t chunk_cap;  uint64_t nchunks;       /* CompressionInfo.db chunk offsets */
    uint64_t  data_length;                                                /* uncompressed length */
    uint32_t  digest;                                                     /* Digest.crc32 value */
    uint32_t  _pad;
    uint64_t  partitions;                                                 /* partitions written */
    uint64_t  rows;                                                       /* rows + markers written */
    /* ---- the rest of the sstable (SURVEY §8 f1), all optional: a NULL pointer skips that component. HOST pointers always.
       outputs[0] decides which components the call computes; in a multi-file call every slot gets its file's own. Capacities are
       checked per slot: a slot too small for its key / filter / summary makes the call return B200C_ETOOSMALL with the lengths that
       slot needs in *_len. Refused (B200C_EUNSUPPORTED) under the two-pass K4 A/B mode (B200C_K4_TWO_PASS). ---- */
    /* first / last partition key written (SortedTableWriter.endPartition :247-250; StatsMetadata.firstKey/lastKey, Summary.db tail):
       key_buf receives first key then last key back to back; lengths below. Needs key_cap >= first_key_len + last_key_len
       (2 * 65535 always suffices). */
    uint8_t*  key_buf;     uint64_t key_cap;      uint32_t first_key_len; uint32_t last_key_len;
    /* Filter.db image: i32 hashCount | i32 wordCount | bitset bytes (BloomFilterSerializer.serialize S/utils/BloomFilterSerializer.java:
       50-55, OffHeapBitSet.serialize S/utils/obs/OffHeapBitSet.java:115-119), every written key added as BloomFilter.add does
       (S/utils/BloomFilter.java:79-122). Geometry comes from the manifest (bloom_hash_count, bloom_words). */
    uint8_t*  filter;      uint64_t filter_cap;   uint64_t filter_len;
    /* Summary.db image (IndexSummary.IndexSummarySerializer.serialize S/io/sstable/indexsummary/IndexSummary.java:401-423 followed by
       first and last key with int length, SSTableReader/IndexSummaryComponent): one sample every manifest.min_index_interval
       Index.db entries (IndexSummaryBuilder.maybeAddEntry S/io/sstable/indexsummary/IndexSummaryBuilder.java:200-228) */
    uint8_t*  summary;     uint64_t summary_cap;  uint64_t summary_len;
    b200c_sstable_stats* stats;
} b200c_output;

typedef struct b200c_result {
    int32_t   noutputs_cap;             /* in: entries in outputs[] */
    int32_t   noutputs;                 /* out */
    b200c_output* outputs;
    uint64_t  bytes_read;               /* uncompressed length of every input (metric numerator of a whole-ring task, CompactionTask.java:258) */
    uint64_t  bytes_in_range;           /* uncompressed bytes of the input partitions inside (token_lo, token_hi] = what ranged scanners
                                           report as getLengthInBytes (S/io/sstable/format/SSTableScanner.java); = bytes_read for the whole ring */
    uint64_t  bytes_written;            /* uncompressed output bytes */
    uint64_t  total_source_rows;        /* rows + markers read, CompactionIterator.totalSourceCQLRows :368 */
    uint64_t  input_partitions;
    uint64_t  merged_row_counts[B200C_MAX_INPUTS]; /* [i] = output partitions merged from i+1 inputs, CompactionIterator.java:188-197 */
    uint64_t  required_data_cap;        /* set on B200C_ETOOSMALL */
    uint64_t  required_index_cap;
    uint64_t  required_chunk_cap;
    b200c_corruption corruption;        /* set on B200C_ECORRUPT */
    double    kernel_ms;                /* device time of all kernels of this call */
    double    total_ms;                 /* host wall time of the call incl. copies */
    uint64_t  kernel_launches;
    uint64_t  index_slow_path_inputs;   /* inputs whose Index.db speculation could not be proven and were walked sequentially on the GPU */
} b200c_result;

/* flags: bit0 = input/outputs buffers are DEVICE pointers (inputs resident in HBM; used for the kernel-only metric).
   With HOST buffers, one output file (max_sstable_bytes == 0) and summary_positions on every input, the call streams: the token range
   is cut into pieces at tokens of Summary.db samples, and piece by piece the Index.db slice between the samples that bracket the
   piece (what a ranged scanner seeks to, SSTableReader.getPositionsForRanges), its Summary positions and the Data.db chunks it
   describes are copied while earlier pieces are already being parsed, merged, compressed and copied back (pin the buffers with
   b200c_host_register, pageable memory serialises the copies). Every output byte is the same as in the one-piece run. Summary
   positions stay hints: if they do not parse or their slices do not tile the file the call runs as one piece; a slice whose first
   entry lies inside the piece's token range (samples that lie about their tokens) is refused with B200C_ECORRUPT.
   Buffers must stay valid until the call returns; nothing is in flight afterwards, whatever the return code. */
int          b200c_compact(b200c_ctx*, const b200c_manifest*, b200c_result*, int flags);

/* the order token the engine derives from a partition key (host function, no device needed): Murmur3Partitioner.getToken
 * (S/dht/Murmur3Partitioner.java:256-296) or, for ByteOrderedPartitioner, the sign-flipped big-endian 8-byte key prefix. For hosts that
 * pick token-range splitters from Summary.db sample keys (one compaction sharded over several GPUs: token_lo / token_hi per shard). */
int64_t      b200c_token(int partitioner, const uint8_t* key, uint32_t len);

/* call_seq: number of b200c_compact calls this context has started; it changes after the counters were reset for the new call, so a poller that
   remembers it can tell the running call's figures from the final state of the previous one */
typedef struct b200c_progress { uint64_t bytes_scanned; uint64_t bytes_total; int32_t stage; int32_t call_seq; } b200c_progress;
int          b200c_poll(b200c_ctx*, b200c_progress*);   /* callable from another thread */
/* ISSTableScanner.getCurrentPosition per input (S/io/sstable/ISSTableScanner.java:34-41, consumed by CompactionIterator.java:289-295):
 * positions[i] = uncompressed Data.db bytes of input i the merge has consumed so far (it advances token range by token range).
 * Writes min(n, ninputs of the running / last call) entries and returns that count. Callable from another thread. */
int          b200c_poll_inputs(b200c_ctx*, uint64_t* positions, int n);
/* callable from another thread; the running b200c_compact returns B200C_ECANCELLED at its next stage boundary with nothing in
 * flight. The request is STICKY: a cancel that lands just before the call starts cancels that call (isStopRequested() can turn true
 * any time after the task was registered, S/db/compaction/CompactionIterator.java:709-742). It is consumed by the call that reports
 * it; the shim calls b200c_cancel_reset when it binds a NEW task to the context, before that task can be stopped. */
void         b200c_cancel(b200c_ctx*);
void         b200c_cancel_reset(b200c_ctx*);

#ifdef __cplusplus
}
#endif
#endif /* B200C_H */
