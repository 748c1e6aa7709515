// compact.cu — b200c_compact: the whole CompactionTask hot loop (S/db/compaction/CompactionTask.java:184-236) as a chain of
// data-parallel kernels on one B200:
//
//   K1  k_decompress_chunks      every input chunk -> U (CRC verified)                          [codec.cuh]
//   K2  k_index_find/chain/emit  Index.db walk of BigTableScanner (format/big/BigTableScanner.java:135-184) done speculatively in
//                                256-byte blocks, proven equal to the sequential parse, + Murmur3 token per key
//   K3  k_bucket_bounds + k_merge_buckets   the partition-level MergeIterator (S/utils/MergeIterator.java:154-219): token space is
//                                cut into buckets, one warp per bucket runs a tournament over its <= 64 sources (one or two
//                                per lane, warp-min by shuffles); equal keys reduce together in source order
//   K4  k_partition_thr/warp     row merge + reconcile + purge + big-format serialisation, size -> scan -> emit, output partitions
//                                counting-sorted by fan-in; cursors in shared memory (fan-in <= 16) or one warp each  [partition*.cuh]
//   K5  k_compress_chunks ...    CompressedSequentialWriter + ChecksumWriter                    [codec.cuh]
//
// No CPU fallback; every error is reported through the return code (B200C_ECORRUPT carries the location).
#include "engine.cuh"
#include "scan.cuh"
#include "codec_defs.cuh"
#include "partition.cuh"
#include "partition_tile.cuh"
#include "meta.cuh"
#include <climits>
#include <vector>
#include <algorithm>
#include <functional>
#include <cmath>

using namespace b200c;

namespace b200c {

int compress_stream_device(b200c_ctx* c, int comp, const uint8_t* d_in, uint64_t n, int chunk_len, int max_clen,
                           uint8_t* d_out, uint64_t out_cap, uint64_t* d_offs, uint64_t* out_len, uint32_t* digest, int ws_base);
int compress_slots_device(b200c_ctx* c, int comp, const uint8_t* d_in, uint64_t n, int chunk_len, int max_clen,
                          uint8_t* slots, int stride, uint32_t* file_len, uint32_t* seg_raw);
int pack_digest_device(b200c_ctx* c, const uint8_t* slots, int stride, const uint32_t* file_len, const uint32_t* seg_raw, uint64_t nchunks,
                       uint8_t* d_out, uint64_t out_cap, uint64_t* d_offs, uint64_t* out_len, uint32_t* digest, int ws_base);
int decompress_stream_device(b200c_ctx* c, int comp, const uint8_t* d_data, uint64_t data_len, const uint64_t* d_offs, uint64_t nchunks,
                             int chunk_len, int max_clen, uint64_t data_length, uint8_t* d_out, int verify, ChunkErr* d_err, uint64_t chunk0, uint64_t count, int tag);
int decompress_multi_device(b200c_ctx* c, K1Seg* segs, int nseg, int verify, ChunkErr* d_err, int ws_slot);

enum { IB = 256 };                       // Index.db speculation block
#ifndef B200C_K4_STAGED_DEFAULT
#define B200C_K4_STAGED_DEFAULT 0          // flipped to 1 once the staged mapping has beaten the global one on the B200 (profiles/)
#endif
#ifndef B200C_K1_BATCH_DEFAULT
#define B200C_K1_BATCH_DEFAULT true
#endif
enum { MAX_RANGES = 16, EV_RANGE = 200, EV_INDEX = 220, EV_K5 = 230 };      // token-range pieces per call; slots of b200c_ctx::ev_pool
#define NONE64 (~0ull)

enum { WS_U = 16, WS_CD, WS_CO, WS_IDX, WS_PARAMS, WS_BBASE, WS_ISTART, WS_ICNT, WS_IEND, WS_IHIT, WS_IBAD, WS_ISCAN,
       WS_TOK, WS_KP, WS_KLEN, WS_UPOS, WS_PBASE, WS_RANGE, WS_BSTART, WS_CONTRIB, WS_HEAD, WS_OPIDX, WS_OPFIRST,
       WS_LIST, WS_CURSOR, WS_STMUNF, WS_STROWS, WS_OVF, WS_BOUND, WS_BPOS, WS_SCRATCH, WS_DSIZE, WS_IPAY, WS_NBLK, WS_IHEAD, WS_DPOS, WS_ISIZE, WS_IPOS, WS_UOUT, WS_IOUT, WS_DOUT, WS_OOFFS, WS_STATS, WS_ERR2, WS_LCS0 = 82, WS_LCS1, WS_LCS2, WS_LCS3, WS_LCS4, WS_ICAP, WS_IOFF, WS_ISCR, WS_PLAN, WS_UOUT2, WS_SUMM, WS_PURGE, WS_K1SEG, WS_INSZ, WS_BIG, WS_INPOS, WS_TMARK, WS_TSCAN, WS_TSTART, WS_META_SG, WS_META_TD, WS_META_BLOOM, WS_META_KEYS, WS_META_SUMENT, WS_META_SUMOFF, WS_META_FLAG, WS_META_WRANK, WS_META_SAMPLE, WS_META_ESIZE, WS_META_EPOS, WS_CCOUNT, WS_SLICE, WS_META_TDD,
       WS_SCANA = 60, WS_CODEC = 70 };

static_assert(WS_ERR2 < WS_SCANA && WS_SCANA + 6 <= WS_CODEC && WS_CODEC + 12 <= WS_LCS0 && WS_META_TDD < WS_SLOTS, "workspace slot map");
struct DevErr { unsigned long long code; };       // min over (kind << 56 | input << 48 | offset); ~0 = none

__device__ __forceinline__ void report_err(DevErr* e, int kind, int input, uint64_t off) {
    atomicMin(&e->code, ((unsigned long long)kind << 56) | ((unsigned long long)(input & 0xFF) << 48) | (off & 0xFFFFFFFFFFFFull));
}

// ---- Murmur3 (Cassandra variant): S/utils/MurmurHash.java:178-260, token = Murmur3Partitioner.getToken :256-296 ---------------
__host__ __device__ __forceinline__ uint64_t rotl64(uint64_t v, int n) { return (v << n) | (v >> (64 - n)); }
__host__ __device__ __forceinline__ uint64_t fmix64(uint64_t k) { k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33; return k; }
__host__ __device__ int64_t murmur3_token(const uint8_t* key, uint32_t len) {
    if (len == 0) return I64_MIN;
    const uint32_t nblocks = len >> 4;
    uint64_t h1 = 0, h2 = 0;
    const uint64_t c1 = 0x87c37b91114253d5ULL, c2 = 0x4cf5ad432745937fULL;
    for (uint32_t i = 0; i < nblocks; i++) {
        uint64_t k1 = 0, k2 = 0;
        for (int b = 0; b < 8; b++) { k1 |= (uint64_t)key[i * 16 + b] << (8 * b); k2 |= (uint64_t)key[i * 16 + 8 + b] << (8 * b); }
        k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
        h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729;
        k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
        h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5;
    }
    const uint8_t* t = key + nblocks * 16;
    uint64_t k1 = 0, k2 = 0;
    int rem = len & 15;
    for (int i = rem - 1; i >= 8; i--) k2 ^= (uint64_t)(int64_t)(int8_t)t[i] << (8 * (i - 8));     // signed tail bytes (:214-233)
    if (rem > 8) { k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2; }
    for (int i = (rem < 8 ? rem : 8) - 1; i >= 0; i--) k1 ^= (uint64_t)(int64_t)(int8_t)t[i] << (8 * i);
    if (rem > 0) { k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1; }
    h1 ^= (uint64_t)len; h2 ^= (uint64_t)len;
    h1 += h2; h2 += h1; h1 = fmix64(h1); h2 = fmix64(h2); h1 += h2;
    int64_t v = (int64_t)h1;
    return v == I64_MIN ? I64_MAX : v;
}

// ---- Index.db slices for token sub-ranges -------------------------------------------------------------------------------------------
// A call for (token_lo, token_hi] needs only the Index.db entries between the last Summary.db sample whose token is <= token_lo and the
// first sample whose token is > token_hi — what a ranged scanner seeks to (BigTableScanner.java:105-132, SSTableReader.getPositionsForRanges
// S/io/sstable/format/SSTableReader.java:724). Binary search over the samples, hashing the ~2 x 17 keys it visits; runs on the host for host
// buffers (so the rest of Index.db never crosses PCIe) and in a one-thread-per-input kernel for device-resident inputs.
struct IdxSlice { uint64_t lo, hi, uend, s_first, s_count; };
__host__ __device__ inline int64_t order_token_of(int partitioner, const uint8_t* key, uint32_t kl) {
    if (partitioner == B200C_PARTITIONER_BYTE_ORDERED) { uint64_t pre = 0; for (uint32_t q = 0; q < 8; q++) pre = (pre << 8) | (q < kl ? key[q] : 0); return (int64_t)(pre ^ 0x8000000000000000ull); }
    return murmur3_token(key, kl);
}
__host__ __device__ inline bool sample_token(const uint8_t* index, uint64_t ilen, uint64_t off, int partitioner, int64_t* tok) {
    if (off + 2 > ilen) return false;
    const uint32_t kl = ((uint32_t)index[off] << 8) | index[off + 1];
    if (off + 2 + kl > ilen) return false;
    *tok = order_token_of(partitioner, index + off + 2, kl);
    return true;
}
__host__ __device__ inline bool compute_index_slice(const uint8_t* index, uint64_t ilen, const uint64_t* summ, uint64_t ns, uint64_t data_length, int partitioner,
                                                    int64_t tlo, int64_t thi, IdxSlice* out) {
    uint64_t a = 0, b = ns; int64_t t = 0;
    if (tlo != I64_MIN) while (a < b) { uint64_t mid = (a + b) / 2; if (!sample_token(index, ilen, summ[mid], partitioner, &t)) return false; if (t <= tlo) a = mid + 1; else b = mid; }
    const uint64_t first = a ? a - 1 : 0;                      // the last sample with token <= token_lo: entries in range may follow it inside its interval
    a = first; b = ns;
    while (a < b) { uint64_t mid = (a + b) / 2; if (!sample_token(index, ilen, summ[mid], partitioner, &t)) return false; if (t <= thi) a = mid + 1; else b = mid; }
    const uint64_t last = a;                                   // first sample with token > token_hi (ns: none)
    out->lo = summ[first]; out->hi = last < ns ? summ[last] : ilen; out->s_first = first; out->s_count = last - first; out->uend = data_length;
    if (out->lo > out->hi || out->hi > ilen) return false;
    if (last < ns) {                                           // the slice's last partition ends where the entry at that sample says the next one starts
        uint64_t off = summ[last]; if (off + 2 > ilen) return false;
        const uint32_t kl = ((uint32_t)index[off] << 8) | index[off + 1]; off += 2 + kl;
        uint64_t pos = 0; if (off >= ilen) return false;
        const uint32_t f = index[off];
        if (f < 0x80) pos = f;
        else { int extra = 0; for (uint32_t x = f; x & 0x80; x <<= 1) extra++; if (extra > 8) extra = 8; if (off + extra >= ilen) return false; pos = extra == 8 ? 0 : (f & (0xFFu >> extra)); for (int k = 1; k <= extra; k++) pos = (pos << 8) | index[off + k]; }
        if (pos > data_length) return false;
        out->uend = pos;
    }
    return true;
}
// data position stored in the Index.db entry at `off` (u16 keyLen | key | vint position | ...)
__host__ __device__ inline bool entry_data_position(const uint8_t* index, uint64_t ilen, uint64_t off, uint64_t data_length, uint64_t* pos_out) {
    if (off + 2 > ilen) return false;
    const uint32_t kl = ((uint32_t)index[off] << 8) | index[off + 1]; off += 2 + kl;
    if (off >= ilen) return false;
    const uint32_t f = index[off]; uint64_t pos;
    if (f < 0x80) pos = f;
    else { int extra = 0; for (uint32_t x = f; x & 0x80; x <<= 1) extra++; if (extra > 8) extra = 8; if (off + extra >= ilen) return false; pos = extra == 8 ? 0 : (f & (0xFFu >> extra)); for (int k = 1; k <= extra; k++) pos = (pos << 8) | index[off + k]; }
    if (pos > data_length) return false;
    *pos_out = pos; return true;
}
__global__ void k_index_slices(const uint8_t* const* __restrict__ index, const uint64_t* __restrict__ ilen, const uint64_t* const* __restrict__ summ, const uint64_t* __restrict__ ns,
                               const uint64_t* __restrict__ dlen, int K, int partitioner, int64_t tlo, int64_t thi, IdxSlice* __restrict__ out, uint32_t* __restrict__ ok) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K) return;
    ok[i] = compute_index_slice(index[i], ilen[i], summ[i], ns[i], dlen[i], partitioner, tlo, thi, &out[i]) ? 1u : 0u;
}

// ---- K2: Index.db ------------------------------------------------------------------------------------------------------------
// One Index.db entry = u16 keyLen | key | vint dataPosition | vint32 payloadSize | payload (RowIndexEntry.java:468-473).
// Structural parse of the entry at offset o of input i; returns its length (0 = not an entry). check_data additionally requires
// Data.db at dataPosition to start with the same u16 keyLen | key (used only to pick speculation starts).
__device__ uint64_t idx_entry(const CParams& P, const uint8_t* __restrict__ IDX, int i, uint64_t o, bool check_data, uint64_t* dpos_out, uint32_t* klen_out) {
    const InDesc& in = P.in[i];
    const uint8_t* b = IDX + in.ibase;
    if (o + 2 > in.ilen) return 0;
    uint32_t kl = ((uint32_t)b[o] << 8) | b[o + 1];
    uint64_t p = o + 2 + kl;
    if (p + 2 > in.ilen) return 0;
    uint64_t pos, ps;
    int n = vint_read(b + p, b + in.ilen, &pos); if (!n) return 0; p += n;
    n = vint_read(b + p, b + in.ilen, &ps); if (!n) return 0; p += n;
    if (ps > 0x7FFFFFFFull || p + ps > in.ilen) return 0;
    if (pos >= in.ulen || pos + 2 + kl + 2 > in.ulen) return 0;
    if (check_data) {
        // a partition starts right after the previous partition's end-of-partition flag and repeats u16 keyLen | key
        const uint8_t* d = P.U + in.ubase + pos;
        if ((pos == 0) != (o == 0)) return 0;        // positions increase strictly with the entry offset: only the first entry sits at 0
        if (pos > 0 && d[-1] != 0x01) return 0;
        for (uint32_t k = 0; k < 2 + kl; k++) if (d[k] != b[o + k]) return 0;
    }
    *dpos_out = pos; *klen_out = kl;
    return p + ps - o;
}

__device__ __forceinline__ int input_of_block(const uint64_t* __restrict__ bbase, int ninputs, uint64_t b) {
    int i = 0; while (i + 1 < ninputs && bbase[i + 1] <= b) i++; return i;
}

__global__ void __launch_bounds__(256) k_index_find(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, const uint64_t* __restrict__ bbase, uint64_t b0,
                                                    uint64_t nblocks, uint64_t* __restrict__ start) {
    uint64_t b = b0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const CParams& P = *Pp;
    int i = input_of_block(bbase, P.ninputs, b);
    uint64_t lb = b - bbase[i], lo = lb * IB, hi = min(lo + IB, P.in[i].ilen);
    // a speculated start must open a chain of 3 entries that all match Data.db with strictly increasing positions (or run into
    // EOF): single-entry matches are too weak (keyLen 0 / 1 candidates inside key or value bytes do occur at GB scale)
    auto chain3 = [&](uint64_t o) -> bool {
        uint64_t prev = 0;
        for (int k = 0; k < 3; k++) {
            uint64_t dpos; uint32_t kl;
            uint64_t len = idx_entry(P, IDX, i, o, true, &dpos, &kl);
            if (!len) return false;
            if (k && dpos <= prev) return false;
            prev = dpos; o += len;
            if (o == P.in[i].ilen) return true;
        }
        return true;
    };
    uint64_t found = NONE64;
    if (lb == 0) { if (chain3(0)) found = 0; }
    else for (uint64_t o = lo; o < hi; o++) if (chain3(o)) { found = o; break; }
    start[b] = found;
}

// Speculation from Summary.db: anchors[] are Index.db offsets of sampled entries (every 128th by default). One thread walks the
// entries between two anchors and records, per block, the lowest entry start it meets. Nothing is taken on trust: chain / verify
// below still prove the result against the sequential parse, a wrong anchor only costs the sequential fallback.
__global__ void __launch_bounds__(128) k_index_find_anchors(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, const uint64_t* __restrict__ bbase, int i,
                                                            const uint64_t* __restrict__ anchors, uint64_t n, uint64_t bias /* file offset the slice starts at */, unsigned long long* __restrict__ start) {
    uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n) return;
    const CParams& P = *Pp;
    const uint64_t ilen = P.in[i].ilen;
    uint64_t o = anchors[a] - bias, end = (a + 1 < n) ? anchors[a + 1] - bias : ilen;
    if (o >= ilen || end > ilen || end <= o) return;
    uint64_t prev_block = NONE64;
    while (o < end) {
        uint64_t dpos; uint32_t kl;
        uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) return;
        uint64_t b = o / IB;
        if (b != prev_block) { atomicMin(&start[bbase[i] + b], (unsigned long long)o); prev_block = b; }
        o += len;
    }
}

// K2 with Summary.db samples, in two walks instead of four passes: every Summary interval (the entries between two samples: 128 by default,
// ~2 KB of Index.db) is one thread. Walk 1 counts the interval's entries and PROVES the samples: the walk from sample a must land exactly on
// sample a + 1 (the last one on the end of the slice) and the first sample must be the slice's first byte — by induction the intervals'
// chains are the sequential parse. Walk 2 (after a scan of the counts) parses again and emits token / key prefix / key length / position.
// Any interval that does not land marks the input: the call then falls back to the speculate-chain-verify path below, whose sequential
// last resort reports real damage with its offset.
__global__ void __launch_bounds__(128) k_index_count_intervals(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, int i, const uint64_t* __restrict__ anchors, uint64_t n,
                                                               uint64_t bias, uint32_t* __restrict__ acnt, uint32_t* __restrict__ bad) {
    uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n) return;
    const CParams& P = *Pp;
    const uint64_t ilen = P.in[i].ilen;
    uint64_t o = anchors[a] - bias; const uint64_t end = (a + 1 < n) ? anchors[a + 1] - bias : ilen;
    uint32_t cnt = 0;
    if ((a == 0 && o != 0) || o >= ilen || end > ilen || end <= o) { bad[i] = 1; acnt[a] = 0; return; }
    while (o < end) {
        uint64_t dpos; uint32_t kl;
        const uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) break;
        cnt++; o += len;
    }
    if (o != end) bad[i] = 1;
    acnt[a] = cnt;
}
__global__ void __launch_bounds__(128) k_index_emit_intervals(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, int i, const uint64_t* __restrict__ anchors, uint64_t n,
                                                              uint64_t bias, const uint64_t* __restrict__ ascan /* of this input's intervals, [n + 1] */, uint64_t g0,
                                                              int64_t* __restrict__ tok, uint64_t* __restrict__ kp, uint16_t* __restrict__ klen, uint64_t* __restrict__ upos) {
    uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n) return;
    const CParams& P = *Pp;
    const InDesc& in = P.in[i];
    uint64_t o = anchors[a] - bias; const uint64_t end = (a + 1 < n) ? anchors[a + 1] - bias : in.ilen;
    uint64_t g = g0 + (ascan[a] - ascan[0]); const uint64_t gend = g0 + (ascan[a + 1] - ascan[0]);
    for (; o < end && g < gend; g++) {
        uint64_t dpos; uint32_t kl;
        const uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) return;                                  // (cannot happen: walk 1 parsed the same bytes)
        const uint8_t* key = IDX + in.ibase + o + 2;
        uint64_t pre = 0; for (uint32_t q = 0; q < 8; q++) pre = (pre << 8) | (q < kl ? key[q] : 0);
        tok[g] = P.partitioner ? (int64_t)(pre ^ 0x8000000000000000ull) : murmur3_token(key, kl);       // (see k_index_emit)
        kp[g] = pre; klen[g] = (uint16_t)kl; upos[g] = in.ubase + dpos;
        o += len;
    }
}

__global__ void __launch_bounds__(256) k_index_chain(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, const uint64_t* __restrict__ bbase, uint64_t b0,
                                                     uint64_t nblocks, const uint64_t* __restrict__ start, uint32_t* __restrict__ cnt, uint64_t* __restrict__ chain_end) {
    uint64_t b = b0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const CParams& P = *Pp;
    int i = input_of_block(bbase, P.ninputs, b);
    uint64_t lb = b - bbase[i], hi = min((lb + 1) * IB, P.in[i].ilen);
    uint64_t o = start[b]; uint32_t n = 0;
    if (o == NONE64) { cnt[b] = 0; chain_end[b] = NONE64; return; }
    while (o < hi) {
        uint64_t dpos; uint32_t kl;
        uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) { o = NONE64 - 1; break; }             // structurally broken chain: caught by verification
        n++; o += len;
    }
    cnt[b] = n; chain_end[b] = o;
}

// every chain must end exactly on the next block's speculated start (or at EOF), and every start must be the end of a chain
__global__ void __launch_bounds__(256) k_index_verify_a(const CParams* __restrict__ Pp, const uint64_t* __restrict__ bbase, uint64_t b0, uint64_t nblocks,
                                                        const uint64_t* __restrict__ start, const uint64_t* __restrict__ chain_end,
                                                        uint32_t* __restrict__ hit, uint32_t* __restrict__ bad) {
    uint64_t b = b0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const CParams& P = *Pp;
    int i = input_of_block(bbase, P.ninputs, b);
    uint64_t lb = b - bbase[i];
    if (lb == 0 && P.in[i].ilen > 0 && start[b] != 0) { bad[i] = 1; return; }
    if (start[b] == NONE64) return;
    uint64_t e = chain_end[b];
    if (e == P.in[i].ilen) return;
    if (e > P.in[i].ilen) { bad[i] = 1; return; }
    uint64_t nb = bbase[i] + e / IB;
    if (start[nb] != e) { bad[i] = 1; return; }
    hit[nb] = 1;
    for (uint64_t k = b + 1; k < nb; k++) if (start[k] != NONE64) { bad[i] = 1; return; }
}
__global__ void __launch_bounds__(256) k_index_verify_b(const CParams* __restrict__ Pp, const uint64_t* __restrict__ bbase, uint64_t b0, uint64_t nblocks,
                                                        const uint64_t* __restrict__ start, const uint32_t* __restrict__ hit, uint32_t* __restrict__ bad) {
    uint64_t b = b0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    int i = input_of_block(bbase, Pp->ninputs, b);
    if (b != bbase[i] && start[b] != NONE64 && !hit[b]) bad[i] = 1;
}
// slow but always-correct path for an input whose speculation could not be proven: one thread walks the file like
// BigTableScanner does and rewrites start[]/cnt[] of its blocks. A structural error here is real corruption.
__global__ void k_index_seq(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, const uint64_t* __restrict__ bbase,
                            uint64_t* __restrict__ start, uint32_t* __restrict__ cnt, const uint32_t* __restrict__ bad, DevErr* __restrict__ err) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    const CParams& P = *Pp;
    if (i >= P.ninputs || !bad[i]) return;
    uint64_t nb = bbase[i + 1] - bbase[i];
    for (uint64_t k = 0; k < nb; k++) { start[bbase[i] + k] = NONE64; cnt[bbase[i] + k] = 0; }
    uint64_t o = 0;
    while (o < P.in[i].ilen) {
        uint64_t dpos; uint32_t kl;
        uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) { report_err(err, 3, i, o); return; }
        uint64_t b = bbase[i] + o / IB;
        if (start[b] == NONE64) start[b] = o;
        cnt[b]++;
        o += len;
    }
}

__global__ void __launch_bounds__(256) k_index_emit(const CParams* __restrict__ Pp, const uint8_t* __restrict__ IDX, const uint64_t* __restrict__ bbase,
        uint64_t nblocks, const uint64_t* __restrict__ start, const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ scan,
        const uint64_t* __restrict__ pbase, int64_t* __restrict__ tok, uint64_t* __restrict__ kp, uint16_t* __restrict__ klen,
        uint64_t* __restrict__ upos, DevErr* __restrict__ err) {
    uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const CParams& P = *Pp;
    uint32_t n = cnt[b];
    if (!n) return;
    int i = input_of_block(bbase, P.ninputs, b);
    const InDesc& in = P.in[i];
    uint64_t g = pbase[i] + (scan[b] - scan[bbase[i]]);
    uint64_t o = start[b];
    for (uint32_t k = 0; k < n; k++, g++) {
        uint64_t dpos; uint32_t kl;
        uint64_t len = idx_entry(P, IDX, i, o, false, &dpos, &kl);
        if (!len) { report_err(err, 3, i, o); return; }
        const uint8_t* key = IDX + in.ibase + o + 2;
        // Index.db <-> Data.db consistency is checked by K4 when it parses the partition header: key length + 8-byte prefix, and for
        // longer keys the token (so this kernel needs Index.db only and can run before Data.db is on the device)
        uint64_t pre = 0; for (uint32_t q = 0; q < 8; q++) pre = (pre << 8) | (q < kl ? key[q] : 0);
        // ByteOrderedPartitioner: the order is the key bytes themselves; the sign-flipped 8-byte prefix is an order-preserving token and
        // the tie path of the merge (cmp_keys) finishes the comparison on the remaining bytes / the length
        tok[g] = P.partitioner ? (int64_t)(pre ^ 0x8000000000000000ull) : murmur3_token(key, kl);
        kp[g] = pre; klen[g] = (uint16_t)kl; upos[g] = in.ubase + dpos;
        o += len;
    }
}

// per input: sentinel position, token-range bounds [plo, phi) (inputs are token sorted), and a sortedness check
__global__ void k_input_ranges(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ pcount,
                               const int64_t* __restrict__ tok, uint64_t* __restrict__ upos, int64_t tlo, int64_t thi, uint64_t* __restrict__ range /*[2*K]*/,
                               unsigned long long* __restrict__ range_bytes /* optional: += uncompressed bytes of the partitions in range */) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    const CParams& P = *Pp;
    if (i >= P.ninputs) return;
    uint64_t n = pcount[i]; const int64_t* t = tok + pbase[i];
    upos[pbase[i] + n] = P.in[i].ubase + P.in[i].uend;
    uint64_t lo = 0, hi = n;
    if (tlo != I64_MIN) { uint64_t a = 0, b = n; while (a < b) { uint64_t m = (a + b) / 2; if (t[m] <= tlo) a = m + 1; else b = m; } lo = a; }   // first > tlo
    { uint64_t a = lo, b = n; while (a < b) { uint64_t m = (a + b) / 2; if (t[m] <= thi) a = m + 1; else b = m; } hi = a; }                     // first > thi
    range[2 * i] = lo; range[2 * i + 1] = hi;
    if (range_bytes && hi > lo) atomicAdd(range_bytes, (unsigned long long)(upos[pbase[i] + hi] - upos[pbase[i] + lo]));
}

// an SSTable is ordered by (token, key) and its partitions do not overlap: tokens must not decrease, equal tokens must come with
// increasing (8-byte key prefix, length) and Data.db positions must increase along Index.db — everything downstream binary-searches
// these arrays, so a file in another partitioner's order (or a damaged one) is rejected here whatever its size
// (SortedTableWriter.verifyPartition S/io/sstable/format/SortedTableWriter.java:165-178 enforces the same order when files are written).
__global__ void __launch_bounds__(256) k_check_order(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ pcount,
                                                     const int64_t* __restrict__ tok, const uint64_t* __restrict__ kp, const uint16_t* __restrict__ klen,
                                                     const uint64_t* __restrict__ upos, DevErr* __restrict__ err) {
    const CParams& P = *Pp;
    for (int i = 0; i < P.ninputs; i++) {
        const uint64_t n = pcount[i], b = pbase[i];
        for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g + 1 < n; g += (uint64_t)gridDim.x * blockDim.x) {
            const uint64_t x = b + g, y = x + 1;
            bool bad = tok[y] < tok[x] || upos[y] <= upos[x];
            if (!bad && tok[y] == tok[x]) bad = kp[y] < kp[x] || (kp[y] == kp[x] && klen[x] <= 8 && klen[y] <= klen[x]);
            if (bad) report_err(err, 3, i, upos[x] - P.in[i].ubase);
        }
    }
}

// token-range pieces: for piece r and input i the byte range [plan[2k], plan[2k+1]) of U (k = r * K + i) holding the partitions with
// token in (T[r], T[r+1]]; same bounds as k_input_ranges
__global__ void k_range_plan(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ pcount,
                             const int64_t* __restrict__ tok, const uint64_t* __restrict__ upos, const int64_t* __restrict__ T, int nr, uint64_t* __restrict__ plan) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    const CParams& P = *Pp;
    if (k >= nr * P.ninputs) return;
    int r = k / P.ninputs, i = k % P.ninputs;
    uint64_t n = pcount[i]; const int64_t* t = tok + pbase[i];
    int64_t tlo = T[r], thi = T[r + 1];
    uint64_t lo = 0, hi = n;
    if (tlo != I64_MIN) { uint64_t a = 0, b = n; while (a < b) { uint64_t m = (a + b) / 2; if (t[m] <= tlo) a = m + 1; else b = m; } lo = a; }
    { uint64_t a = lo, b = n; while (a < b) { uint64_t m = (a + b) / 2; if (t[m] <= thi) a = m + 1; else b = m; } hi = a; }
    plan[2 * k] = upos[pbase[i] + lo]; plan[2 * k + 1] = upos[pbase[i] + hi];
}
__global__ void __launch_bounds__(256) k_add_u64(uint64_t* __restrict__ a, uint64_t n, uint64_t v) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] += v;
}

// ---- K3: partition-level merge -------------------------------------------------------------------------------------------------
struct MergeGeom { uint64_t umin, width, nbuckets; };     // bucket b covers unsigned-token range [umin + b*width, umin + (b+1)*width)

__global__ void k_merge_geom(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ range,
                             const int64_t* __restrict__ tok, uint64_t nbuckets, MergeGeom* __restrict__ g) {
    const CParams& P = *Pp;
    uint64_t umin = ~0ull, umax = 0; bool any = false;
    for (int i = 0; i < P.ninputs; i++) {
        uint64_t lo = range[2 * i], hi = range[2 * i + 1];
        if (lo >= hi) continue;
        uint64_t a = (uint64_t)tok[pbase[i] + lo] ^ 0x8000000000000000ull, b = (uint64_t)tok[pbase[i] + hi - 1] ^ 0x8000000000000000ull;
        umin = min(umin, a); umax = max(umax, b); any = true;
    }
    if (!any) { umin = 0; umax = 0; }
    g->umin = umin; g->nbuckets = nbuckets; g->width = (umax - umin) / nbuckets + 1;
}

// bstart[b * K + i] = first partition of input i (absolute index in its arrays) whose token falls in bucket >= b
__global__ void __launch_bounds__(256) k_bucket_bounds(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ range,
                                                       const int64_t* __restrict__ tok, const MergeGeom* __restrict__ gp, uint64_t* __restrict__ bstart) {
    const CParams& P = *Pp; const int K = P.ninputs;
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t nb = gp->nbuckets;
    if (t >= (nb + 1) * (uint64_t)K) return;
    uint64_t b = t / K; int i = (int)(t % K);
    uint64_t lo = range[2 * i], hi = range[2 * i + 1];
    uint64_t res;
    if (b == 0) res = lo;
    else if (b >= nb) res = hi;
    else {
        unsigned long long hi128 = __umul64hi(b, gp->width), lo128 = b * gp->width;
        uint64_t bound = gp->umin + lo128;
        if (hi128 || bound < lo128) res = hi;                 // boundary beyond the token space
        else {
            const int64_t* tk = tok + pbase[i];
            uint64_t a = lo, z = hi;
            while (a < z) { uint64_t m = (a + z) / 2; if (((uint64_t)tk[m] ^ 0x8000000000000000ull) < bound) a = m + 1; else z = m; }
            res = a;
        }
    }
    bstart[t] = res;
}

__device__ __forceinline__ int64_t warp_min_i64(int64_t v) {
#pragma unroll
    for (int d = 16; d; d >>= 1) { int64_t o = __shfl_xor_sync(FULL_MASK, v, d); v = o < v ? o : v; }
    return v;
}

// full key comparison of two partitions (DecoratedKey.compareTo tie on token: unsigned lexicographic, S/db/DecoratedKey.java:79-91)
__device__ int cmp_keys(const uint8_t* __restrict__ U, uint64_t ua, uint32_t la, uint64_t kpa, uint64_t ub, uint32_t lb, uint64_t kpb) {
    if (kpa != kpb) return kpa < kpb ? -1 : 1;
    if (la <= 8 || lb <= 8) return la == lb ? 0 : (la < lb ? -1 : 1);
    return cmp_bytes(U + ua + 2 + 8, (int)la - 8, U + ub + 2 + 8, (int)lb - 8);
}

// One warp per token bucket. Lane l owns sources l and l+32. Each step: warp-min of the head tokens (the tournament), ties on
// token are resolved by key bytes, all heads equal to the winner are emitted as one output partition (contributors in source
// order, first one flagged) and advanced. contrib entry = head<<63 | src<<56 | partition index (40 bits).
__global__ void __launch_bounds__(128) k_merge_buckets(const CParams* __restrict__ Pp, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ range,
        const int64_t* __restrict__ tok, const uint64_t* __restrict__ kp, const uint16_t* __restrict__ klen, const uint64_t* __restrict__ upos,
        const uint64_t* __restrict__ bstart, uint64_t nbuckets, uint64_t* __restrict__ contrib, uint32_t* __restrict__ head, unsigned long long* __restrict__ hist) {
    __shared__ uint32_t s_hist[MAXK];
    const CParams& P = *Pp; const int K = P.ninputs;
    const int lane = threadIdx.x & 31;
    for (int k = threadIdx.x; k < MAXK; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    uint64_t b = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b < nbuckets) {
        uint64_t cur[2], end[2], base[2]; int64_t t[2]; bool valid[2];
        uint64_t cpos = 0;
        for (int s = 0; s < 2; s++) {
            int src = lane + 32 * s;
            cur[s] = end[s] = 0; base[s] = 0; valid[s] = false; t[s] = I64_MAX;
            if (src < K) {
                cur[s] = bstart[b * K + src]; end[s] = bstart[(b + 1) * K + src]; base[s] = pbase[src];
                cpos += cur[s] - range[2 * src];
                valid[s] = cur[s] < end[s];
                if (valid[s]) t[s] = tok[base[s] + cur[s]];
            }
        }
#pragma unroll
        for (int d = 16; d; d >>= 1) cpos += __shfl_xor_sync(FULL_MASK, cpos, d);
        for (;;) {
            bool any = __any_sync(FULL_MASK, valid[0] || valid[1]);
            if (!any) break;
            int64_t lmin = I64_MAX;
            if (valid[0]) lmin = t[0];
            if (valid[1] && t[1] < lmin) lmin = t[1];
            int64_t wmin = warp_min_i64(lmin);
            bool tie0 = valid[0] && t[0] == wmin, tie1 = valid[1] && t[1] == wmin;
            uint32_t m0 = __ballot_sync(FULL_MASK, tie0), m1 = __ballot_sync(FULL_MASK, tie1);
            if (__popc(m0) + __popc(m1) > 1) {
                // same token from several sources: almost always the same key; compare key bytes to be exact
                for (;;) {
                    int ls = m0 ? 0 : 1; int ll = __ffs(ls == 0 ? m0 : m1) - 1;             // leader = lowest source among the tied
                    uint64_t g0 = base[0] + cur[0], g1 = base[1] + cur[1];
                    uint64_t lg = __shfl_sync(FULL_MASK, ls == 0 ? g0 : g1, ll);
                    uint64_t lkp = kp[lg]; uint32_t lkl = klen[lg]; uint64_t lup = upos[lg];
                    int c0 = 0, c1 = 0;
                    if (tie0) c0 = cmp_keys(P.U, upos[g0], klen[g0], kp[g0], lup, lkl, lkp);
                    if (tie1) c1 = cmp_keys(P.U, upos[g1], klen[g1], kp[g1], lup, lkl, lkp);
                    uint32_t less0 = __ballot_sync(FULL_MASK, tie0 && c0 < 0), less1 = __ballot_sync(FULL_MASK, tie1 && c1 < 0);
                    if (less0 | less1) { tie0 = tie0 && c0 < 0; tie1 = tie1 && c1 < 0; m0 = less0; m1 = less1; continue; }
                    tie0 = tie0 && c0 == 0; tie1 = tie1 && c1 == 0;
                    m0 = __ballot_sync(FULL_MASK, tie0); m1 = __ballot_sync(FULL_MASK, tie1);
                    break;
                }
            }
            int n0 = __popc(m0), gsize = n0 + __popc(m1);
            uint32_t ltm = (1u << lane) - 1u;
            if (tie0) { uint64_t p = cpos + __popc(m0 & ltm); contrib[p] = ((uint64_t)(p == cpos) << 63) | ((uint64_t)lane << 56) | cur[0]; head[p] = (p == cpos); }
            if (tie1) { uint64_t p = cpos + n0 + __popc(m1 & ltm); contrib[p] = ((uint64_t)(p == cpos) << 63) | ((uint64_t)(lane + 32) << 56) | cur[1]; head[p] = (p == cpos); }
            if (lane == 0) atomicAdd(&s_hist[gsize - 1], 1u);
            cpos += gsize;
            if (tie0) { cur[0]++; valid[0] = cur[0] < end[0]; if (valid[0]) t[0] = tok[base[0] + cur[0]]; }
            if (tie1) { cur[1]++; valid[1] = cur[1] < end[1]; if (valid[1]) t[1] = tok[base[1] + cur[1]]; }
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < MAXK; k += blockDim.x) if (s_hist[k]) atomicAdd(&hist[k], (unsigned long long)s_hist[k]);
}

__global__ void __launch_bounds__(256) k_op_first(const uint32_t* __restrict__ head, const uint64_t* __restrict__ opidx, uint64_t ncontrib, uint64_t* __restrict__ op_first) {
    uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < ncontrib && head[c]) op_first[opidx[c]] = c;
    if (c == ncontrib) op_first[opidx[ncontrib]] = ncontrib;
}

// ---- K4 wrappers -----------------------------------------------------------------------------------------------------------------
// Output partitions are processed in fan-in order (`list` = counting sort of the partitions by m, so a warp's threads run the same
// number of cursors). Per-partition results go to arrays indexed by the partition number j; totals come from k_sum_stats.
struct RunStats { unsigned long long merged_unfiltereds, rows_out, partitions_out; };

// Work-list order. Partitions are counting-sorted by key = (class, tile, fan-in m, size bucket):
//   class  = which kernel handles the fan-in (<= 8, <= 12, <= 16, <= 32, <= 64): each class is one contiguous slice of the list
//            (12: the cursors of a thread live in shared memory, and two thirds of the fan-ins above 8 of a 16-way merge are <= 12 —
//            8 instead of 6 blocks per SM for them),
//   tile   = j >> tile_shift: token-contiguous groups of output partitions whose input bytes (~32 MiB) stay L2 resident, so every
//            class streams through U once instead of once per (m, size) bin,
//   m, size bucket: threads of a warp run the same number of cursors over similarly sized partitions (less divergence).
enum { SORT_BUCKETS = 16, SORT_BINS = MAXK * SORT_BUCKETS };
// wide_bound: partitions whose inputs exceed it go to the warp-per-partition kernel whatever their fan-in (one lane per source parses in
// parallel, the tournament runs on shuffles): a single thread walking hundreds of KB is the slowest thing the GPU can do (schema W)
__device__ __forceinline__ uint32_t fanin_class(uint32_t m, uint64_t bound, uint64_t wide_bound) { return (bound > wide_bound && m <= 32) ? 3u : (m <= 8 ? 0u : (m <= 12 ? 1u : (m <= 16 ? 2u : (m <= 32 ? 3u : 4u)))); }
__device__ __forceinline__ uint64_t sort_key(uint32_t m, uint64_t bound, uint64_t j, uint32_t tile_shift, uint64_t ntiles, uint64_t wide_bound) {
    uint64_t avg = bound / (m ? m : 1);
    uint32_t bucket = (uint32_t)min((uint64_t)(SORT_BUCKETS - 1), avg >> 5);
    return ((uint64_t)fanin_class(m, bound, wide_bound) * ntiles + (j >> tile_shift)) * SORT_BINS + (m - 1) * SORT_BUCKETS + bucket;
}
__global__ void __launch_bounds__(256) k_class_hist(const uint64_t* __restrict__ op_first, const uint64_t* __restrict__ bound, uint64_t nparts,
                                                    uint32_t tile_shift, uint64_t ntiles, uint64_t wide_bound, unsigned long long* __restrict__ hist) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nparts; j += (uint64_t)gridDim.x * blockDim.x)
        atomicAdd(&hist[sort_key((uint32_t)(op_first[j + 1] - op_first[j]), bound[j], j, tile_shift, ntiles, wide_bound)], 1ull);
}
// warp-aggregated counting-sort scatter: list[cursor[key]++] = j
__global__ void __launch_bounds__(256) k_fanin_scatter(const uint64_t* __restrict__ op_first, const uint64_t* __restrict__ bound, uint64_t nparts,
                                                       uint32_t tile_shift, uint64_t ntiles, uint64_t wide_bound, unsigned long long* __restrict__ cursor, uint32_t* __restrict__ list) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = j < nparts;
    uint64_t key = valid ? sort_key((uint32_t)(op_first[j + 1] - op_first[j]), bound[j], j, tile_shift, ntiles, wide_bound) : ~0ull;
    uint32_t peers = __match_any_sync(FULL_MASK, key);
    int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (valid && lane == leader) base = atomicAdd(&cursor[key], (unsigned long long)__popc(peers));
    base = __shfl_sync(FULL_MASK, base, leader);
    if (valid) list[base + __popc(peers & ((1u << lane) - 1u))] = (uint32_t)j;
}

typedef Cur32 K4Cur;                                           // cursor of the thread-per-partition kernels (partition.cuh)
enum { SLOT_BYTES = sizeof(K4Cur), K4_SMEM_COLS = 8 };        // per-source cursor in shared memory

// mode 0: size pass only (EMIT = false). mode 1: the single serialisation pass — bytes go to scratch at dbase + doff[j] (capacity
// dcapv[j]), sizes/stats are recorded, no Index.db. mode 2: final emit of every written partition at dbase + dpos[j] with its Index.db
// entry. mode 3: like 2 but only partitions whose scratch (Data bytes or promoted-index slot) overflowed in mode 1.
struct K4Args {
    const CParams* P; const uint64_t* contrib; const uint64_t* op_first; const uint32_t* list; const uint64_t* upos; const uint64_t* pbase;
    const uint64_t* kp; const uint16_t* klen; const int64_t* tok;
    uint64_t* dsize; uint32_t* ipay; uint32_t* nblk; uint32_t* ihead; uint32_t* st_munf; uint32_t* st_rows; uint8_t* ovf;
    const uint64_t* doff; const uint64_t* dcapv; const uint64_t* dpos; const uint64_t* ipos; uint8_t* dbase; uint8_t* iout; DevErr* err; int mode;
    uint64_t jlo, jhi;               // modes 2/3: only partitions jlo <= j < jhi (one output file of a multi-file compaction)
    // mode 1: promoted-index slots (IXS_* layout in partition.cuh) of the partitions that can exceed one column-index block
    const uint64_t* ioff; const uint32_t* icapv; uint8_t* iscr;
    int m3_nblk;                     // mode 3 also re-emits partitions with a promoted index (two-pass A/B mode: there are no slots)
    const uint8_t* only_big;         // mode 1: when set, only partitions flagged here (the staged kernel took the others)
    // statistics side band (meta.cuh), gathered in the pass that visits every partition exactly once (mode 1); null otherwise
    StatGlobal* sg; TdropTable* td; uint32_t* ccount;
};

template <bool EMIT> __device__ __forceinline__ bool k4_prologue(const K4Args& a, uint64_t j, uint8_t*& dout, uint64_t& dcap, uint64_t& dposv, uint8_t*& iout, uint32_t& nbf, uint32_t& ipf, uint32_t& ixs_cap) {
    dout = nullptr; dcap = ~0ull; dposv = 0; iout = nullptr; nbf = 0; ipf = 0; ixs_cap = 0;
    if (!EMIT) return true;
    if (a.mode == 1) {
        if (a.only_big && !a.only_big[j]) return false;
        dout = a.dbase + a.doff[j]; dcap = a.dcapv[j];
        uint32_t slot = a.icapv[j];
        if (slot) { iout = a.iscr + a.ioff[j]; nbf = (slot - IXS_HEAD) / IXS_BLOCK_STRIDE; ixs_cap = nbf * IXS_PER_BLOCK; }
        return true;
    }
    if (!a.dsize[j] || j < a.jlo || j >= a.jhi) return false;
    if (a.mode == 3 && !(a.ovf[j] || (a.m3_nblk && a.nblk[j] > 1))) return false;
    dout = a.dbase + a.dpos[j]; dposv = a.dpos[j]; iout = a.iout + a.ipos[j]; nbf = a.nblk[j]; ipf = a.ipay[j];
    return true;
}
template <bool EMIT> __device__ __forceinline__ void k4_epilogue(const K4Args& a, uint64_t j, uint64_t c0, PartOut out, PartStats st, int e) {
    if (EMIT && a.mode >= 2) { if (e || out.dsize != a.dsize[j]) report_err(a.err, 8, 0, j); return; }
    if (e) { uint64_t en = a.contrib[c0]; int src = (int)((en >> 56) & 0x7F); report_err(a.err, e == PERR_UNSUPPORTED ? 9 : 4, src, a.upos[a.pbase[src] + (en & 0xFFFFFFFFFFull)] - a.P->in[src].ubase); out = PartOut{0, 0, 0, 0, 0}; st = PartStats{0, 0}; }
    a.dsize[j] = out.dsize; a.ipay[j] = out.ipay; a.nblk[j] = out.nblk; a.ihead[j] = out.ihead; a.ovf[j] = (uint8_t)out.ovf;
    if (a.ccount) a.ccount[j] = out.cells;
    a.st_munf[j] = (uint32_t)st.merged_unfiltereds; a.st_rows[j] = (uint32_t)st.rows_out;
}

template <int M_CAP, int NT, bool EMIT, bool CX = false>
__global__ void __launch_bounds__(NT) k_partition_thr(const K4Args a, uint64_t lo, uint64_t hi) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    // per thread in shared memory: M_CAP cursors, then (for tables with <= K4_SMEM_COLS columns) the merged-row scratch; +8 bytes
    // so that consecutive threads start in different banks. Wider tables keep the merged row in local memory.
    const int ncols_s = a.P->mcols <= K4_SMEM_COLS ? a.P->mcols : 0;
    const int stride = M_CAP * SLOT_BYTES + ncols_s * (int)sizeof(MCell) + 8;
    K4Cur* cur = (K4Cur*)(s_raw + (size_t)threadIdx.x * stride);
    MCell merged_local[MAXCOLS];
    MCell* merged = ncols_s ? (MCell*)(cur + M_CAP) : merged_local;
    DT open_dt[M_CAP];                                   // only touched when the partition holds range tombstone markers
    uint64_t t = lo + (uint64_t)blockIdx.x * NT + threadIdx.x;
    if (t >= hi) return;
    uint64_t j = a.list[t];
    uint8_t *dout, *iout; uint64_t dcap, dposv; uint32_t nbf, ipf, ixs_cap;
    if (!k4_prologue<EMIT>(a, j, dout, dcap, dposv, iout, nbf, ipf, ixs_cap)) return;
    uint64_t c0 = a.op_first[j]; uint32_t m = (uint32_t)(a.op_first[j + 1] - c0);
    PartOut out{0, 0, 0, 0, 0}; PartStats st{0, 0}; int e = 0;
    StatAcc acc; const bool stats = a.sg != nullptr && a.mode == 1;
    if (stats) acc.init(a.P->now, a.td);
    if (m > (uint32_t)M_CAP) e = PERR_UNSUPPORTED;
    else process_partition<EMIT, K4Cur, XlateGlobal, M_CAP, CX>(*a.P, XlateGlobal(), a.contrib, c0, m, a.upos, a.pbase, a.kp, a.klen, a.tok, dout, dcap, dposv, iout, nbf, ipf, ixs_cap, cur, open_dt, merged, out, st, e, stats ? &acc : nullptr);
    k4_epilogue<EMIT>(a, j, c0, out, st, e);
    if (stats && !e) stat_flush(a.sg, acc);
}

// fan-in above 16: a whole warp per partition, cursors in registers (partition_tile.cuh)
template <int S, bool EMIT>
__global__ void __launch_bounds__(128) k_partition_warp(const K4Args a, uint64_t lo, uint64_t hi) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    auto tile = cg::tiled_partition<32>(cg::this_thread_block());
    const int tid = threadIdx.x / 32;
    MCell* s_cells = (MCell*)s_raw + (size_t)tid * a.P->mcols;
    uint64_t t = lo + (uint64_t)blockIdx.x * 4 + tid;
    if (t >= hi) return;
    uint64_t j = a.list[t];
    uint8_t *dout, *iout; uint64_t dcap, dposv; uint32_t nbf, ipf, ixs_cap;
    if (!k4_prologue<EMIT>(a, j, dout, dcap, dposv, iout, nbf, ipf, ixs_cap)) return;
    uint64_t c0 = a.op_first[j]; uint32_t m = (uint32_t)(a.op_first[j + 1] - c0);
    PartOut out{0, 0, 0, 0, 0}; PartStats st{0, 0}; int e = 0;
    StatAcc acc; const bool stats = a.sg != nullptr && a.mode == 1;
    if (stats) acc.init(a.P->now, a.td);
    process_partition_tile<32, S, EMIT>(tile, *a.P, a.contrib, c0, m, a.upos, a.pbase, a.kp, a.klen, a.tok, dout, dcap, dposv, iout, nbf, ipf, ixs_cap, s_cells, out, st, e, stats ? &acc : nullptr);
    if (tile.thread_rank() == 0) { k4_epilogue<EMIT>(a, j, c0, out, st, e); if (stats && !e) stat_flush(a.sg, acc); }
}

// ---- K4, staged mapping (the default for partitions of up to ST_MAXP input bytes and fan-in <= ST_MAXM) ------------------------------
// The thread-per-partition kernels above parse Data.db straight from global memory: every field is a dependent load of a 32-byte
// sector from L2 or HBM. Here a block owns a TILE = a token-contiguous run of output partitions. Because every input is sorted by
// token, the input partitions of a tile are ONE contiguous byte range per source; those <= K ranges are copied into shared memory
// by the TMA unit (cp.async.bulk + an mbarrier counting the bytes), each byte crossing L2 -> SM exactly once in full 16-byte
// words, and the threads then run the same process_partition() on the copy: P.U points at the tile, cursors shrink to 32 bytes
// (32-bit positions, 16-bit header offsets). Tiles are cut where the running input bytes pass a multiple of ST_BYTES, the running
// contributor count a multiple of ST_CM, or the partition count a multiple of ST_MAXPART, so that the tile, its cursors and the
// per-thread merged rows fit ~70 KB and three blocks share an SM.
enum { ST_THREADS = 64, ST_MAXPART = 128, ST_BYTES = 32768, ST_MAXP = 8192, ST_CM = 448, ST_MAXM = 16,
       ST_STAGE_CAP = ST_BYTES + ST_MAXP + 32 * MAXK + 64, ST_CUR_CAP = ST_CM + ST_MAXM + 48,
       ST_HEAD = (16 + ((sizeof(CParams) + 15) & ~15) + MAXK * 8 * 3 + MAXK * 4 * 2 + 127) & ~127 };
static_assert(ST_STAGE_CAP < 65536 - 64, "staged tiles are addressed with 16-bit header offsets");

__global__ void __launch_bounds__(256) k_tile_marks(uint64_t nparts, const uint64_t* __restrict__ inpos, const uint64_t* __restrict__ op_first,
                                                    const uint8_t* __restrict__ big, uint32_t* __restrict__ mark, unsigned long long* __restrict__ nbig) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nparts) return;
    bool m = j == 0 || (j % ST_MAXPART) == 0 || big[j];
    if (!m) m = big[j - 1] || inpos[j] / ST_BYTES != inpos[j - 1] / ST_BYTES || op_first[j] / ST_CM != op_first[j - 1] / ST_CM;
    mark[j] = m ? 1u : 0u;
    if (big[j]) atomicAdd(nbig, 1ull);
}
__global__ void __launch_bounds__(256) k_tile_starts(uint64_t nparts, const uint32_t* __restrict__ mark, const uint64_t* __restrict__ tscan, uint32_t* __restrict__ tile_start) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nparts && mark[j]) tile_start[tscan[j]] = (uint32_t)j;
    if (j == nparts) tile_start[tscan[nparts]] = (uint32_t)nparts;
}

template <bool WIDE>
__global__ void __launch_bounds__(ST_THREADS) k_partition_staged(const K4Args a, const uint32_t* __restrict__ tile_start, const uint8_t* __restrict__ big) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* s_bar = (uint64_t*)smem;
    CParams* sP = (CParams*)(smem + 16);
    unsigned long long* s_lo = (unsigned long long*)(smem + 16 + ((sizeof(CParams) + 15) & ~15));
    unsigned long long* s_hi = s_lo + MAXK;
    uint64_t* s_g0 = (uint64_t*)(s_hi + MAXK);
    uint32_t* s_sbase = (uint32_t*)(s_g0 + MAXK);
    uint32_t* s_len = s_sbase + MAXK;
    uint8_t* stage = smem + ST_HEAD;
    CurS* curs = (CurS*)(stage + ST_STAGE_CAP);
    MCell* cells = (MCell*)(curs + ST_CUR_CAP);
    const int tid = threadIdx.x;
    const uint32_t j0 = tile_start[blockIdx.x], j1 = tile_start[blockIdx.x + 1];
    if (j0 >= j1 || big[j0]) return;                                  // a big partition is a tile of its own: the global-memory kernels take it
    const CParams& GP = *a.P;
    const int K = GP.ninputs;
    {   // header of the parameters -> shared memory, with U redirected to the tile
        const uint32_t* g = (const uint32_t*)a.P; uint32_t* d = (uint32_t*)sP;
        for (int i = tid; i < (int)(sizeof(CParams) / 4); i += ST_THREADS) d[i] = g[i];
        for (int i = tid; i < MAXK; i += ST_THREADS) { ((uint32_t*)s_lo)[i] = 0xFFFFFFFFu; ((uint32_t*)s_lo)[MAXK + i] = 0; s_len[i] = 0; }
        if (tid == 0) mbar_init(s_bar, 1);
    }
    __syncthreads();
    if (tid == 0) sP->U = stage;
    const uint64_t c0 = a.op_first[j0], c1 = a.op_first[j1];
    // first and last contribution of every source in this tile. A source's partitions appear in increasing order along the contributor list,
    // so the first / last POSITION of a source gives its lowest / highest partition: native 32-bit shared-memory min / max atomics on the
    // position (64-bit ones on the partition index would be compare-and-swap loops, 32 lanes deep on the same address)
    uint32_t* s_first = (uint32_t*)s_lo; uint32_t* s_last = s_first + MAXK;
    for (uint64_t c = c0 + tid; c < c1; c += ST_THREADS) {
        const int src = (int)((a.contrib[c] >> 56) & 0x7F);
        atomicMin(&s_first[src], (uint32_t)(c - c0)); atomicMax(&s_last[src], (uint32_t)(c - c0));
    }
    __syncthreads();
    if (tid < K && s_first[tid] != 0xFFFFFFFFu) {
        const uint64_t ilo = a.contrib[c0 + s_first[tid]] & 0xFFFFFFFFFFull, ihi = a.contrib[c0 + s_last[tid]] & 0xFFFFFFFFFFull;
        const uint64_t b0 = a.upos[a.pbase[tid] + ilo] & ~15ull, b1 = (a.upos[a.pbase[tid] + ihi + 1] + 15) & ~15ull;
        s_g0[tid] = b0; s_len[tid] = (uint32_t)min(b1 - b0, (uint64_t)0x7FFFFFF0u);
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t tot = 0;
        for (int i = 0; i < K; i++) { s_sbase[i] = tot; tot += s_len[i]; if (tot > (uint32_t)ST_STAGE_CAP) break; }
        if (tot > (uint32_t)ST_STAGE_CAP - 64) { s_len[0] = 0xFFFFFFFFu; report_err(a.err, 8, 0, j0); }      // cannot happen: the tile plan bounds it
        else {
            mbar_arrive_expect_tx(s_bar, tot);
            for (int i = 0; i < K; i++) if (s_len[i]) bulk_copy_g2s(stage + s_sbase[i], GP.U + s_g0[i], s_len[i], s_bar);
        }
    }
    __syncthreads();
    if (s_len[0] == 0xFFFFFFFFu) return;
    mbar_wait(s_bar, 0);
    // The lanes leave the wait loop one by one, and threads that were apart when a convergence barrier (BSSY) was set up do not re-join at its
    // BSYNC: without this barrier every lane ran the whole partition code ALONE (ncu: 1.0 active threads per instruction, 10 x slower than
    // the round-1 kernel — profiles/r2_k4_staged_divergence.txt). A block-wide barrier re-converges the warps before the per-partition work.
    __syncthreads();
    // partitions of the tile in fan-in order (counting sort in shared memory): the lanes of a warp then walk similar numbers of cursors
    uint8_t* s_order = (uint8_t*)s_lo;                               // (the first/last arrays are dead now) 128 entries + 20 counters behind them
    uint32_t* s_cnt = (uint32_t*)(s_order + ST_MAXPART);
    const uint32_t np = j1 - j0;
    if (tid < ST_MAXM + 2) s_cnt[tid] = 0;
    __syncthreads();
    for (uint32_t p = tid; p < np; p += ST_THREADS) { const uint32_t m = (uint32_t)(a.op_first[j0 + p + 1] - a.op_first[j0 + p]); atomicAdd(&s_cnt[min(m, (uint32_t)ST_MAXM + 1)], 1u); }
    __syncthreads();
    if (tid == 0) { uint32_t acc = 0; for (int k = 0; k <= ST_MAXM + 1; k++) { const uint32_t n = s_cnt[k]; s_cnt[k] = acc; acc += n; } }
    __syncthreads();
    for (uint32_t p = tid; p < np; p += ST_THREADS) { const uint32_t m = (uint32_t)(a.op_first[j0 + p + 1] - a.op_first[j0 + p]); s_order[atomicAdd(&s_cnt[min(m, (uint32_t)ST_MAXM + 1)], 1u)] = (uint8_t)p; }
    __syncthreads();
    const XlateStaged xl{s_sbase, s_g0};
    const int ncols_s = WIDE ? 0 : sP->mcols;
    MCell merged_local[WIDE ? MAXCOLS : 1];
    MCell* merged = WIDE ? merged_local : cells + (size_t)tid * ncols_s;
    DT open_dt[ST_MAXM];
    StatAcc acc; acc.init(sP->now, a.td);
    for (uint32_t t = tid; t < np; t += ST_THREADS) {
        const uint32_t j = j0 + s_order[t];
        const uint64_t cj = a.op_first[j]; const uint32_t m = (uint32_t)(a.op_first[j + 1] - cj);
        // the largest fan-in among the lanes that walk this round together (a subset of the warp is fine: it is only a loop bound)
        const uint32_t m_uni = min((uint32_t)ST_MAXM, __reduce_max_sync(__activemask(), m));
        uint8_t *dout, *iout; uint64_t dcap, dposv; uint32_t nbf, ipf, ixs_cap;
        if (!k4_prologue<true>(a, j, dout, dcap, dposv, iout, nbf, ipf, ixs_cap)) continue;
        PartOut out{0, 0, 0, 0, 0}; PartStats st{0, 0}; int e = 0;
        if (m > (uint32_t)ST_MAXM || cj - c0 + m > (uint64_t)ST_CUR_CAP) e = PERR_UNSUPPORTED;
        else process_partition<true>(*sP, xl, a.contrib, cj, m, a.upos, a.pbase, a.kp, a.klen, a.tok, dout, dcap, dposv, iout, nbf, ipf, ixs_cap, curs + (cj - c0), open_dt, merged, out, st, e,
                                     a.sg ? &acc : nullptr, m_uni);
        k4_epilogue<true>(a, j, cj, out, st, e);
    }
    if (a.sg) stat_flush_warp(a.sg, acc);               // (no thread returns after the barrier wait: every lane gets here)
}

// ---- K4 statistics pass of one output file (multi-file output with the side band) ---------------------------------------------------
// The file boundaries of a leveled compaction are known only after K5, so the per-cell / per-row reductions cannot come from the
// serialisation pass. Per file, this runs the same process_partition() again over the written partitions jlo <= j < jhi in the
// non-emitting (counting-sink) instantiation: nothing is written but the file's StatGlobal / TdropTable and ccount[j]. A kernel of
// its own, so that the serialisation kernels keep their code. Every fan-in class takes the thread-per-partition mapping (64 cursors
// per thread above 16; the warp kernels of those classes compute the same values). No lane returns early: the accumulators are folded
// per warp (stat_flush_warp) before the StatGlobal atomics, one flush per warp instead of one per partition. A partition the kernel
// refuses fails the call (the serialisation pass refused it first so far; a disagreement must not drop it from Statistics.db silently).
template <int M_CAP, int NT, bool CX>
__global__ void __launch_bounds__(NT) k_partition_stats(const K4Args a, uint64_t lo, uint64_t hi) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    const int ncols_s = a.P->mcols <= K4_SMEM_COLS ? a.P->mcols : 0;
    const int stride = M_CAP * SLOT_BYTES + ncols_s * (int)sizeof(MCell) + 8;
    K4Cur* cur = (K4Cur*)(s_raw + (size_t)threadIdx.x * stride);
    MCell merged_local[MAXCOLS];
    MCell* merged = ncols_s ? (MCell*)(cur + M_CAP) : merged_local;
    DT open_dt[M_CAP];
    StatAcc acc; acc.init(a.P->now, a.td);
    const uint64_t t = lo + (uint64_t)blockIdx.x * NT + threadIdx.x;
    uint64_t j = 0; bool work = t < hi;
    if (work) { j = a.list[t]; work = j >= a.jlo && j < a.jhi && a.dsize[j]; }
    if (work) {
        const uint64_t c0 = a.op_first[j]; const uint32_t m = (uint32_t)(a.op_first[j + 1] - c0);
        PartOut out{0, 0, 0, 0, 0}; PartStats st{0, 0}; int e = 0;
        if (m > (uint32_t)M_CAP) e = PERR_UNSUPPORTED;
        else process_partition<false, K4Cur, XlateGlobal, M_CAP, CX>(*a.P, XlateGlobal(), a.contrib, c0, m, a.upos, a.pbase, a.kp, a.klen, a.tok, nullptr, ~0ull, 0, nullptr, 0, 0, 0, cur, open_dt, merged, out, st, e, &acc);
        if (e) {
            const uint64_t en = a.contrib[c0]; const int src = (int)((en >> 56) & 0x7F);
            report_err(a.err, e == PERR_UNSUPPORTED ? 9 : 4, src, a.upos[a.pbase[src] + (en & 0xFFFFFFFFFFull)] - a.P->in[src].ubase);
            acc.init(a.P->now, a.td);
        } else a.ccount[j] = out.cells;
    }
    stat_flush_warp(a.sg, acc);                           // (block sizes are multiples of 32 and every lane gets here)
}

// upper bound of an output partition's size: the sum of its input partitions plus 25 % + 32 bytes (re-based deltas can lengthen
// vints by a byte or two per field; a partition that still does not fit is caught by the overflow flag and re-emitted by mode 3)
// icap[j]: bytes of promoted-index slot (0 when the partition cannot reach a second column-index block)
__global__ void __launch_bounds__(256) k_bounds(const uint64_t* __restrict__ contrib, const uint64_t* __restrict__ op_first, uint64_t nparts,
                                                const uint64_t* __restrict__ upos, const uint64_t* __restrict__ pbase, uint64_t* __restrict__ bound,
                                                uint32_t column_index_size, uint32_t* __restrict__ icap, uint32_t* __restrict__ insz, uint8_t* __restrict__ big) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nparts) return;
    uint64_t sum = 0;
    for (uint64_t c = op_first[j]; c < op_first[j + 1]; c++) { uint64_t e = contrib[c]; uint64_t g = pbase[(e >> 56) & 0x7F] + (e & 0xFFFFFFFFFFull); sum += upos[g + 1] - upos[g]; }
    uint64_t b = (sum + (sum >> 2) + 32 + 15) & ~15ull;
    bound[j] = b;
    insz[j] = (uint32_t)min(sum, (uint64_t)0xFFFFFFFFull);
    big[j] = (sum > (uint64_t)ST_MAXP || op_first[j + 1] - op_first[j] > (uint64_t)ST_MAXM) ? 1 : 0;      // not for the staged kernel
    uint64_t nb_max = b / column_index_size + 2;          // a block closes once it holds >= column_index_size bytes
    icap[j] = (b > column_index_size && nb_max < (1u << 23)) ? (uint32_t)(IXS_HEAD + nb_max * IXS_BLOCK_STRIDE) : 0u;
}

// scratch -> dense Data stream; one warp per output partition (partitions are tens of bytes to a few KB)
__global__ void __launch_bounds__(256) k_gather(uint64_t nparts, const uint64_t* __restrict__ dsize, const uint64_t* __restrict__ dpos, const uint64_t* __restrict__ bpos,
                                                const uint8_t* __restrict__ ovf, const uint8_t* __restrict__ scratch, uint8_t* __restrict__ uout) {
    uint64_t j = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= nparts) return;
    uint64_t n = dsize[j];
    if (!n || ovf[j]) return;
    const uint8_t* s = scratch + bpos[j]; uint8_t* d = uout + dpos[j];
    int lane = threadIdx.x & 31;
    for (uint64_t i = lane; i < n; i += 32) d[i] = s[i];
}

// Index.db entries of partitions without a promoted index: u16 keyLen | key | vint position | vint32 0  (RowIndexEntry.serialize :468-473)
__global__ void __launch_bounds__(256) k_index_simple(const CParams* __restrict__ Pp, uint64_t nparts, const uint64_t* __restrict__ contrib, const uint64_t* __restrict__ op_first,
        const uint64_t* __restrict__ upos, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ dsize, const uint64_t* __restrict__ dpos,
        const uint32_t* __restrict__ nblk, const uint8_t* __restrict__ ovf, const uint32_t* __restrict__ ihead, const uint64_t* __restrict__ ipos, uint8_t* __restrict__ iout) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nparts || !dsize[j] || nblk[j] > 1 || ovf[j]) return;
    uint64_t e = contrib[op_first[j]]; uint64_t g = pbase[(e >> 56) & 0x7F] + (e & 0xFFFFFFFFFFull);
    const uint8_t* k = Pp->U + upos[g];
    uint32_t n = ihead[j];                          // 2 + keyLen: the bytes are identical to the partition header in Data.db
    Sink<true> s{iout + ipos[j], 0, true, ~0ull};
    s.copy(k, n); s.vint(dpos[j]); s.u8(0);
}

// Index.db entries with a promoted index (IndexedEntry.serialize, S/io/sstable/format/big/RowIndexEntry.java:625-642), assembled from
// the slot the scratch pass filled: u16 keyLen | key | vint position | vint32 payload | vint headerLength | DeletionTime | vint32 nBlocks |
// IndexInfo x n | i32 offset x n
__global__ void __launch_bounds__(128) k_index_promoted(const CParams* __restrict__ Pp, uint64_t nparts, const uint64_t* __restrict__ contrib, const uint64_t* __restrict__ op_first,
        const uint64_t* __restrict__ upos, const uint64_t* __restrict__ pbase, const uint64_t* __restrict__ dsize, const uint64_t* __restrict__ dpos,
        const uint32_t* __restrict__ nblk, const uint8_t* __restrict__ ovf, const uint32_t* __restrict__ ihead, const uint32_t* __restrict__ ipay, const uint64_t* __restrict__ ipos,
        const uint64_t* __restrict__ ioff, const uint32_t* __restrict__ icap, const uint8_t* __restrict__ iscr, uint8_t* __restrict__ iout) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nparts || !dsize[j] || nblk[j] <= 1 || ovf[j]) return;
    uint64_t e = contrib[op_first[j]]; uint64_t g = pbase[(e >> 56) & 0x7F] + (e & 0xFFFFFFFFFFull);
    const uint8_t* k = Pp->U + upos[g];
    const uint8_t* slot = iscr + ioff[j];
    const uint32_t nb_max = (icap[j] - IXS_HEAD) / IXS_BLOCK_STRIDE, nb = nblk[j], n = ihead[j];
    DT pd; pd.mfda = ((const int64_t*)slot)[0]; pd.ldt = ((const int64_t*)slot)[1];
    const uint32_t pdsz = dt_is_live(pd) ? 1u : 12u, hdr_len = (uint32_t)((const int64_t*)slot)[2];     // key + partition deletion + static row
    const uint32_t infos = ipay[j] - vint_size(hdr_len) - pdsz - vint_size(nb) - 4 * nb;
    Sink<true> s{iout + ipos[j], 0, true, ~0ull};
    s.copy(k, n); s.vint(dpos[j]); s.vint(ipay[j]);
    s.vint(hdr_len); write_partition_dt(s, pd); s.vint(nb);
    s.copy(slot + IXS_HEAD + 4 * (size_t)nb_max, infos); s.copy(slot + IXS_HEAD, 4 * nb);
}

__global__ void __launch_bounds__(256) k_sum_stats(uint64_t nparts, const uint64_t* __restrict__ dsize, const uint32_t* __restrict__ st_munf, const uint32_t* __restrict__ st_rows, RunStats* __restrict__ stats) {
    unsigned long long a = 0, r = 0, w = 0;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nparts; j += (uint64_t)gridDim.x * blockDim.x) { a += st_munf[j]; r += st_rows[j]; w += dsize[j] ? 1 : 0; }
#pragma unroll
    for (int d = 16; d; d >>= 1) { a += __shfl_xor_sync(FULL_MASK, a, d); r += __shfl_xor_sync(FULL_MASK, r, d); w += __shfl_xor_sync(FULL_MASK, w, d); }
    if ((threadIdx.x & 31) == 0) { if (a) atomicAdd(&stats->merged_unfiltereds, a); if (r) atomicAdd(&stats->rows_out, r); if (w) atomicAdd(&stats->partitions_out, w); }
}

// Index.db entry size once the data position is known: u16 keyLen | key | vint position | vint32 payload size | payload
__global__ void __launch_bounds__(256) k_index_sizes(uint64_t nparts, const uint64_t* __restrict__ dsize, const uint64_t* __restrict__ dpos,
                                                     const uint32_t* __restrict__ ipay, const uint32_t* __restrict__ ihead, uint32_t* __restrict__ isize) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nparts) return;
    isize[j] = dsize[j] ? ihead[j] + vint_size(dpos[j]) + vint_size(ipay[j]) + ipay[j] : 0;
}

// ---- LCS output switching (MaxSSTableSizeWriter.shouldSwitchWriterInCurrentLocation, S/db/compaction/writers/MaxSSTableSizeWriter.java:76-79;
// CompactionAwareWriter.maybeSwitchWriter :166-173): before each partition the writer starts a new file when the bytes already
// flushed to disk (whole compressed chunks + CRCs) exceed the limit. woffs = exclusive scan of the compressed chunk sizes of the
// window that starts at byte start_b of the merged stream.
__global__ void k_find_cut(const uint64_t* __restrict__ dpos, uint64_t jlo, uint64_t nparts, uint64_t start_b, const uint64_t* __restrict__ woffs,
                           uint64_t nwin, uint32_t L, uint64_t limit, uint64_t* __restrict__ out /*[0]=j, [1]=status 0 found / 1 end / 2 need a longer window*/) {
    uint64_t a = jlo + 1, b = nparts;
    // chunks already FLUSHED when the writer stands at byte x of the file: the buffer is flushed lazily, when the next byte needs room
    // (BufferedDataOutputStreamPlus.write S/io/util/BufferedDataOutputStreamPlus.java:87-139), so a chunk that is exactly full is still
    // in memory and does not count towards getEstimatedOnDiskBytesWritten (CompressedSequentialWriter.java:128-131)
    auto flushed = [&](uint64_t x) -> uint64_t { return x ? (x - 1) / L : 0; };
    while (a < b) {
        uint64_t mid = (a + b) / 2; uint64_t full = flushed(dpos[mid] - start_b);
        bool cond = full > nwin || woffs[full] > limit;
        if (cond) b = mid; else a = mid + 1;
    }
    out[0] = a;
    if (a >= nparts) { out[1] = 1; return; }
    uint64_t full = flushed(dpos[a] - start_b);
    out[1] = full > nwin ? 2 : 0;
}
__global__ void __launch_bounds__(256) k_rel_pos(const uint64_t* __restrict__ dpos, uint64_t jlo, uint64_t jhi, uint64_t start_b, uint64_t* __restrict__ dposf) {
    uint64_t j = jlo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j <= jhi) dposf[j] = dpos[j] - start_b;
}

} // namespace b200c

// ---------------------------------------------------------------------------------------------------------------------------------
extern "C" {

int b200c_compact(b200c_ctx* c, const b200c_manifest* m, b200c_result* res, int flags) {
    if (!c || !m || !res) return B200C_EINVAL;
    auto t_start = std::chrono::steady_clock::now();
    cudaSetDevice(c->device);
    c->prog_stage.store(0); c->prog_scanned.store(0);
    for (int i = 0; i < B200C_MAX_INPUTS; i++) c->prog_input_pos[i].store(0);
    c->prog_seq.fetch_add(1);              // after the resets: figures read behind a new call_seq belong to this call
    if (m->abi_version != B200C_ABI_VERSION || m->ninputs <= 0) { c->err = "bad manifest"; return B200C_EINVAL; }
    if (m->partitioner != B200C_PARTITIONER_MURMUR3 && m->partitioner != B200C_PARTITIONER_BYTE_ORDERED) { c->err = "partitioner not supported (Murmur3Partitioner and ByteOrderedPartitioner are)"; return B200C_EUNSUPPORTED; }
    if (m->partitioner == B200C_PARTITIONER_BYTE_ORDERED && (m->token_lo != INT64_MIN || m->token_hi != INT64_MAX || m->npurge_ranges)) { c->err = "ByteOrderedPartitioner: token sub-ranges are not expressible"; return B200C_EUNSUPPORTED; }
    if (m->npurge_ranges < 0 || (m->npurge_ranges && (!m->purge_range_hi || !m->purge_range_max_ts))) { c->err = "purge table"; return B200C_EINVAL; }
    for (int k = 1; k < m->npurge_ranges; k++) if (m->purge_range_hi[k] <= m->purge_range_hi[k - 1]) { c->err = "purge_range_hi must ascend"; return B200C_EINVAL; }
    if (c->cancel.exchange(0)) { c->err = "cancelled"; return B200C_ECANCELLED; }        // stop requested before the task got here
    // the rest of the sstable (Filter.db / Summary.db / Statistics.db side band / first+last key), per output file; output 0 says which parts
    const b200c_output& o0 = res->outputs[0];
    const bool want_meta = o0.key_buf || o0.filter || o0.summary || o0.stats;
    if (want_meta && getenv("B200C_K4_TWO_PASS")) { c->err = "metadata side band with the two-pass K4 mode (B200C_K4_TWO_PASS)"; return B200C_EUNSUPPORTED; }
    if (want_meta && o0.filter && m->bloom_words && (m->bloom_hash_count <= 0 || m->bloom_words > (1ull << 31))) { c->err = "bloom geometry"; return B200C_EINVAL; }
    if (m->ninputs > MAXK) { c->err = "more than 64 inputs per call"; return B200C_EUNSUPPORTED; }
    if (m->tombstone_option != 0 || m->enforce_strict_liveness) { c->err = "tombstone_option / strict liveness"; return B200C_EUNSUPPORTED; }
    if (m->nstatic_columns < 0 || m->nstatic_columns > MAXSTAT) { c->err = "more than 16 static columns"; return B200C_EUNSUPPORTED; }
    if (m->nclustering > MAXCLUST || m->ncolumns >= 64 || m->ncolumns < 0) { c->err = "schema outside the supported envelope"; return B200C_EUNSUPPORTED; }
    for (int k = 0; k < m->nstatic_columns; k++) if ((m->static_columns[k].type >> 8) & 0xFF) { c->err = "multi-cell static column"; return B200C_EUNSUPPORTED; }
    if (res->noutputs_cap < 1 || !res->outputs) { c->err = "no output slot"; return B200C_EINVAL; }
    if (m->out_chunk_len <= 0 || m->out_chunk_len > 65536 || (m->out_chunk_len & (m->out_chunk_len - 1))) { c->err = "output chunk_len"; return B200C_EUNSUPPORTED; }
    const bool dev = flags & B200C_FLAG_DEVICE_PTRS;
    const bool lcs = m->max_sstable_bytes != 0;
    const int K = m->ninputs;
    // whatever way this call ends, nothing may still be copying from or into the caller's buffers
    struct CopyGuard { b200c_ctx* c; cudaStream_t main; ~CopyGuard() { c->stream = main; cudaStreamSynchronize(c->stream5); cudaStreamSynchronize(c->copy_stream); cudaStreamSynchronize(c->copy_out); } } copy_guard{c, c->stream};

    // ---- Index.db slices: a token sub-range with Summary.db samples touches only its part of every Index.db ------------------------------
    bool have_summaries = true;
    for (int i = 0; i < K; i++) if (m->inputs[i].index_len && !(m->inputs[i].summary_positions && m->inputs[i].nsummary)) have_summaries = false;
    const bool sliced = have_summaries && !lcs && (m->token_lo != INT64_MIN || m->token_hi != INT64_MAX) && !getenv("B200C_NO_INDEX_SLICES");
    std::vector<IdxSlice> isl(K);
    for (int i = 0; i < K; i++) isl[i] = IdxSlice{0, m->inputs[i].index_len, m->inputs[i].data_length, 0, have_summaries ? m->inputs[i].nsummary : 0};
    if (sliced) {
        if (!dev) {
            for (int i = 0; i < K; i++) { const b200c_input& in = m->inputs[i];
                if (in.index_len && !compute_index_slice(in.index, in.index_len, in.summary_positions, in.nsummary, in.data_length, m->partitioner, m->token_lo, m->token_hi, &isl[i])) {
                    c->err = "Summary.db positions of input " + std::to_string(i) + " do not point at Index.db entries"; res->corruption.input = i; res->corruption.kind = 3; res->corruption.chunk = 0; res->corruption.offset = 0; return B200C_ECORRUPT; } }
        } else {
            uint8_t* w; B200C_TRY(ws_typed(c, WS_SLICE, (size_t)K * (8 * 5 + sizeof(IdxSlice) + 4) + 64, &w));
            std::vector<uint64_t> hv((size_t)K * 5);
            for (int i = 0; i < K; i++) { const b200c_input& in = m->inputs[i]; hv[i] = (uint64_t)(uintptr_t)in.index; hv[K + i] = in.index_len; hv[2 * K + i] = (uint64_t)(uintptr_t)in.summary_positions; hv[3 * K + i] = in.nsummary; hv[4 * K + i] = in.data_length; }
            uint64_t* dv = (uint64_t*)w; IdxSlice* dsl = (IdxSlice*)(dv + 5 * K); uint32_t* dok = (uint32_t*)(dsl + K);
            B200C_CUDA_TRY(c, cudaMemcpyAsync(dv, hv.data(), hv.size() * 8, cudaMemcpyHostToDevice, c->stream));
            k_index_slices<<<(K + 63) / 64, 64, 0, c->stream>>>((const uint8_t* const*)dv, dv + K, (const uint64_t* const*)(dv + 2 * K), dv + 3 * K, dv + 4 * K, K, m->partitioner, m->token_lo, m->token_hi, dsl, dok);
            std::vector<uint32_t> ok(K);
            B200C_CUDA_TRY(c, cudaMemcpyAsync(isl.data(), dsl, sizeof(IdxSlice) * K, cudaMemcpyDeviceToHost, c->stream));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(ok.data(), dok, 4 * K, cudaMemcpyDeviceToHost, c->stream));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            for (int i = 0; i < K; i++) if (m->inputs[i].index_len && !ok[i]) { c->err = "Summary.db positions of input " + std::to_string(i) + " do not point at Index.db entries"; res->corruption.input = i; res->corruption.kind = 3; res->corruption.chunk = 0; res->corruption.offset = 0; return B200C_ECORRUPT; }
                         else if (!m->inputs[i].index_len) isl[i] = IdxSlice{0, 0, m->inputs[i].data_length, 0, 0};
        }
    }

    // ---- layout of the concatenated device buffers -------------------------------------------------------------------------------
    std::vector<uint64_t> ubase(K + 1), ibase(K + 1), cbase(K + 1), obase(K + 1), bbase(K + 1);
    CParams hp; memset(&hp, 0, sizeof(hp));
    std::vector<InDesc> hin(K); memset(hin.data(), 0, sizeof(InDesc) * K);
    uint64_t uo = 0, io = 0, co = 0, oo = 0, bo = 0;
    for (int i = 0; i < K; i++) {
        const b200c_input& in = m->inputs[i];
        if (in.chunk_len <= 0 || in.chunk_len > 65536 || (in.chunk_len & (in.chunk_len - 1))) { c->err = "input chunk_len"; return B200C_EUNSUPPORTED; }
        if (in.ncolumns < 0 || in.ncolumns >= 64) { c->err = "input columns"; return B200C_EUNSUPPORTED; }
        if (in.nchunks != (in.data_length + in.chunk_len - 1) / (uint64_t)in.chunk_len) { c->err = "chunk count does not match data_length"; return B200C_EINVAL; }
        if (in.compressor != COMP_LZ4 && !comp_is_snappy(in.compressor) && in.compressor != COMP_NONE) { c->err = "unknown compressor"; return B200C_EINVAL; }
        ubase[i] = uo; uo += (in.data_length + 64 + 65535) & ~65535ull;
        const uint64_t ilen_i = isl[i].hi - isl[i].lo;               // Index.db bytes this call reads from input i
        ibase[i] = io; io += (ilen_i + 64 + 255) & ~255ull;
        cbase[i] = co; co += (in.data_len + 64 + 255) & ~255ull;
        obase[i] = oo; oo += in.nchunks + 1;
        bbase[i] = bo; bo += (ilen_i + IB - 1) / IB;
        InDesc& d = hin[i];
        d.ubase = ubase[i]; d.ulen = in.data_length; d.ibase = ibase[i]; d.ilen = ilen_i; d.uend = isl[i].uend;
        d.min_ts = in.header_stats.min_timestamp; d.min_ldt = in.header_stats.min_local_deletion_time; d.min_ttl = in.header_stats.min_ttl;
        d.ncols = in.ncolumns;
        for (int k = 0; k < in.ncolumns; k++) {
            if (in.column_map[k] < 0 || in.column_map[k] >= m->ncolumns || (k && in.column_map[k] <= in.column_map[k - 1])) { c->err = "column_map must be strictly increasing (both headers are name ordered)"; return B200C_EINVAL; }
            d.colmap[k] = in.column_map[k];
        }
        d.nstat = in.nstatic_columns; d._pad = 0;
        if (in.nstatic_columns < 0 || in.nstatic_columns > m->nstatic_columns) { c->err = "input static columns"; return B200C_EINVAL; }
        for (int k = 0; k < in.nstatic_columns; k++) {
            if (in.static_column_map[k] < 0 || in.static_column_map[k] >= m->nstatic_columns || (k && in.static_column_map[k] <= in.static_column_map[k - 1])) { c->err = "static_column_map must be strictly increasing"; return B200C_EINVAL; }
            d.smap[k] = in.static_column_map[k];
        }
    }
    ubase[K] = uo; ibase[K] = io; cbase[K] = co; obase[K] = oo; bbase[K] = bo;
    if (uo >= (1ull << 40)) { c->err = "decompressed inputs of 1 TiB or more per call"; return B200C_EUNSUPPORTED; }      // stream offsets are 40-bit in the K4 cursors
    (void)bo;
    hp.ninputs = K; hp.nclust = m->nclustering; hp.ncols = m->ncolumns; hp.column_index_size = m->column_index_size > 0 ? m->column_index_size : 65536;
    for (int k = 0; k < m->nclustering; k++) { hp.ctype[k] = m->clustering[k].type; hp.cfix[k] = m->clustering[k].fixed_len; }
    for (int k = 0; k < m->ncolumns; k++) {                 // multi-cell columns: include/b200c.h B200C_COLUMN_COMPLEX / _FIXED; they follow the simple ones
        const int ptype = ((m->columns[k].type >> 8) & 0xFF) - 1;
        hp.vfix[k] = m->columns[k].fixed_len & 0xFFFF;
        if (ptype >= 0) {
            if (ptype > TYPE_TIMEUUID) { c->err = "cell path class"; return B200C_EINVAL; }
            if (hp.ncx >= MAXCX) { c->err = "more than 8 multi-cell columns"; return B200C_EUNSUPPORTED; }
            if (!hp.ncx) hp.cx_first = k;
            hp.ptype[hp.ncx] = ptype; hp.pfix[hp.ncx] = (int32_t)((uint32_t)m->columns[k].fixed_len >> 16); hp.ncx++;
        } else if (hp.ncx) { c->err = "simple column behind a multi-cell one (ColumnMetadata order: simple columns first)"; return B200C_EINVAL; }
        if ((m->columns[k].type & 0xFF) == B200C_TYPE_COUNTER) {      // counter columns: cells merged shard by shard (partition.cuh ctr_merge), CX kernels
            if (ptype >= 0) { c->err = "collection of counters"; return B200C_EINVAL; }
            hp.ctr_mask |= 1ull << k;
        }
    }
    if (!hp.ncx) hp.cx_first = m->ncolumns;
    for (int k = 0; k < m->nstatic_columns; k++) if ((m->static_columns[k].type & 0xFF) == B200C_TYPE_COUNTER) hp.sctr_mask |= 1ull << k;
    hp.nstat = m->nstatic_columns; hp.mcols = std::max(m->ncolumns, m->nstatic_columns);
    for (int k = 0; k < m->nstatic_columns; k++) hp.sfix[k] = m->static_columns[k].fixed_len;
    hp.o_min_ts = m->out_stats.min_timestamp; hp.o_min_ldt = m->out_stats.min_local_deletion_time; hp.o_min_ttl = m->out_stats.min_ttl;
    hp.now = m->now_in_sec; hp.gc_before = m->gc_before; hp.purge_max_ts = m->purge_max_timestamp;
    hp.partitioner = m->partitioner;

    // Token-range streaming (host buffers, one output file): Index.db goes to the device first; once K2 has turned it into tokens and
    // positions the token space is cut into `want_ranges` pieces, the Data.db chunks each piece needs are copied piece by piece on the
    // copy stream, and K1/K3/K4/K5 of piece r run underneath the copies of the pieces after it and the read-back of the pieces before
    // it. Device-resident inputs and multi-file (LCS) outputs run as one piece.
    // Piece boundaries as fractions of the token-sorted input: small pieces first (the kernels can start as soon as little data
    // has arrived), doubling afterwards (few pieces = little per-piece overhead). B200C_RANGES=n forces n equal pieces (tests, tuning).
    std::vector<double> cuts; bool forced_ranges = false;          // interior cut points in (0, 1)
    if (!dev && !lcs) {
        if (const char* e = getenv("B200C_RANGES")) {
            int n = std::max(1, std::min((int)MAX_RANGES, atoi(e))); forced_ranges = true;
            for (int r = 1; r < n; r++) cuts.push_back((double)r / n);
        } else if (co >= (1536ull << 20)) {
            // The kernels of a piece take longer than its copies (configs[1]: 430 ms of kernels, 320 ms of PCIe), so the pipeline is kernel
            // bound as long as no piece waits for its own data: a small first piece (the kernels start early), then EQUAL pieces. Doubling
            // pieces (B200C_SCHEDULE=geometric, the round-1 schedule) end with a piece of half the input that cannot start before the
            // last byte has arrived: 84 ms of idle kernels on configs[1].
            const double f0 = std::min(0.5, std::max(1.0 / 16, (double)(512ull << 20) / (double)co));
            const char* sch = getenv("B200C_SCHEDULE");
            if (sch && !strcmp(sch, "geometric")) { for (double f = f0; f < 1.0 && cuts.size() + 1 < MAX_RANGES; f *= 2) cuts.push_back(f); }
            else {
                const double piece = std::max((double)co / 8, (double)(768ull << 20));
                int n = (int)std::ceil((1.0 - f0) * (double)co / piece); n = std::max(1, std::min(n, (int)MAX_RANGES - 1));
                for (int k = 0; k < n; k++) cuts.push_back(f0 + (1.0 - f0) * k / n);
            }
        }
    }
    int want_ranges = (int)cuts.size() + 1;
    // with Summary.db positions for every input the Index.db walk does not need Data.db: its copies are then scheduled after K2.
    // Device-resident inputs take the same route when the call is a token sub-range: K2 first, then only the chunks the range crosses are decoded.
    const bool deferred = !lcs && have_summaries && (!dev || sliced);
    if (!deferred) { want_ranges = 1; cuts.clear(); }
    // Index.db streaming (host buffers, several pieces): the pieces are cut on the HOST, at tokens of Summary.db samples of the input with the
    // most samples, and every piece brings its own Index.db slices (the samples bracketing its token range, as a ranged scanner would seek),
    // its Summary positions and its Data.db chunks. K2 runs per piece: nothing waits for the whole Index.db (4.3 GB = 80 ms of PCIe on
    // configs[1]) any more, and the per-partition arrays are piece sized.
    std::vector<int64_t> T{m->token_lo, m->token_hi};
    std::vector<std::vector<IdxSlice>> psl(1, isl);                 // per piece and input: Index.db slice ...
    std::vector<uint64_t> pustart((size_t)K, 0);                    // ... and where the Data.db bytes its entries describe start ([ustart, slice.uend))
    bool istream = false;
    if (deferred && !dev && want_ranges > 1) {
        // Summary.db is a hint here as everywhere: if its positions do not parse or the slices they give do not tile the call's own
        // slice, the call runs as one piece (K2 over the whole Index.db, as before)
        auto plan = [&]() -> bool {
            int imax = 0; uint64_t nmax = 0;
            for (int i = 0; i < K; i++) if (isl[i].s_count > nmax) { nmax = isl[i].s_count; imax = i; }
            if (nmax < (uint64_t)want_ranges * (forced_ranges ? 1 : 32)) return false;
            const b200c_input& big = m->inputs[imax];
            std::vector<int64_t> t2{m->token_lo};
            for (int r = 1; r < want_ranges; r++) {
                const uint64_t sidx = isl[imax].s_first + std::min<uint64_t>(nmax - 1, (uint64_t)(nmax * cuts[r - 1]));
                int64_t t = 0;
                if (!sample_token(big.index, big.index_len, big.summary_positions[sidx], m->partitioner, &t)) return false;
                if (t > t2.back() && t < m->token_hi) t2.push_back(t);
            }
            t2.push_back(m->token_hi);
            const int n2 = (int)t2.size() - 1;
            if (n2 < 2) return false;
            std::vector<std::vector<IdxSlice>> p2(n2, isl); std::vector<uint64_t> u2((size_t)n2 * K, 0);
            for (int r = 0; r < n2; r++) for (int i = 0; i < K; i++) {
                const b200c_input& in = m->inputs[i];
                IdxSlice& sl = p2[r][i];
                if (!in.index_len) { sl = IdxSlice{0, 0, in.data_length, 0, 0}; u2[(size_t)r * K + i] = in.data_length; continue; }
                if (!compute_index_slice(in.index, in.index_len, in.summary_positions, in.nsummary, in.data_length, m->partitioner, t2[r], t2[r + 1], &sl)) return false;
                // every entry must lie in some piece's slice: consecutive slices touch or overlap, the first starts and the last ends with the call's own
                if (r == 0 && sl.lo != isl[i].lo) return false;
                if (r == n2 - 1 && sl.hi != isl[i].hi) return false;
                if (r > 0 && (sl.lo > p2[r - 1][i].hi || sl.lo < p2[r - 1][i].lo || sl.hi < p2[r - 1][i].hi)) return false;
                uint64_t pos = sl.uend;
                if (sl.hi > sl.lo && !entry_data_position(in.index, in.index_len, sl.lo, in.data_length, &pos)) return false;
                if (pos > sl.uend) return false;
                u2[(size_t)r * K + i] = pos;
            }
            T = t2; psl = p2; pustart = u2;
            return true;
        };
        istream = plan();
    }
    const int nr = (int)T.size() - 1;
    uint8_t *U, *CD, *IDX; uint64_t* CO; CParams* dP; uint64_t* d_bbase; DevErr* d_err; ChunkErr* d_cerr; RunStats* d_stats; unsigned long long* d_hist;
    B200C_TRY(ws_typed(c, WS_U, uo + 64, &U));
    B200C_TRY(ws_typed(c, WS_CD, co + 64, &CD));
    B200C_TRY(ws_typed(c, WS_CO, oo + 1, &CO));
    B200C_TRY(ws_typed(c, WS_IDX, io + 64, &IDX));
    // Summary.db positions on the device: one run per piece and input (file offsets; K2 subtracts the slice start — no kernel rides on the copy stream)
    std::vector<std::vector<uint64_t>> psb(nr, std::vector<uint64_t>(K + 1, 0));
    uint64_t summ_total = 0;
    for (int r = 0; r < nr; r++) for (int i = 0; i <= K; i++) { psb[r][i] = summ_total; if (i < K) summ_total += psl[r][i].s_count; }
    uint64_t* d_summ; B200C_TRY(ws_typed(c, WS_SUMM, summ_total + 1, &d_summ));
    { uint8_t* pp; B200C_TRY(ws_typed(c, WS_PARAMS, sizeof(CParams) + sizeof(InDesc) * (size_t)K, &pp)); dP = (CParams*)pp; hp.in = (const InDesc*)(pp + sizeof(CParams)); }
    B200C_TRY(ws_typed(c, WS_BBASE, (size_t)K + 1, &d_bbase));
    { uint8_t* p; B200C_TRY(ws_typed(c, WS_ERR2, 4096, &p)); d_err = (DevErr*)p; d_cerr = (ChunkErr*)(p + 64); d_stats = (RunStats*)(p + 128); d_hist = (unsigned long long*)(p + 256); }
    hp.U = U;
    cudaStream_t st = c->stream;
    if (m->npurge_ranges) {
        int64_t* d_pt; B200C_TRY(ws_typed(c, WS_PURGE, 2 * (size_t)m->npurge_ranges, &d_pt));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_pt, m->purge_range_hi, 8 * (size_t)m->npurge_ranges, cudaMemcpyHostToDevice, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_pt + m->npurge_ranges, m->purge_range_max_ts, 8 * (size_t)m->npurge_ranges, cudaMemcpyHostToDevice, st));
        hp.purge_hi = d_pt; hp.purge_ts = d_pt + m->npurge_ranges; hp.npurge = m->npurge_ranges;
    }
    // metadata state (meta.cuh), device resident across the pieces of the call
    StatGlobal* d_sg = nullptr; TdropTable* d_td = nullptr; uint32_t* d_bloom = nullptr; uint8_t* d_mkeys = nullptr;
    uint64_t written_total = 0, samples_total = 0; uint8_t* d_sument = nullptr; uint64_t* d_sumoff = nullptr; uint64_t sument_bound = 0;
    const uint32_t meta_interval = m->min_index_interval > 0 ? (uint32_t)m->min_index_interval : 128u;
    const uint64_t bloom_words = (want_meta && o0.filter) ? m->bloom_words : 0;
    std::vector<uint8_t> sg_init(want_meta ? sizeof(StatGlobal) : 0, 0);          // initial StatGlobal (a multi-file call resets to it per file)
    if (want_meta) {
        B200C_TRY(ws_typed(c, WS_META_SG, 1, &d_sg));
        B200C_TRY(ws_typed(c, WS_META_TD, 1, &d_td));
        B200C_TRY(ws_typed(c, WS_META_BLOOM, bloom_words * 2 + 16, &d_bloom));
        B200C_TRY(ws_typed(c, WS_META_KEYS, (size_t)2 * 65536, &d_mkeys));
        StatGlobal* g0 = (StatGlobal*)sg_init.data();
        g0->min_ts = I64_MAX; g0->max_ts = I64_MIN; g0->min_ldt = I64_MAX; g0->max_ldt = I64_MIN; g0->min_ttl = INT_MAX; g0->max_ttl = INT_MIN;
        auto offsets = [](long long* o, int n) { long long last = 1; o[0] = 1; for (int i = 1; i < n; i++) { long long next = llround((double)last * 1.2); if (next == last) next++; o[i] = next; last = next; } };
        offsets(g0->psize_off, META_PSIZE - 1); offsets(g0->cells_off, META_CELLS - 1);       // EstimatedHistogram.newOffsets (S/utils/EstimatedHistogram.java:91-109)
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_sg, sg_init.data(), sizeof(StatGlobal), cudaMemcpyHostToDevice, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));                                            // (sg_init is pageable host memory)
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_td, 0, sizeof(TdropTable), st));
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_td->key, 0xFF, sizeof(d_td->key), st));
        if (bloom_words) B200C_CUDA_TRY(c, cudaMemsetAsync(d_bloom, 0, bloom_words * 8, st));
    }
    B200C_CUDA_TRY(c, cudaMemsetAsync(d_err, 0xFF, 64, st));
    B200C_CUDA_TRY(c, cudaMemsetAsync(d_cerr, 0xFF, 64, st));
    B200C_CUDA_TRY(c, cudaMemsetAsync(d_stats, 0, 128 + MAXK * 8 + 128, st));
    B200C_CUDA_TRY(c, cudaMemcpyAsync((void*)hp.in, hin.data(), sizeof(InDesc) * (size_t)K, cudaMemcpyHostToDevice, st));
    B200C_CUDA_TRY(c, cudaMemcpyAsync(dP, &hp, sizeof(hp), cudaMemcpyHostToDevice, st));
    B200C_CUDA_TRY(c, cudaMemcpyAsync(d_bbase, bbase.data(), (K + 1) * 8, cudaMemcpyHostToDevice, st));
    cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    uint64_t bytes_read = 0;
    // inputs are staged on a second stream, one event per input, so that the kernels of input i overlap the copy of input i+1
    // (the workspace was possibly re-allocated above: make sure that is ordered before the copies)
    cudaStream_t cs = c->copy_stream;
    B200C_CUDA_TRY(c, cudaEventRecord(c->ev0, st));
    B200C_CUDA_TRY(c, cudaStreamWaitEvent(cs, c->ev0, 0));
    std::vector<uint64_t> h2d_next(K, 0), k1_next(K, 0);      // deferred mode: first chunk of input i not yet copied / not yet decompressed
    // device-resident inputs taking the piece route (a token sub-range): the host schedules the chunk-range copies, so it needs the offsets too
    std::vector<std::vector<uint64_t>> co_host(dev && deferred ? K : 0);
    for (size_t i = 0; i < co_host.size(); i++) {
        co_host[i].resize(m->inputs[i].nchunks);
        if (m->inputs[i].nchunks) B200C_CUDA_TRY(c, cudaMemcpyAsync(co_host[i].data(), m->inputs[i].chunk_offsets, m->inputs[i].nchunks * 8, cudaMemcpyDeviceToHost, cs));
    }
    if (!co_host.empty()) B200C_CUDA_TRY(c, cudaStreamSynchronize(cs));
    auto chunk_off = [&](int i, uint64_t ch) -> uint64_t { const b200c_input& in = m->inputs[i]; return ch >= in.nchunks ? in.data_len : (co_host.empty() ? in.chunk_offsets[ch] : co_host[i][ch]); };
    auto copy_chunks = [&](int i, uint64_t a, uint64_t b) -> int {      // compressed bytes of chunks [a, b) of input i -> CD
        const b200c_input& in = m->inputs[i];
        if (a >= b) return B200C_OK;
        uint64_t lo = chunk_off(i, a), hi = chunk_off(i, b);
        if (lo > hi || hi > in.data_len) { c->err = "chunk offsets of input " + std::to_string(i) + " are not increasing"; res->corruption.input = i; res->corruption.kind = 2; res->corruption.chunk = a; res->corruption.offset = 0; return B200C_ECORRUPT; }
        if (hi > lo) B200C_CUDA_TRY(c, cudaMemcpyAsync(CD + cbase[i] + lo, in.data + lo, hi - lo, kind, cs));
        return B200C_OK;
    };
    // what each piece needs from each input: chunks to copy (deferred mode) and to decompress
    struct Need { uint64_t h2d_a, h2d_b, k1_a, k1_b; };
    std::vector<Need> need((size_t)nr * K, Need{0, 0, 0, 0});
    std::vector<uint64_t> range_bytes(nr, 0);
    std::vector<uint64_t> range_end((size_t)nr * K, 0);          // per piece and input: Data.db position behind the piece (scanner accounting)
    for (int i = 0; i < K; i++) { bytes_read += m->inputs[i].data_length; range_end[(size_t)(nr - 1) * K + i] = m->inputs[i].data_length; }
    for (int r = 0; r < nr; r++) range_bytes[r] = bytes_read;
    auto need_of = [&](int r, int i, uint64_t a, uint64_t b) {      // piece r reads bytes [a, b) of input i's decompressed stream
        const b200c_input& in = m->inputs[i];
        range_end[(size_t)r * K + i] = b;
        Need& nd = need[(size_t)r * K + i];
        if (b > a) {
            uint64_t ca = a / in.chunk_len, cb = std::min<uint64_t>(in.nchunks, (b + in.chunk_len - 1) / in.chunk_len);
            nd.h2d_a = std::max(ca, h2d_next[i]); nd.h2d_b = std::max(cb, nd.h2d_a); h2d_next[i] = nd.h2d_b;
            nd.k1_a = std::max(ca, k1_next[i]); nd.k1_b = std::max(cb, nd.k1_a); k1_next[i] = nd.k1_b;
        }
    };
    for (int i = 0; i < K; i++) {
        const b200c_input& in = m->inputs[i];
        if (!deferred && in.data_len) B200C_CUDA_TRY(c, cudaMemcpyAsync(CD + cbase[i], in.data, in.data_len, kind, cs));
        if (in.nchunks) B200C_CUDA_TRY(c, cudaMemcpyAsync(CO + obase[i], in.chunk_offsets, in.nchunks * 8, kind, cs));
        if (!istream) {
            if (isl[i].hi > isl[i].lo) B200C_CUDA_TRY(c, cudaMemcpyAsync(IDX + ibase[i], in.index + isl[i].lo, isl[i].hi - isl[i].lo, kind, cs));
            if (isl[i].s_count) {
                B200C_CUDA_TRY(c, cudaMemcpyAsync(d_summ + psb[0][i], in.summary_positions + isl[i].s_first, isl[i].s_count * 8, kind, cs));
            }
        }
        B200C_CUDA_TRY(c, cudaEventRecord(c->ev_in[i], cs));
    }
    if (istream) {
        // piece after piece: the Index.db bytes not copied yet (consecutive slices overlap by a sample interval), the piece's Summary positions,
        // its Data.db chunks; EV_RANGE + r fires when piece r is on the device
        std::vector<uint64_t> idx_copied(K);
        for (int i = 0; i < K; i++) idx_copied[i] = isl[i].lo;
        for (int r = 0; r < nr; r++) {
            uint64_t tot = 0;
            for (int i = 0; i < K; i++) {
                const b200c_input& in = m->inputs[i]; const IdxSlice& sl = psl[r][i];
                const uint64_t from = std::max(sl.lo, idx_copied[i]);
                if (sl.hi > from) { B200C_CUDA_TRY(c, cudaMemcpyAsync(IDX + ibase[i] + (from - isl[i].lo), in.index + from, sl.hi - from, kind, cs)); idx_copied[i] = sl.hi; }
                if (sl.s_count) {
                    B200C_CUDA_TRY(c, cudaMemcpyAsync(d_summ + psb[r][i], in.summary_positions + sl.s_first, sl.s_count * 8, kind, cs));
                }
                need_of(r, i, pustart[(size_t)r * K + i], sl.uend);
                tot += sl.uend - pustart[(size_t)r * K + i];
                B200C_TRY(copy_chunks(i, need[(size_t)r * K + i].h2d_a, need[(size_t)r * K + i].h2d_b));
            }
            range_bytes[r] = tot;
            B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_RANGE + r], cs));
        }
    }
    c->prog_total.store(bytes_read); c->prog_scanned.store(0);
    for (int i = 0; i < K; i++) c->prog_input_pos[i].store(0);
    c->prog_ninputs.store(K);
    timing_begin(c);

    // stage clock: marks on the main stream; the time between two marks is charged to the stage of the first
    struct Mark { int stage; cudaEvent_t ev; };
    std::vector<Mark> marks;
    size_t k5_marks = 0;
    auto mark = [&](int stage) {
        size_t k = marks.size();
        if (k >= c->ev_marks.size()) { cudaEvent_t e; cudaEventCreate(&e); c->ev_marks.push_back(e); }
        cudaEventRecord(c->ev_marks[k], st); marks.push_back(Mark{stage, c->ev_marks[k]});
    };
    auto finish_marks = [&]() {
        for (int k = 0; k < 8; k++) c->stage_ms[k] = 0;
        for (size_t k = 0; k + 1 < marks.size(); k++) { float ms = 0; cudaEventElapsedTime(&ms, marks[k].ev, marks[k + 1].ev); if (marks[k].stage >= 0) c->stage_ms[marks[k].stage] += ms; }
        for (size_t k = 0; k + 1 < k5_marks; k += 2) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev_k5[k], c->ev_k5[k + 1]) == cudaSuccess) c->stage_ms[5] += ms; }      // K5 on stream5: overlaps the next piece's stages
        c->nstages = 6;
    };
    c->nstages = 0;
    mark(0);

    // ---- K1: decompress + verify (deferred mode: K1 runs per token range further down) ---------------------------------------------------
    c->prog_stage.store(1);
    auto k1 = [&](int i, uint64_t a, uint64_t b) -> int {           // chunks [a, b) of input i
        const b200c_input& in = m->inputs[i];
        if (a >= b) return B200C_OK;
        return decompress_stream_device(c, in.compressor, CD + cbase[i], in.data_len, CO + obase[i], in.nchunks, in.chunk_len,
                                        in.max_compressed_len, in.data_length, U + ubase[i], 1, d_cerr, a, b - a, i);
    };
    // several inputs' chunk ranges in one thread-per-chunk launch when there are enough of them (B200C_K1_BATCH=0 switches it off)
    const int k1_batch_env = []() { const char* e = getenv("B200C_K1_BATCH"); return e ? atoi(e) : (B200C_K1_BATCH_DEFAULT ? 1 : 0); }();     // 2: batch even tiny launches (tests)
    const bool k1_batching = k1_batch_env != 0;
    std::vector<K1Seg> segs; segs.reserve(K);
    auto k1_many = [&](const std::vector<uint64_t>& from, const std::vector<uint64_t>& to) -> int {      // chunks [from[i], to[i]) of every input
        segs.clear(); uint64_t total = 0;
        for (int i = 0; i < K && k1_batching; i++) {
            const b200c_input& in = m->inputs[i];
            if (from[i] >= to[i] || in.compressor != COMP_LZ4 || (in.chunk_len & 7)) continue;
            K1Seg g; memset(&g, 0, sizeof(g));
            g.data = CD + cbase[i]; g.data_len = in.data_len; g.offs = CO + obase[i]; g.nchunks = in.nchunks; g.data_length = in.data_length; g.out = U + ubase[i];
            g.chunk0 = from[i]; g.count = to[i] - from[i]; g.chunk_len = in.chunk_len; g.max_clen = in.max_compressed_len; g.tag = i;
            if (!dev || !co_host.empty()) { const uint64_t a = chunk_off(i, from[i]), b = chunk_off(i, to[i]); g.rec_span = b > a ? b - a : 0; }      // (0 / unknown: the whole file)
            segs.push_back(g); total += g.count;
        }
        const bool batched = total >= (k1_batch_env == 2 ? 1u : 32768u);
        if (batched) B200C_TRY(decompress_multi_device(c, segs.data(), (int)segs.size(), 1, d_cerr, WS_K1SEG));
        for (int i = 0; i < K; i++) {
            const b200c_input& in = m->inputs[i];
            if (batched && in.compressor == COMP_LZ4 && !(in.chunk_len & 7)) continue;
            B200C_TRY(k1(i, from[i], to[i]));
        }
        return B200C_OK;
    };
    for (int i = 0; i < K; i++) B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_in[i], 0));      // chunk offsets (and, unless the pieces bring their own, Index.db / Data.db) are there
    if (!deferred) {
        if (dev && k1_batching) {          // device-resident inputs: the staging copies are device-to-device, decode in one launch
            std::vector<uint64_t> z(K, 0), e(K);
            for (int i = 0; i < K; i++) e[i] = m->inputs[i].nchunks;
            B200C_TRY(k1_many(z, e));
        } else for (int i = 0; i < K; i++) B200C_TRY(k1(i, 0, m->inputs[i].nchunks));
    }
    uint64_t* h = (uint64_t*)c->h_pinned;
    // the request is consumed by the call that reports it (b200c.h: sticky until then, so one that lands before the call is not lost)
    auto check_cancel = [&]() -> int { if (c->cancel.exchange(0)) { c->err = "cancelled"; cudaStreamSynchronize(st); timing_end(c); return B200C_ECANCELLED; } return B200C_OK; };
    auto chunk_error = [&](uint64_t word) -> int {                  // word = d_cerr: (input << 48 | chunk << 8 | kind)
        int which = (int)(word >> 48), kindc = (int)(word & 0xff); uint64_t chunk = (word >> 8) & 0xFFFFFFFFFFull;
        res->corruption.input = which; res->corruption.kind = kindc; res->corruption.chunk = chunk; res->corruption.offset = 0;
        c->err = std::string(kindc == 1 ? "chunk CRC mismatch" : "malformed compressed chunk") + " in input " + std::to_string(which) + " chunk " + std::to_string(chunk);
        timing_end(c);
        return B200C_ECORRUPT;
    };
    auto index_data_mismatch = [&](uint64_t word) -> int {
        res->corruption.input = (int)((word >> 48) & 0xFF); res->corruption.kind = 3; res->corruption.chunk = 0; res->corruption.offset = word & 0xFFFFFFFFFFFFull;
        c->err = "Index.db does not match Data.db in input " + std::to_string(res->corruption.input);
        timing_end(c);
        return B200C_ECORRUPT;
    };

    // ---- K2: Index.db -> tokens, key prefixes, positions of the partitions the slices `sl` describe (speculate from the Summary.db samples,
    //      prove against the sequential parse, emit), order check, and the partitions of every input inside (tlo, thi] ---------------------
    uint64_t total_parts = 0;
    std::vector<uint64_t> pcount(K, 0), pbase(K + 1, 0);
    int64_t* d_tok = nullptr; uint64_t *d_kp = nullptr, *d_upos = nullptr, *d_pbase = nullptr, *d_pcount = nullptr, *d_range = nullptr; uint16_t* d_klen = nullptr;
    B200C_TRY(ws_typed(c, WS_PBASE, (size_t)2 * K + 2, &d_pbase)); d_pcount = d_pbase + K + 1;
    B200C_TRY(ws_typed(c, WS_RANGE, (size_t)2 * K + 16, &d_range));
    unsigned long long* d_rbytes = (unsigned long long*)(d_stats + 1) + 1;      // (zeroed with the stats block; every K2 run adds its range)
    res->index_slow_path_inputs = 0;
    uint64_t slow_inputs = 0;
    auto k2_run = [&](const std::vector<IdxSlice>& sl, const std::vector<uint64_t>& sb, int64_t tlo, int64_t thi) -> int {
        c->prog_stage.store(2);
        uint64_t bo2 = 0;
        for (int i = 0; i < K; i++) {
            const uint64_t ilen_i = sl[i].hi - sl[i].lo;
            bbase[i] = bo2; bo2 += (ilen_i + IB - 1) / IB;
            hin[i].ibase = ibase[i] + (sl[i].lo - isl[i].lo); hin[i].ilen = ilen_i; hin[i].uend = sl[i].uend;
        }
        bbase[K] = bo2;
        const uint64_t nblocks = bo2;
        B200C_CUDA_TRY(c, cudaMemcpyAsync((void*)hp.in, hin.data(), sizeof(InDesc) * (size_t)K, cudaMemcpyHostToDevice, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_bbase, bbase.data(), (K + 1) * 8, cudaMemcpyHostToDevice, st));
        auto alloc_arrays = [&]() -> int {
            B200C_TRY(check_cancel());
            if (total_parts - K >= (1ull << 40)) { c->err = "too many partitions"; return B200C_EUNSUPPORTED; }
            B200C_TRY(ws_typed(c, WS_TOK, total_parts + 1, &d_tok));
            B200C_TRY(ws_typed(c, WS_KP, total_parts + 1, &d_kp));
            B200C_TRY(ws_typed(c, WS_KLEN, total_parts + 1, &d_klen));
            B200C_TRY(ws_typed(c, WS_UPOS, total_parts + 1, &d_upos));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(d_pbase, pbase.data(), (K + 1) * 8, cudaMemcpyHostToDevice, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(d_pcount, pcount.data(), K * 8, cudaMemcpyHostToDevice, st));
            return B200C_OK;
        };
        // ---- B200C_K2_INTERVALS=1 (A/B, measured slower: 11.8 vs 7.7 ms at 16 x 256 MiB — a thread's 2 KB serial walk, twice, against the
        //      256-byte blocks of the default path): one thread per Summary interval, count + prove, scan, emit -----------------------------
        bool emitted = false;
        const bool k2_intervals = getenv("B200C_K2_INTERVALS") != nullptr;
        bool intervals_ok = have_summaries && k2_intervals;
        for (int i = 0; i < K && intervals_ok; i++)      // (sparse samples: an interval is one thread's serial walk — leave those to the block-parallel path)
            if (sl[i].hi > sl[i].lo && (!sl[i].s_count || (sl[i].hi - sl[i].lo) / sl[i].s_count > (64u << 10))) intervals_ok = false;
        if (intervals_ok) {
            std::vector<uint64_t> abase(K + 1, 0);
            for (int i = 0; i < K; i++) abase[i + 1] = abase[i] + sl[i].s_count;
            const uint64_t na = abase[K];
            uint32_t *d_acnt, *d_abad; uint64_t* d_ascan;
            B200C_TRY(ws_typed(c, WS_ICNT, na + 1, &d_acnt));
            B200C_TRY(ws_typed(c, WS_ISCAN, na + 2, &d_ascan));
            B200C_TRY(ws_typed(c, WS_IBAD, (size_t)K + 1, &d_abad));
            B200C_CUDA_TRY(c, cudaMemsetAsync(d_abad, 0, (K + 1) * 4, st));
            for (int i = 0; i < K; i++) if (sl[i].s_count)
                B200C_LAUNCH(c, k_index_count_intervals, (unsigned)((sl[i].s_count + 127) / 128), 128, 0, dP, IDX, i, d_summ + sb[i], sl[i].s_count, sl[i].lo, d_acnt + abase[i], d_abad);
            if (na) B200C_TRY(exclusive_scan<uint32_t>(c, d_acnt, na, d_ascan, WS_SCANA, 0)); else B200C_CUDA_TRY(c, cudaMemsetAsync(d_ascan, 0, 16, st));
            for (int i = 0; i <= K; i++) B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 8 + i, d_ascan + abase[i], 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_cerr, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 300, d_abad, (K + 1) * 4, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            if (h[0] != ~0ull) return chunk_error(h[0]);
            bool any_bad = false;
            for (int i = 0; i < K; i++) if (((uint32_t*)(h + 300))[i]) any_bad = true;
            if (!any_bad) {
                total_parts = 0;
                for (int i = 0; i < K; i++) { pcount[i] = h[8 + i + 1] - h[8 + i]; pbase[i] = total_parts; total_parts += pcount[i] + 1; }
                pbase[K] = total_parts;
                B200C_TRY(alloc_arrays());
                for (int i = 0; i < K; i++) if (sl[i].s_count)
                    B200C_LAUNCH(c, k_index_emit_intervals, (unsigned)((sl[i].s_count + 127) / 128), 128, 0, dP, IDX, i, d_summ + sb[i], sl[i].s_count, sl[i].lo, d_ascan + abase[i], pbase[i],
                                 d_tok, d_kp, d_klen, d_upos);
                emitted = true;
            }
        }
        if (!emitted) {
        uint64_t *d_istart, *d_iend, *d_iscan; uint32_t *d_icnt, *d_ihit, *d_ibad;
        B200C_TRY(ws_typed(c, WS_ISTART, nblocks + 1, &d_istart));
        B200C_TRY(ws_typed(c, WS_IEND, nblocks + 1, &d_iend));
        B200C_TRY(ws_typed(c, WS_ICNT, nblocks + 1, &d_icnt));
        B200C_TRY(ws_typed(c, WS_IHIT, nblocks + 1, &d_ihit));
        B200C_TRY(ws_typed(c, WS_IBAD, (size_t)K + 1, &d_ibad));
        B200C_TRY(ws_typed(c, WS_ISCAN, nblocks + 2, &d_iscan));
        if (nblocks) B200C_CUDA_TRY(c, cudaMemsetAsync(d_ihit, 0, nblocks * 4, st));
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_ibad, 0, (K + 1) * 4, st));
        for (int i = 0; i < K; i++) {
            const uint64_t nb = bbase[i + 1] - bbase[i];
            if (!nb) continue;
            unsigned g = (unsigned)((nb + 255) / 256);
            if (have_summaries) {
                B200C_CUDA_TRY(c, cudaMemsetAsync(d_istart + bbase[i], 0xFF, nb * 8, st));
                const uint64_t ns = sl[i].s_count;
                B200C_LAUNCH(c, k_index_find_anchors, (unsigned)((ns + 127) / 128), 128, 0, dP, IDX, d_bbase, i, d_summ + sb[i], ns, sl[i].lo, (unsigned long long*)d_istart);
            } else B200C_LAUNCH(c, k_index_find, g, 256, 0, dP, IDX, d_bbase, bbase[i], bbase[i + 1], d_istart);
            B200C_LAUNCH(c, k_index_chain, g, 256, 0, dP, IDX, d_bbase, bbase[i], bbase[i + 1], d_istart, d_icnt, d_iend);
            B200C_LAUNCH(c, k_index_verify_a, g, 256, 0, dP, d_bbase, bbase[i], bbase[i + 1], d_istart, d_iend, d_ihit, d_ibad);
            B200C_LAUNCH(c, k_index_verify_b, g, 256, 0, dP, d_bbase, bbase[i], bbase[i + 1], d_istart, d_ihit, d_ibad);
        }
        if (nblocks) {
            B200C_LAUNCH(c, k_index_seq, (K + 63) / 64, 64, 0, dP, IDX, d_bbase, d_istart, d_icnt, d_ibad, d_err);
            B200C_TRY(exclusive_scan<uint32_t>(c, d_icnt, nblocks, d_iscan, WS_SCANA, 0));
        } else B200C_CUDA_TRY(c, cudaMemsetAsync(d_iscan, 0, 16, st));
        // read back: chunk errors, index errors, per-input partition counts
        for (int i = 0; i <= K; i++) B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 8 + i, d_iscan + bbase[i], 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_cerr, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 1, d_err, 8, cudaMemcpyDeviceToHost, st));
        if (nblocks) B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 300, d_ibad, (K + 1) * 4, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        if (nblocks) for (int i = 0; i < K && i < 64; i++) if (((uint32_t*)(h + 300))[i]) slow_inputs |= 1ull << i;
        res->index_slow_path_inputs = __builtin_popcountll(slow_inputs);
        if (h[0] != ~0ull) return chunk_error(h[0]);
        if (h[1] != ~0ull) {
            res->corruption.input = (int)((h[1] >> 48) & 0xFF); res->corruption.kind = (int)(h[1] >> 56); res->corruption.chunk = 0; res->corruption.offset = h[1] & 0xFFFFFFFFFFFFull;
            c->err = "malformed Index.db in input " + std::to_string(res->corruption.input);
            timing_end(c);
            return B200C_ECORRUPT;
        }
        total_parts = 0;
        for (int i = 0; i < K; i++) { pcount[i] = h[8 + i + 1] - h[8 + i]; pbase[i] = total_parts; total_parts += pcount[i] + 1; }
        pbase[K] = total_parts;
        B200C_TRY(alloc_arrays());
        if (nblocks) B200C_LAUNCH(c, k_index_emit, (unsigned)((nblocks + 255) / 256), 256, 0, dP, IDX, d_bbase, nblocks, d_istart, d_icnt, d_iscan, d_pbase,
                                  d_tok, d_kp, d_klen, d_upos, d_err);
        }      // (legacy path)
        if (total_parts > (uint64_t)K) B200C_LAUNCH(c, k_check_order, 1184, 256, 0, dP, d_pbase, d_pcount, d_tok, d_kp, d_klen, d_upos, d_err);
        B200C_LAUNCH(c, k_input_ranges, (K + 63) / 64, 64, 0, dP, d_pbase, d_pcount, d_tok, d_upos, tlo, thi, d_range, d_rbytes);
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_range, 2 * K * 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 200, d_err, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        if (h[200] != ~0ull) return index_data_mismatch(h[200]);
        for (int i = 0; i < K; i++) if (h[2 * i] > h[2 * i + 1] || h[2 * i + 1] > pcount[i]) return index_data_mismatch((uint64_t)i << 48);
        // a slice that does not start with the call's own slice starts at a sample at or below tlo: its first entry is not in range. One that
        // is — the Summary.db positions lied about the tokens — could hide partitions of this range in the previous slice: refuse it.
        for (int i = 0; i < K; i++) if (pcount[i] && sl[i].lo != isl[i].lo && h[2 * i] == 0) {
            c->err = "Summary.db positions of input " + std::to_string(i) + " do not bracket the token range"; res->corruption.input = i; res->corruption.kind = 3; res->corruption.chunk = 0; res->corruption.offset = sl[i].lo;
            timing_end(c); return B200C_ECORRUPT; }
        return B200C_OK;
    };
    mark(1);
    if (!istream) B200C_TRY(k2_run(isl, psb[0], m->token_lo, m->token_hi));

    // ---- token ranges: T[0] < T[1] < ... < T[nr]; piece r merges the partitions with token in (T[r], T[r+1]]. Several pieces: planned on the
    //      host above (Index.db streaming). One piece of a token sub-range over device-resident inputs: the chunks it crosses come from here.
    if (deferred && !istream) {
        int64_t* d_T; uint64_t* d_plan;
        B200C_TRY(ws_typed(c, WS_PLAN, (size_t)nr + 2 + 2 * (size_t)nr * K, &d_T)); d_plan = (uint64_t*)(d_T + nr + 2);
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_T, T.data(), (nr + 1) * 8, cudaMemcpyHostToDevice, st));
        B200C_LAUNCH(c, k_range_plan, (unsigned)((nr * K + 63) / 64), 64, 0, dP, d_pbase, d_pcount, d_tok, d_upos, d_T, nr, d_plan);
        uint64_t* hplan = h + 2048;
        B200C_CUDA_TRY(c, cudaMemcpyAsync(hplan, d_plan, 2 * (size_t)nr * K * 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        for (int r = 0; r < nr; r++) {
            uint64_t tot = 0;
            for (int i = 0; i < K; i++) {
                const b200c_input& in = m->inputs[i];
                uint64_t a = hplan[2 * ((size_t)r * K + i)], b = hplan[2 * ((size_t)r * K + i) + 1];
                if (a < ubase[i] || b < a || b > ubase[i] + in.data_length) return index_data_mismatch(((uint64_t)i << 48));
                a -= ubase[i]; b -= ubase[i]; tot += b - a;
                need_of(r, i, a, b);
            }
            range_bytes[r] = tot;
        }
        // all copies are queued now, piece after piece; EV_RANGE + r fires when piece r is on the device
        for (int r = 0; r < nr; r++) {
            for (int i = 0; i < K; i++) B200C_TRY(copy_chunks(i, need[(size_t)r * K + i].h2d_a, need[(size_t)r * K + i].h2d_b));
            B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_RANGE + r], cs));
        }
    }

    // ---- per-piece state -------------------------------------------------------------------------------------------------------------
    const bool to_host_stream = !dev && !lcs;          // one output file in host memory: K5 pieces leave through an OutStream
    static const bool two_pass = getenv("B200C_K4_TWO_PASS") != nullptr;     // A/B switch: size pass + full emit pass instead of scratch + gather
    b200c_output& out0 = res->outputs[0];
    OutStream os;
    // B200C_K5_OVERLAP=1 (A/B, measured: no gain — 489.0 vs 490.6 ms per configs[1] step; K4 and K5 are both bound by shared memory and latency, the
    // time K5 spends under the next piece's K1..K3 comes back as slower K2..K4): K5 of piece r on its own stream instead of the main one
    const bool k5_async = to_host_stream && nr > 1 && []() { const char* e = getenv("B200C_K5_OVERLAP"); return e ? atoi(e) != 0 : false; }();
    int k5_last = -1;
    if (to_host_stream) B200C_TRY(out_stream_begin(os, c, m->out_compressor, m->out_chunk_len, m->out_max_compressed_len, out0.data, out0.data_cap, WS_CODEC));
    const uint64_t L = (uint64_t)m->out_chunk_len;
    uint64_t ubase_total = 0, ilen_total = 0, ncontrib_total = 0, nparts_total = 0;
    uint64_t tail_len = 0; const uint8_t* tail_ptr = nullptr;       // bytes of the merged stream not yet handed to K5 (< one chunk)
    bool index_fits = true;
    // arrays that outlive the loop when there is a single piece (the LCS writer below works on them)
    uint64_t nparts = 0, ulen_out = 0, ilen_out = 0;
    uint64_t *d_dsize = nullptr, *d_dpos = nullptr, *d_ipos = nullptr, *d_contrib = nullptr, *d_opfirst = nullptr, *d_ioff = nullptr; uint32_t *d_ipay = nullptr, *d_nblk = nullptr, *d_ihead = nullptr, *d_isize = nullptr, *d_icap = nullptr;
    uint32_t *d_stmunf = nullptr, *d_strows = nullptr; uint8_t* d_ovf = nullptr;
    uint8_t *UOUT = nullptr, *IOUT = nullptr, *ISCR = nullptr;
    K4Args ka; memset(&ka, 0, sizeof(ka));
    std::function<int(int)> launch_k4;
    std::function<int(uint64_t, uint64_t)> launch_k4_stats;
    uint32_t* d_ccount = nullptr; uint32_t* d_wflag = nullptr; uint64_t* d_wrank = nullptr;     // side band: cells per partition, written flags / ranks

    for (int r = 0; r < nr; r++) {
        B200C_TRY(check_cancel());
        // ---- K2 of this piece (Index.db streaming), then its K1 (deferred mode) --------------------------------------------------------
        if (istream) {
            mark(1);
            B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_pool[EV_RANGE + r], 0));
            B200C_TRY(k2_run(psl[r], psb[r], T[r], T[r + 1]));
        }
        mark(0);
        c->prog_stage.store(1);
        if (deferred) {
            B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_pool[EV_RANGE + r], 0));
            std::vector<uint64_t> a(K), b(K);
            for (int i = 0; i < K; i++) { a[i] = need[(size_t)r * K + i].k1_a; b[i] = need[(size_t)r * K + i].k1_b; }
            B200C_TRY(k1_many(a, b));
        }
        // ---- K3: partition merge -------------------------------------------------------------------------------------------------------
        mark(2);
        c->prog_stage.store(3);
        B200C_LAUNCH(c, k_input_ranges, (K + 63) / 64, 64, 0, dP, d_pbase, d_pcount, d_tok, d_upos, T[r], T[r + 1], d_range, (unsigned long long*)nullptr);
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_range, 2 * K * 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 200, d_cerr, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        if (h[200] != ~0ull) return chunk_error(h[200]);
        uint64_t ncontrib = 0;
        for (int i = 0; i < K; i++) ncontrib += h[2 * i + 1] - h[2 * i];
        ncontrib_total += ncontrib;
        const uint64_t nbuckets = std::max<uint64_t>(1, ncontrib / 256);
        uint64_t *d_bstart, *d_opidx; uint32_t* d_head; MergeGeom* d_geom;
        B200C_TRY(ws_typed(c, WS_BSTART, (nbuckets + 1) * K + 8, &d_bstart)); d_geom = (MergeGeom*)(d_range + 2 * K + 2);
        B200C_TRY(ws_typed(c, WS_CONTRIB, ncontrib + 1, &d_contrib));
        B200C_TRY(ws_typed(c, WS_HEAD, ncontrib + 1, &d_head));
        B200C_TRY(ws_typed(c, WS_OPIDX, ncontrib + 2, &d_opidx));
        nparts = 0;
        if (ncontrib) {
            B200C_LAUNCH(c, k_merge_geom, 1, 1, 0, dP, d_pbase, d_range, d_tok, nbuckets, d_geom);
            B200C_LAUNCH(c, k_bucket_bounds, (unsigned)(((nbuckets + 1) * K + 255) / 256), 256, 0, dP, d_pbase, d_range, d_tok, d_geom, d_bstart);
            B200C_LAUNCH(c, k_merge_buckets, (unsigned)((nbuckets + 3) / 4), 128, 0, dP, d_pbase, d_range, d_tok, d_kp, d_klen, d_upos, d_bstart, nbuckets, d_contrib, d_head, d_hist);
            B200C_TRY(exclusive_scan<uint32_t>(c, d_head, ncontrib, d_opidx, WS_SCANA, 0));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_opidx + ncontrib, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            nparts = h[0];
        }
        if (nparts >= (1ull << 32)) { c->err = "too many output partitions"; return B200C_EUNSUPPORTED; }
        nparts_total += nparts;
        B200C_TRY(ws_typed(c, WS_OPFIRST, nparts + 2, &d_opfirst));
        uint32_t* d_list; unsigned long long* d_cursor = nullptr; uint64_t *d_bound = nullptr, *d_bpos = nullptr;
        uint32_t* d_insz = nullptr; uint8_t* d_big = nullptr;
        B200C_TRY(ws_typed(c, WS_LIST, nparts + 1, &d_list));
        B200C_TRY(ws_typed(c, WS_BOUND, nparts + 1, &d_bound));
        B200C_TRY(ws_typed(c, WS_BPOS, nparts + 2, &d_bpos));
        B200C_TRY(ws_typed(c, WS_ICAP, nparts + 1, &d_icap));
        B200C_TRY(ws_typed(c, WS_IOFF, nparts + 2, &d_ioff));
        uint64_t n_le8 = 0, n_le12 = 0, n_le16 = 0, n_le32 = 0;
        if (ncontrib) {
            B200C_LAUNCH(c, k_op_first, (unsigned)((ncontrib + 1 + 255) / 256), 256, 0, d_head, d_opidx, ncontrib, d_opfirst);
            // counting sort of the output partitions by (fan-in, size bucket)
            B200C_TRY(ws_typed(c, WS_INSZ, nparts + 1, &d_insz));
            B200C_TRY(ws_typed(c, WS_BIG, nparts + 2, &d_big));
            B200C_LAUNCH(c, k_bounds, (unsigned)((nparts + 255) / 256), 256, 0, d_contrib, d_opfirst, nparts, d_upos, d_pbase, d_bound,
                         (uint32_t)std::min<uint64_t>(std::max<int64_t>(1, m->column_index_size), 0x7fffffff), d_icap, d_insz, d_big);
            // tile = token-contiguous run of output partitions whose inputs total ~32 MiB
            uint64_t per_part = std::max<uint64_t>(1, range_bytes[r] / std::max<uint64_t>(1, nparts));
            uint32_t tile_shift = 12; while (tile_shift < 24 && ((1ull << (tile_shift + 1)) * per_part) <= (32ull << 20)) tile_shift++;
            const uint64_t ntiles = (nparts >> tile_shift) + 1, nkeys = 5 * ntiles * SORT_BINS;
            const uint64_t wide_bound = []() -> uint64_t { const char* e = getenv("B200C_K4_WIDE_WARP"); return e ? strtoull(e, nullptr, 10) : 0; }() ?: ~0ull;    // bytes; unset / 0 = off (A/B)
            B200C_TRY(ws_typed(c, WS_CURSOR, nkeys + 2, &d_cursor));
            B200C_CUDA_TRY(c, cudaMemsetAsync(d_cursor, 0, (nkeys + 2) * 8, st));
            B200C_LAUNCH(c, k_class_hist, 1184, 256, 0, d_opfirst, d_bound, nparts, tile_shift, ntiles, wide_bound, d_cursor);
            B200C_TRY(exclusive_scan<uint64_t>(c, (const uint64_t*)d_cursor, nkeys, (uint64_t*)d_cursor, WS_SCANA, 0));
            for (int k = 1; k <= 4; k++) B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 512 + k, (uint64_t*)d_cursor + (uint64_t)k * ntiles * SORT_BINS, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            n_le8 = h[513]; n_le12 = h[514]; n_le16 = h[515]; n_le32 = h[516];
            B200C_LAUNCH(c, k_fanin_scatter, (unsigned)((nparts + 255) / 256), 256, 0, d_opfirst, d_bound, nparts, tile_shift, ntiles, wide_bound, d_cursor, d_list);
        }
        B200C_TRY(check_cancel());

        // ---- K4: row merge + serialise ---------------------------------------------------------------------------------------------------
        mark(3);
        c->prog_stage.store(4);
        B200C_TRY(ws_typed(c, WS_DSIZE, nparts + 1, &d_dsize));
        B200C_TRY(ws_typed(c, WS_DPOS, nparts + 2, &d_dpos));
        B200C_TRY(ws_typed(c, WS_IPOS, nparts + 2, &d_ipos));
        B200C_TRY(ws_typed(c, WS_IPAY, nparts + 1, &d_ipay));
        B200C_TRY(ws_typed(c, WS_NBLK, nparts + 1, &d_nblk));
        B200C_TRY(ws_typed(c, WS_IHEAD, nparts + 1, &d_ihead));
        B200C_TRY(ws_typed(c, WS_ISIZE, nparts + 1, &d_isize));
        B200C_TRY(ws_typed(c, WS_STMUNF, nparts + 1, &d_stmunf));
        B200C_TRY(ws_typed(c, WS_STROWS, nparts + 1, &d_strows));
        B200C_TRY(ws_typed(c, WS_OVF, nparts + 1, &d_ovf));
        const size_t cols_s = hp.mcols <= K4_SMEM_COLS ? (size_t)hp.mcols * sizeof(MCell) : 0;
        const size_t smem8 = (size_t)128 * (8 * SLOT_BYTES + cols_s + 8), smem12 = (size_t)64 * (12 * SLOT_BYTES + cols_s + 8), smem16 = (size_t)64 * (16 * SLOT_BYTES + cols_s + 8), smem64 = (size_t)32 * (64 * SLOT_BYTES + cols_s + 8), cell_smem32 = (size_t)4 * hp.mcols * sizeof(MCell);
        memset(&ka, 0, sizeof(ka));
        ka.P = dP; ka.contrib = d_contrib; ka.op_first = d_opfirst; ka.list = d_list; ka.upos = d_upos; ka.pbase = d_pbase; ka.kp = d_kp; ka.klen = d_klen; ka.tok = d_tok;
        ka.dsize = d_dsize; ka.ipay = d_ipay; ka.nblk = d_nblk; ka.ihead = d_ihead; ka.st_munf = d_stmunf; ka.st_rows = d_strows; ka.ovf = d_ovf;
        ka.dpos = d_dpos; ka.ipos = d_ipos; ka.err = d_err; ka.jlo = 0; ka.jhi = nparts; ka.m3_nblk = two_pass ? 1 : 0;
        if (want_meta) {
            B200C_TRY(ws_typed(c, WS_CCOUNT, nparts + 1, &d_ccount));
            B200C_TRY(ws_typed(c, WS_META_FLAG, nparts + 1, &d_wflag));
            B200C_TRY(ws_typed(c, WS_META_WRANK, nparts + 2, &d_wrank));
            if (!lcs) { ka.sg = d_sg; ka.td = d_td; ka.ccount = d_ccount; }      // multi-file: per file, by k_partition_stats (launch_k4_stats)
        }
        // one launch per fan-in class over its slice of the sorted list
        const uint64_t np_ = nparts;
        launch_k4 = [&, n_le8, n_le12, n_le16, n_le32, np_, smem8, smem12, smem16, smem64, cell_smem32](int mode) -> int {
            ka.mode = mode;
            const bool emit = mode != 0;
            if (hp.ncx || hp.ctr_mask || hp.sctr_mask) {
                // tables with multi-cell (complex) or counter columns: the CX instantiations of the thread kernels, for every fan-in (64 cursors per thread above 16);
                // single serialisation pass only (the size-pass A/B mode is refused above)
                if (!emit) { c->err = "B200C_K4_TWO_PASS with multi-cell columns"; return B200C_EUNSUPPORTED; }
                if (n_le8) B200C_LAUNCH(c, (k_partition_thr<8, 128, true, true>), (unsigned)((n_le8 + 127) / 128), 128, smem8, ka, 0ull, n_le8);
                if (n_le12 > n_le8) B200C_LAUNCH(c, (k_partition_thr<12, 64, true, true>), (unsigned)((n_le12 - n_le8 + 63) / 64), 64, smem12, ka, n_le8, n_le12);
                if (n_le16 > n_le12) B200C_LAUNCH(c, (k_partition_thr<16, 64, true, true>), (unsigned)((n_le16 - n_le12 + 63) / 64), 64, smem16, ka, n_le12, n_le16);
                if (np_ > n_le16) B200C_LAUNCH(c, (k_partition_thr<64, 32, true, true>), (unsigned)((np_ - n_le16 + 31) / 32), 32, smem64, ka, n_le16, np_);
                return B200C_OK;
            }
            if (n_le8) {
                unsigned g = (unsigned)((n_le8 + 127) / 128);
                if (emit) B200C_LAUNCH(c, (k_partition_thr<8, 128, true>), g, 128, smem8, ka, 0ull, n_le8);
                else B200C_LAUNCH(c, (k_partition_thr<8, 128, false>), g, 128, smem8, ka, 0ull, n_le8);
            }
            if (n_le12 > n_le8) {
                unsigned g = (unsigned)((n_le12 - n_le8 + 63) / 64);
                if (emit) B200C_LAUNCH(c, (k_partition_thr<12, 64, true>), g, 64, smem12, ka, n_le8, n_le12);
                else B200C_LAUNCH(c, (k_partition_thr<12, 64, false>), g, 64, smem12, ka, n_le8, n_le12);
            }
            if (n_le16 > n_le12) {
                unsigned g = (unsigned)((n_le16 - n_le12 + 63) / 64);
                if (emit) B200C_LAUNCH(c, (k_partition_thr<16, 64, true>), g, 64, smem16, ka, n_le12, n_le16);
                else B200C_LAUNCH(c, (k_partition_thr<16, 64, false>), g, 64, smem16, ka, n_le12, n_le16);
            }
            if (n_le32 > n_le16) {
                unsigned g = (unsigned)((n_le32 - n_le16 + 3) / 4);
                if (emit) B200C_LAUNCH(c, (k_partition_warp<1, true>), g, 128, cell_smem32, ka, n_le16, n_le32);
                else B200C_LAUNCH(c, (k_partition_warp<1, false>), g, 128, cell_smem32, ka, n_le16, n_le32);
            }
            if (np_ > n_le32) {
                unsigned g = (unsigned)((np_ - n_le32 + 3) / 4);
                if (emit) B200C_LAUNCH(c, (k_partition_warp<2, true>), g, 128, cell_smem32, ka, n_le32, np_);
                else B200C_LAUNCH(c, (k_partition_warp<2, false>), g, 128, cell_smem32, ka, n_le32, np_);
            }
            return B200C_OK;
        };
        // statistics of the output file holding partitions [jlo, jhi) into d_sg / d_td (multi-file output with the side band)
        launch_k4_stats = [&, n_le8, n_le12, n_le16, np_, smem8, smem12, smem16, smem64](uint64_t jlo, uint64_t jhi) -> int {
            K4Args sa = ka; sa.sg = d_sg; sa.td = d_td; sa.ccount = d_ccount; sa.jlo = jlo; sa.jhi = jhi;
            if (hp.ncx || hp.ctr_mask || hp.sctr_mask) {
                if (n_le8) B200C_LAUNCH(c, (k_partition_stats<8, 128, true>), (unsigned)((n_le8 + 127) / 128), 128, smem8, sa, 0ull, n_le8);
                if (n_le12 > n_le8) B200C_LAUNCH(c, (k_partition_stats<12, 64, true>), (unsigned)((n_le12 - n_le8 + 63) / 64), 64, smem12, sa, n_le8, n_le12);
                if (n_le16 > n_le12) B200C_LAUNCH(c, (k_partition_stats<16, 64, true>), (unsigned)((n_le16 - n_le12 + 63) / 64), 64, smem16, sa, n_le12, n_le16);
                if (np_ > n_le16) B200C_LAUNCH(c, (k_partition_stats<64, 32, true>), (unsigned)((np_ - n_le16 + 31) / 32), 32, smem64, sa, n_le16, np_);
            } else {
                if (n_le8) B200C_LAUNCH(c, (k_partition_stats<8, 128, false>), (unsigned)((n_le8 + 127) / 128), 128, smem8, sa, 0ull, n_le8);
                if (n_le12 > n_le8) B200C_LAUNCH(c, (k_partition_stats<12, 64, false>), (unsigned)((n_le12 - n_le8 + 63) / 64), 64, smem12, sa, n_le8, n_le12);
                if (n_le16 > n_le12) B200C_LAUNCH(c, (k_partition_stats<16, 64, false>), (unsigned)((n_le16 - n_le12 + 63) / 64), 64, smem16, sa, n_le12, n_le16);
                if (np_ > n_le16) B200C_LAUNCH(c, (k_partition_stats<64, 32, false>), (unsigned)((np_ - n_le16 + 31) / 32), 32, smem64, sa, n_le16, np_);
            }
            return B200C_OK;
        };
        if (want_meta && lcs && c->k4st_attr_set != (int)(smem8 + 1)) {
            cudaFuncSetAttribute(k_partition_stats<8, 128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8);
            cudaFuncSetAttribute(k_partition_stats<12, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem12);
            cudaFuncSetAttribute(k_partition_stats<16, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16);
            cudaFuncSetAttribute(k_partition_stats<64, 32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem64);
            cudaFuncSetAttribute(k_partition_stats<8, 128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8);
            cudaFuncSetAttribute(k_partition_stats<12, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem12);
            cudaFuncSetAttribute(k_partition_stats<16, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16);
            cudaFuncSetAttribute(k_partition_stats<64, 32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem64);
            c->k4st_attr_set = (int)(smem8 + 1);
        }
        if (c->k4_attr_set != (int)(smem8 + 1)) {      // > 48 KiB of dynamic shared memory needs an explicit opt-in, once per context/device
            cudaFuncSetAttribute(k_partition_thr<8, 128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8);
            cudaFuncSetAttribute(k_partition_thr<8, 128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8);
            cudaFuncSetAttribute(k_partition_thr<12, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem12);
            cudaFuncSetAttribute(k_partition_thr<12, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem12);
            cudaFuncSetAttribute(k_partition_thr<16, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16);
            cudaFuncSetAttribute(k_partition_thr<16, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16);
            cudaFuncSetAttribute(k_partition_thr<8, 128, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8);
            cudaFuncSetAttribute(k_partition_thr<12, 64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem12);
            cudaFuncSetAttribute(k_partition_thr<16, 64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16);
            cudaFuncSetAttribute(k_partition_thr<64, 32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem64);
            // B200C_K4_CARVEOUT=percent of the SM's unified L1/shared memory left to shared memory (A/B: fewer resident blocks, more L1 for the
            // scattered reads of Data.db); unset: the driver sizes the carve-out for the most blocks that fit
            if (const char* e = getenv("B200C_K4_CARVEOUT")) { const int pct = atoi(e);
                cudaFuncSetAttribute(k_partition_thr<8, 128, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
                cudaFuncSetAttribute(k_partition_thr<12, 64, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
                cudaFuncSetAttribute(k_partition_thr<16, 64, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct); }
            c->k4_attr_set = (int)(smem8 + 1);
        }
        uint8_t* SCRATCH = nullptr;
        ulen_out = 0; ilen_out = 0;
        if (nparts) {
            if (two_pass) {
                B200C_CUDA_TRY(c, cudaMemsetAsync(d_ovf, 0, nparts, st));
                B200C_TRY(launch_k4(0));
            } else {
                B200C_TRY(exclusive_scan<uint64_t>(c, d_bound, nparts, d_bpos, WS_SCANA, 0));
                B200C_TRY(exclusive_scan<uint32_t>(c, d_icap, nparts, d_ioff, WS_SCANA + 3, 0));
                B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_bpos + nparts, 8, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 1, d_ioff + nparts, 8, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                B200C_TRY(ws_typed(c, WS_SCRATCH, h[0] + 64, &SCRATCH));
                B200C_TRY(ws_typed(c, WS_ISCR, h[1] + 64, &ISCR));
                ka.doff = d_bpos; ka.dcapv = d_bound; ka.dbase = SCRATCH; ka.iout = nullptr; ka.ioff = d_ioff; ka.icapv = d_icap; ka.iscr = ISCR;
                const bool staged = !hp.ncx && !hp.ctr_mask && !hp.sctr_mask && []() { const char* e = getenv("B200C_K4_STAGED"); return e ? atoi(e) != 0 : (B200C_K4_STAGED_DEFAULT != 0); }();      // A/B switch (read per call; tables with multi-cell columns: thread kernels)
                if (staged) {
                    // tile plan: exclusive scan of the input bytes, cut marks, scan of the marks, tile starts
                    uint64_t *d_inpos, *d_tscan; uint32_t *d_mark, *d_tstart; unsigned long long* d_nbig = (unsigned long long*)(d_stats + 1);
                    B200C_TRY(ws_typed(c, WS_INPOS, nparts + 2, &d_inpos));
                    B200C_TRY(ws_typed(c, WS_TMARK, nparts + 2, &d_mark));
                    B200C_TRY(ws_typed(c, WS_TSCAN, nparts + 2, &d_tscan));
                    B200C_TRY(ws_typed(c, WS_TSTART, nparts + 2, &d_tstart));
                    B200C_TRY(exclusive_scan<uint32_t>(c, d_insz, nparts, d_inpos, WS_SCANA, 0));
                    B200C_CUDA_TRY(c, cudaMemsetAsync(d_nbig, 0, 8, st));
                    B200C_LAUNCH(c, k_tile_marks, (unsigned)((nparts + 255) / 256), 256, 0, nparts, d_inpos, d_opfirst, d_big, d_mark, d_nbig);
                    B200C_TRY(exclusive_scan<uint32_t>(c, d_mark, nparts, d_tscan, WS_SCANA, 0));
                    B200C_LAUNCH(c, k_tile_starts, (unsigned)((nparts + 1 + 255) / 256), 256, 0, nparts, d_mark, d_tscan, d_tstart);
                    B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_tscan + nparts, 8, cudaMemcpyDeviceToHost, st));
                    B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 1, d_nbig, 8, cudaMemcpyDeviceToHost, st));
                    B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                    const uint64_t ntiles = h[0], nbig = h[1];
                    const bool wide = m->ncolumns > K4_SMEM_COLS;
                    const size_t smem_st = (size_t)ST_HEAD + ST_STAGE_CAP + (size_t)ST_CUR_CAP * sizeof(CurS) + (wide ? 0 : (size_t)ST_THREADS * hp.mcols * sizeof(MCell)) + 16;
                    if (c->k4s_attr_set != (int)smem_st) {
                        cudaFuncSetAttribute(k_partition_staged<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_st);
                        cudaFuncSetAttribute(k_partition_staged<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_st);
                        c->k4s_attr_set = (int)smem_st;
                    }
                    ka.mode = 1; ka.only_big = nullptr;
                    if (wide) B200C_LAUNCH(c, k_partition_staged<true>, (unsigned)ntiles, ST_THREADS, smem_st, ka, d_tstart, d_big);
                    else B200C_LAUNCH(c, k_partition_staged<false>, (unsigned)ntiles, ST_THREADS, smem_st, ka, d_tstart, d_big);
                    if (nbig) { ka.only_big = d_big; B200C_TRY(launch_k4(1)); ka.only_big = nullptr; }
                } else B200C_TRY(launch_k4(1));
            }
            B200C_LAUNCH(c, k_sum_stats, 1184, 256, 0, nparts, d_dsize, d_stmunf, d_strows, d_stats);
            B200C_TRY(exclusive_scan<uint64_t>(c, d_dsize, nparts, d_dpos, WS_SCANA, 0));
            if (ubase_total) B200C_LAUNCH(c, k_add_u64, (unsigned)((nparts + 1 + 255) / 256), 256, 0, d_dpos, nparts + 1, ubase_total);     // positions in the file, not in the piece
            B200C_LAUNCH(c, k_index_sizes, (unsigned)((nparts + 255) / 256), 256, 0, nparts, d_dsize, d_dpos, d_ipay, d_ihead, d_isize);
            B200C_TRY(exclusive_scan<uint32_t>(c, d_isize, nparts, d_ipos, WS_SCANA + 3, 0));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_dpos + nparts, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 1, d_ipos + nparts, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 2, d_err, 8, cudaMemcpyDeviceToHost, st));
            if (want_meta && !lcs) {                   // (multi-file: per file, in the writer loop below)
                B200C_LAUNCH(c, k_written_flags, (unsigned)((nparts + 255) / 256), 256, 0, nparts, d_dsize, d_wflag);
                B200C_TRY(exclusive_scan<uint32_t>(c, d_wflag, nparts, d_wrank, WS_SCANA, 0));
                B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 3, d_wrank + nparts, 8, cudaMemcpyDeviceToHost, st));
            }
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            if (h[2] != ~0ull) {
                int kinde = (int)(h[2] >> 56);
                res->corruption.input = (int)((h[2] >> 48) & 0xFF); res->corruption.kind = 4; res->corruption.chunk = 0; res->corruption.offset = h[2] & 0xFFFFFFFFFFFFull;
                timing_end(c);
                if (kinde == 9) { c->err = "unsupported feature in input " + std::to_string(res->corruption.input) + " (outside the envelope: shadowable deletion, a fan-in or layout the kernels refuse, or a counter context the reference never writes inside a merge)"; return B200C_EUNSUPPORTED; }
                c->err = "malformed Data.db in input " + std::to_string(res->corruption.input) + " near offset " + std::to_string(res->corruption.offset);
                return B200C_ECORRUPT;
            }
            ulen_out = h[0] - ubase_total; ilen_out = h[1];
        }
        B200C_TRY(check_cancel());
        mark(4);
        // the merged stream of this piece goes behind the unconsumed tail of the previous one; UOUT + tail_len is file offset ubase_total
        if (k5_async && r >= 2) B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_pool[EV_K5 + 1 + (r & 1)], 0));      // K5 of piece r - 2 has read this buffer
        B200C_TRY(ws_typed(c, (r & 1) ? WS_UOUT2 : WS_UOUT, tail_len + ulen_out + 64, &UOUT));
        if (r) B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_pool[EV_INDEX], 0));          // IOUT of the previous piece has left
        B200C_TRY(ws_typed(c, WS_IOUT, ilen_out + 64, &IOUT));
        if (tail_len) B200C_CUDA_TRY(c, cudaMemcpyAsync(UOUT, tail_ptr, tail_len, cudaMemcpyDeviceToDevice, st));
        uint8_t* const ubias = (uint8_t*)((uintptr_t)UOUT + tail_len - ubase_total);          // ubias + (file offset) = address
        if (nparts && ulen_out) {
            ka.dbase = ubias; ka.iout = IOUT; ka.doff = nullptr; ka.dcapv = nullptr;
            if (two_pass) B200C_TRY(launch_k4(2));
            else {
                B200C_LAUNCH(c, k_gather, (unsigned)((nparts + 7) / 8), 256, 0, nparts, d_dsize, d_dpos, d_bpos, d_ovf, SCRATCH, ubias);
                B200C_LAUNCH(c, k_index_simple, (unsigned)((nparts + 255) / 256), 256, 0, dP, nparts, d_contrib, d_opfirst, d_upos, d_pbase, d_dsize, d_dpos, d_nblk, d_ovf, d_ihead, d_ipos, IOUT);
                B200C_LAUNCH(c, k_index_promoted, (unsigned)((nparts + 127) / 128), 128, 0, dP, nparts, d_contrib, d_opfirst, d_upos, d_pbase, d_dsize, d_dpos, d_nblk, d_ovf, d_ihead, d_ipay, d_ipos,
                             d_ioff, d_icap, ISCR, IOUT);
                B200C_TRY(launch_k4(3));
            }
        }
        if (want_meta && !lcs && nparts && ulen_out) {
            // per key / per partition metadata of this piece: bloom bits, HLL registers, histograms, index-summary samples, first / last key
            const uint64_t nwritten = h[3];
            const uint64_t ns = (written_total + nwritten + meta_interval - 1) / meta_interval - (written_total + meta_interval - 1) / meta_interval;
            uint32_t *d_samplej, *d_esize; uint64_t* d_epos;
            B200C_TRY(ws_typed(c, WS_META_SAMPLE, ns + 1, &d_samplej));
            B200C_TRY(ws_typed(c, WS_META_ESIZE, ns + 1, &d_esize));
            B200C_TRY(ws_typed(c, WS_META_EPOS, ns + 2, &d_epos));
            MetaArgs ma; memset(&ma, 0, sizeof(ma));
            ma.P = dP; ma.contrib = d_contrib; ma.op_first = d_opfirst; ma.upos = d_upos; ma.pbase = d_pbase; ma.dsize = d_dsize; ma.ipos = d_ipos; ma.ihead = d_ihead;
            ma.ccount = d_ccount; ma.wrank = d_wrank; ma.nparts = nparts; ma.index_base = ilen_total; ma.written_base = written_total; ma.sg = d_sg;
            ma.bloom = d_bloom; ma.bloom_bits = bloom_words * 64; ma.bloom_k = m->bloom_hash_count; ma.interval = meta_interval; ma.sample_j = d_samplej;
            ma.first_key = d_mkeys; ma.last_key = d_mkeys + 65536;
            B200C_LAUNCH(c, k_meta_keys, (unsigned)((nparts + 255) / 256), 256, 0, ma);
            if (ns && o0.summary) {
                B200C_LAUNCH(c, k_summary_sizes, (unsigned)((ns + 255) / 256), 256, 0, ma, ns, d_esize);
                B200C_TRY(exclusive_scan<uint32_t>(c, d_esize, ns, d_epos, WS_SCANA, 0));
                B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 4, d_epos + ns, 8, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                B200C_TRY(ws_grow_keep<uint8_t>(c, WS_META_SUMENT, sument_bound + h[4] + 64, sument_bound, &d_sument));
                B200C_TRY(ws_grow_keep<uint64_t>(c, WS_META_SUMOFF, samples_total + ns + 2, samples_total, &d_sumoff));
                B200C_LAUNCH(c, k_summary_emit, (unsigned)((ns + 255) / 256), 256, 0, ma, ns, d_epos, d_sument, d_sumoff);
                B200C_LAUNCH(c, k_meta_advance, 1, 1, 0, d_sg, ns, d_epos);
                sument_bound += h[4]; samples_total += ns;
            }
            written_total += nwritten;
        }
        c->prog_scanned.store(bytes_read * (4 * (uint64_t)r + 3) / (4 * (uint64_t)nr));
        if (deferred || r == nr - 1) for (int i = 0; i < K; i++) c->prog_input_pos[i].store(range_end[(size_t)r * K + i]);

        // ---- K5 of this piece (one output file in host memory): whole chunks go out now, the rest waits for the next piece -------------
        mark(5);
        c->prog_stage.store(5);
        if (to_host_stream) {
            if (ilen_out) {                                  // Index.db is final after K4: read it back while K5 compresses
                if (ilen_total + ilen_out > out0.index_cap || !out0.index) index_fits = false;
                if (index_fits) {
                    B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_INDEX + 1], st));
                    B200C_CUDA_TRY(c, cudaStreamWaitEvent(c->copy_out, c->ev_pool[EV_INDEX + 1], 0));
                    B200C_CUDA_TRY(c, cudaMemcpyAsync(out0.index + ilen_total, IOUT, ilen_out, cudaMemcpyDeviceToHost, c->copy_out));
                }
            }
            B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_INDEX], c->copy_out));
            const uint64_t avail = tail_len + ulen_out;
            uint64_t take = (r == nr - 1) ? avail : avail / L * L;
            const uint64_t slice = std::max<uint64_t>(L, std::max<uint64_t>(512ull << 20, bytes_read / 32) / L * L);      // pieces of ~512 MiB keep the read-back close behind
            if (k5_async) {
                // K5 of this piece on its own stream: it needs UOUT only, so K1..K3 of the next piece — and the host->device copies they wait for —
                // run on top of it; K4 of piece r + 2 waits for it before it reuses this UOUT buffer
                B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_K5], st));
                B200C_CUDA_TRY(c, cudaStreamWaitEvent(c->stream5, c->ev_pool[EV_K5], 0));
                while (c->ev_k5.size() < k5_marks + 2) { cudaEvent_t e; cudaEventCreate(&e); c->ev_k5.push_back(e); }
                cudaEventRecord(c->ev_k5[k5_marks], c->stream5);
                c->stream = c->stream5;
            }
            int arc = B200C_OK;
            for (uint64_t off = 0; off < take && arc == B200C_OK; off += slice) arc = out_stream_append(os, UOUT + off, std::min(slice, take - off));
            if (k5_async) {
                c->stream = st;
                cudaEventRecord(c->ev_k5[k5_marks + 1], c->stream5); k5_marks += 2;
                B200C_CUDA_TRY(c, cudaEventRecord(c->ev_pool[EV_K5 + 1 + (r & 1)], c->stream5));
                k5_last = EV_K5 + 1 + (r & 1);
            }
            B200C_TRY(arc);
            tail_len = avail - take; tail_ptr = UOUT + take;
        }
        ubase_total += ulen_out; ilen_total += ilen_out;
    }
    // (progress: the last piece left bytes_scanned at (4 nr - 1) / (4 nr) of the input; the wrap-up below takes it to the total)

    // ---- K5 wrap-up / remaining writers ------------------------------------------------------------------------------------------------
    int rc = B200C_OK;
    auto finish_common = [&](RunStats& rs) -> int {          // error word, stats, histogram, stage clock
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_err, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 8, d_stats, sizeof(RunStats), cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 16, d_hist, MAXK * 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 201, d_rbytes, 8, cudaMemcpyDeviceToHost, st));
        mark(-1);
        int trc = timing_end(c);
        if (trc != B200C_OK) return trc;
        finish_marks();
        if (h[0] != ~0ull) { c->err = "internal error: size/emit pass disagreement at output partition " + std::to_string(h[0] & 0xFFFFFFFFFFFFull); return B200C_ECUDA; }
        memcpy(&rs, h + 8, sizeof(rs));
        memset(res->merged_row_counts, 0, sizeof(res->merged_row_counts));
        for (int k = 0; k < MAXK; k++) res->merged_row_counts[k] = h[16 + k];
        res->bytes_read = bytes_read; res->bytes_in_range = h[201]; res->bytes_written = ubase_total; res->total_source_rows = rs.merged_unfiltereds + nparts_total /* one applyToStatic -> updateProgress per merged partition */; res->input_partitions = ncontrib_total;
        res->kernel_ms = c->last_ms; res->kernel_launches = c->launches_call;
        return B200C_OK;
    };
    // Filter.db / Summary.db / first+last key / statistics side band of the single output -> the caller's (host) buffers
    auto finish_meta = [&](b200c_output& out) -> int {
        if (!want_meta) return B200C_OK;
        TdropDense* d_tdd; B200C_TRY(ws_typed(c, WS_META_TDD, 1, &d_tdd));
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_tdd, 0, 8, st));
        B200C_LAUNCH(c, k_tdrop_compact, TDROP_SLOTS / 1024, 1024, 0, d_td, d_tdd);
        B200C_LAUNCH(c, k_tdrop_final, TDROP_SLOTS / 1024, 1024, 0, d_td, d_tdd, d_sg);
        std::vector<uint8_t> hb(sizeof(StatGlobal)); StatGlobal* g = (StatGlobal*)hb.data();
        B200C_CUDA_TRY(c, cudaMemcpyAsync(g, d_sg, sizeof(StatGlobal), cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        out.first_key_len = written_total ? g->first_len : 0; out.last_key_len = written_total ? g->last_len : 0;
        int mrc = B200C_OK;                                 // a component that does not fit is skipped; the others (and every *_len) are still filled
        if (out.key_buf && out.key_cap < (uint64_t)out.first_key_len + out.last_key_len) { c->err = "key buffer too small"; mrc = B200C_ETOOSMALL; }
        else if (out.key_buf) {
            if (out.first_key_len) B200C_CUDA_TRY(c, cudaMemcpyAsync(out.key_buf, d_mkeys, out.first_key_len, cudaMemcpyDeviceToHost, st));
            if (out.last_key_len) B200C_CUDA_TRY(c, cudaMemcpyAsync(out.key_buf + out.first_key_len, d_mkeys + 65536, out.last_key_len, cudaMemcpyDeviceToHost, st));
        }
        if (out.filter) {                                   // BloomFilterSerializer.serialize: i32 hashCount | i32 words | bitset bytes
            out.filter_len = bloom_words ? 8 + bloom_words * 8 : 0;
            if (out.filter_len > out.filter_cap) { c->err = "filter buffer too small"; mrc = B200C_ETOOSMALL; }
            else if (bloom_words) {
                const uint32_t k = (uint32_t)m->bloom_hash_count, w = (uint32_t)bloom_words;
                uint8_t hd[8] = {(uint8_t)(k >> 24), (uint8_t)(k >> 16), (uint8_t)(k >> 8), (uint8_t)k, (uint8_t)(w >> 24), (uint8_t)(w >> 16), (uint8_t)(w >> 8), (uint8_t)w};
                memcpy(out.filter, hd, 8);
                B200C_CUDA_TRY(c, cudaMemcpyAsync(out.filter + 8, d_bloom, bloom_words * 8, cudaMemcpyDeviceToHost, st));
            }
        }
        if (out.summary) {                                  // IndexSummarySerializer.serialize + first / last key (S/io/sstable/indexsummary/IndexSummary.java:401-423)
            const uint64_t n = samples_total, eb = sument_bound, fl = out.first_key_len, ll = out.last_key_len;
            out.summary_len = written_total ? 24 + 4 * n + eb + 4 + fl + 4 + ll : 0;
            if (out.summary_len > out.summary_cap) { c->err = "summary buffer too small"; mrc = B200C_ETOOSMALL; }
            else if (written_total) {
                uint8_t* p = out.summary;
                auto be32 = [&](uint32_t v) { *p++ = (uint8_t)(v >> 24); *p++ = (uint8_t)(v >> 16); *p++ = (uint8_t)(v >> 8); *p++ = (uint8_t)v; };
                auto be64 = [&](uint64_t v) { be32((uint32_t)(v >> 32)); be32((uint32_t)v); };
                be32(meta_interval); be32((uint32_t)n); be64(4 * n + eb); be32(128); be32((uint32_t)((written_total + meta_interval - 1) / meta_interval));
                std::vector<uint64_t> offs(n);
                if (n) B200C_CUDA_TRY(c, cudaMemcpyAsync(offs.data(), d_sumoff, n * 8, cudaMemcpyDeviceToHost, st));
                if (eb) B200C_CUDA_TRY(c, cudaMemcpyAsync(p + 4 * n, d_sument, eb, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                for (uint64_t i = 0; i < n; i++) { uint32_t v = (uint32_t)(offs[i] + 4 * n); *p++ = (uint8_t)v; *p++ = (uint8_t)(v >> 8); *p++ = (uint8_t)(v >> 16); *p++ = (uint8_t)(v >> 24); }
                p += eb;
                std::vector<uint8_t> kb(fl + ll + 1);
                if (fl) B200C_CUDA_TRY(c, cudaMemcpyAsync(kb.data(), d_mkeys, fl, cudaMemcpyDeviceToHost, st));
                if (ll) B200C_CUDA_TRY(c, cudaMemcpyAsync(kb.data() + fl, d_mkeys + 65536, ll, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                be32((uint32_t)fl); memcpy(p, kb.data(), fl); p += fl; be32((uint32_t)ll); memcpy(p, kb.data() + fl, ll); p += ll;
            }
        }
        if (out.stats) {
            b200c_sstable_stats* s = out.stats; memset(s, 0, sizeof(*s));
            s->min_timestamp = (g->seen & 1) ? g->min_ts : I64_MIN; s->max_timestamp = (g->seen & 1) ? g->max_ts : I64_MAX;     // MinMaxLongTracker defaults
            s->min_local_deletion_time = (g->seen & 2) ? g->min_ldt : I64_MAX; s->max_local_deletion_time = (g->seen & 2) ? g->max_ldt : I64_MAX;
            s->min_ttl = (g->seen & 4) ? g->min_ttl : 0; s->max_ttl = (g->seen & 4) ? g->max_ttl : 0;
            s->total_rows = g->rows; s->total_columns_set = g->cols; s->total_cells = g->cells; s->total_tombstones = g->tombs;
            s->has_partition_level_deletions = g->pdel ? 1 : 0; s->tdrop_overflow = g->tdrop_overflow ? 1 : 0; s->has_legacy_counter_shards = (g->seen & 8) ? 1 : 0;
            for (int i = 0; i < META_PSIZE; i++) s->partition_size_hist[i] = g->psize[i];
            for (int i = 0; i < META_CELLS; i++) s->cells_per_partition_hist[i] = g->cells_hist[i];
            s->ntdrop = (uint32_t)std::min<uint64_t>(g->tdrop_n, B200C_TDROP_CAP);
            for (uint32_t i = 0; i < s->ntdrop; i++) { s->tdrop_point[i] = g->tdrop_point[i]; s->tdrop_count[i] = g->tdrop_count[i]; }
            for (int i = 0; i < META_HLL; i++) s->hll_registers[i] = (uint8_t)g->hll[i];
        }
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        return mrc;
    };
    // side band of one file of a multi-file output: partitions [jlo, jhi), Index.db positions relative to the file (iposf). Every file starts
    // from a fresh StatGlobal, tombstone table, bloom filter and summary; ranks count from the file's first written partition.
    // B200C_LCS_META_SPLIT=<file>: append one JSON line per file with where its side band's time goes (tools/bench_lcs_metadata.py)
    const char* split_path = lcs && want_meta ? getenv("B200C_LCS_META_SPLIT") : nullptr;
    int split_file = 0;
    auto file_meta = [&](uint64_t jlo, uint64_t jhi, const uint64_t* iposf, b200c_output& out) -> int {
        const uint64_t cnt = jhi - jlo;
        cudaEvent_t sev[4] = {nullptr, nullptr, nullptr, nullptr}; auto sw0 = std::chrono::steady_clock::now(), sw1 = sw0, sw2 = sw0;
        if (split_path) for (auto& e : sev) cudaEventCreate(&e);
        if (split_path) cudaEventRecord(sev[0], st);
        B200C_CUDA_TRY(c, cudaMemcpyAsync(d_sg, sg_init.data(), sizeof(StatGlobal), cudaMemcpyHostToDevice, st));
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_td, 0, sizeof(TdropTable), st));
        B200C_CUDA_TRY(c, cudaMemsetAsync(d_td->key, 0xFF, sizeof(d_td->key), st));
        if (bloom_words) B200C_CUDA_TRY(c, cudaMemsetAsync(d_bloom, 0, bloom_words * 8, st));
        B200C_TRY(launch_k4_stats(jlo, jhi));
        if (split_path) cudaEventRecord(sev[1], st);
        B200C_LAUNCH(c, k_written_flags, (unsigned)((cnt + 255) / 256), 256, 0, cnt, d_dsize + jlo, d_wflag);
        B200C_TRY(exclusive_scan<uint32_t>(c, d_wflag, cnt, d_wrank, WS_SCANA, 0));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 3, d_wrank + cnt, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 5, d_err, 8, cudaMemcpyDeviceToHost, st));
        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));                  // (also: sg_init has been copied)
        if ((h[5] >> 56) == 9 || (h[5] >> 56) == 4) {                                         // the statistics pass refused a partition the serialisation pass wrote
            res->corruption.input = (int)((h[5] >> 48) & 0xFF); res->corruption.kind = 4; res->corruption.chunk = 0; res->corruption.offset = h[5] & 0xFFFFFFFFFFFFull;
            timing_end(c);
            c->err = std::string((h[5] >> 56) == 9 ? "unsupported feature" : "malformed Data.db") + " in input " + std::to_string(res->corruption.input) + " (statistics pass of an output file)";
            return (h[5] >> 56) == 9 ? B200C_EUNSUPPORTED : B200C_ECORRUPT;
        }
        if (split_path) sw1 = std::chrono::steady_clock::now();
        const uint64_t nwritten = h[3], ns = (nwritten + meta_interval - 1) / meta_interval;
        uint32_t *d_samplej, *d_esize; uint64_t* d_epos;
        B200C_TRY(ws_typed(c, WS_META_SAMPLE, ns + 1, &d_samplej));
        B200C_TRY(ws_typed(c, WS_META_ESIZE, ns + 1, &d_esize));
        B200C_TRY(ws_typed(c, WS_META_EPOS, ns + 2, &d_epos));
        MetaArgs ma; memset(&ma, 0, sizeof(ma));
        ma.P = dP; ma.contrib = d_contrib; ma.op_first = d_opfirst + jlo; ma.upos = d_upos; ma.pbase = d_pbase; ma.dsize = d_dsize + jlo; ma.ipos = iposf + jlo; ma.ihead = d_ihead + jlo;
        ma.ccount = d_ccount + jlo; ma.wrank = d_wrank; ma.nparts = cnt; ma.index_base = 0; ma.written_base = 0; ma.sg = d_sg;
        ma.bloom = d_bloom; ma.bloom_bits = bloom_words * 64; ma.bloom_k = m->bloom_hash_count; ma.interval = meta_interval; ma.sample_j = d_samplej;
        ma.first_key = d_mkeys; ma.last_key = d_mkeys + 65536;
        if (cnt) B200C_LAUNCH(c, k_meta_keys, (unsigned)((cnt + 255) / 256), 256, 0, ma);
        written_total = nwritten; samples_total = 0; sument_bound = 0;
        if (ns && o0.summary) {
            B200C_LAUNCH(c, k_summary_sizes, (unsigned)((ns + 255) / 256), 256, 0, ma, ns, d_esize);
            B200C_TRY(exclusive_scan<uint32_t>(c, d_esize, ns, d_epos, WS_SCANA, 0));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 4, d_epos + ns, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            B200C_TRY(ws_typed(c, WS_META_SUMENT, h[4] + 64, &d_sument));
            B200C_TRY(ws_typed(c, WS_META_SUMOFF, ns + 2, &d_sumoff));
            B200C_LAUNCH(c, k_summary_emit, (unsigned)((ns + 255) / 256), 256, 0, ma, ns, d_epos, d_sument, d_sumoff);
            sument_bound = h[4]; samples_total = ns;
        }
        if (split_path) { cudaEventRecord(sev[2], st); B200C_CUDA_TRY(c, cudaStreamSynchronize(st)); sw2 = std::chrono::steady_clock::now(); }
        const int mrc = finish_meta(out);
        if (split_path) {
            cudaEventRecord(sev[3], st); cudaEventSynchronize(sev[3]);
            const auto sw3 = std::chrono::steady_clock::now();
            float ms[3] = {0, 0, 0}; for (int k = 0; k < 3; k++) cudaEventElapsedTime(&ms[k], sev[k], sev[k + 1]);
            auto wall = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            if (FILE* fp = fopen(split_path, "a")) {
                fprintf(fp, "{\"file\": %d, \"partitions\": %llu, \"stats_pass_ms\": %.3f, \"keys_summary_ms\": %.3f, \"finish_ms\": %.3f, \"wall_stats_ms\": %.3f, \"wall_keys_summary_ms\": %.3f, \"wall_finish_ms\": %.3f}\n",
                        split_file, (unsigned long long)cnt, ms[0], ms[1], ms[2], wall(sw0, sw1), wall(sw1, sw2), wall(sw2, sw3));
                fclose(fp);
            }
            for (auto& e : sev) cudaEventDestroy(e);
            split_file++;
        }
        return mrc;
    };
    if (to_host_stream) {
        b200c_output& out = out0;
        uint64_t out_len = 0; uint32_t digest = 0; uint64_t* d_ooffs = nullptr;
        if (k5_last >= 0) B200C_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_pool[k5_last], 0));      // every piece's K5 is done before the digest
        B200C_TRY(out_stream_finish(os, &out_len, &digest, &d_ooffs));
        const uint64_t nchunks_out = os.nchunks;
        RunStats rs; B200C_TRY(finish_common(rs));
        res->noutputs = 1;
        res->required_data_cap = std::max<uint64_t>(out_len, 1); res->required_index_cap = ilen_total; res->required_chunk_cap = nchunks_out;
        out.data_len = out_len; out.index_len = ilen_total; out.nchunks = nchunks_out; out.data_length = ubase_total; out.digest = digest;
        out.partitions = rs.partitions_out; out.rows = rs.rows_out;
        { int mrc = finish_meta(out); if (mrc != B200C_OK) rc = mrc; }
        if (!os.fits || !index_fits || out_len > out.data_cap || ilen_total > out.index_cap || nchunks_out > out.chunk_cap) { c->err = "output buffers too small"; rc = B200C_ETOOSMALL; }
        else {
            if (nchunks_out) B200C_CUDA_TRY(c, cudaMemcpyAsync(out.chunk_offsets, d_ooffs, nchunks_out * 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        }
        B200C_CUDA_TRY(c, cudaStreamSynchronize(c->copy_out));
    } else if (!lcs) {
        // one output file in device memory
        b200c_output& out = out0;
        const uint64_t nchunks_out = (ulen_out + L - 1) / L;
        const uint64_t bound = b200c_compress_bound(m->out_compressor, ulen_out, m->out_chunk_len);
        res->required_data_cap = bound; res->required_index_cap = ilen_out; res->required_chunk_cap = nchunks_out;
        if (out.data_cap < bound) { c->err = "output data buffer too small"; timing_end(c); return B200C_ETOOSMALL; }
        uint64_t* d_ooffs; B200C_TRY(ws_typed(c, WS_OOFFS, nchunks_out + 2, &d_ooffs));
        uint64_t out_len = 0; uint32_t digest = 0;
        B200C_TRY(compress_stream_device(c, m->out_compressor, UOUT, ulen_out, m->out_chunk_len, m->out_max_compressed_len, out.data, bound, d_ooffs, &out_len, &digest, WS_CODEC));
        RunStats rs; B200C_TRY(finish_common(rs));
        res->noutputs = 1;
        out.data_len = out_len; out.index_len = ilen_out; out.nchunks = nchunks_out; out.data_length = ulen_out; out.digest = digest;
        out.partitions = rs.partitions_out; out.rows = rs.rows_out;
        { int mrc = finish_meta(out); if (mrc != B200C_OK) rc = mrc; }
        if (out_len > out.data_cap || ilen_out > out.index_cap || nchunks_out > out.chunk_cap) { c->err = "output buffers too small"; rc = B200C_ETOOSMALL; }
        else {
            if (ilen_out) B200C_CUDA_TRY(c, cudaMemcpyAsync(out.index, IOUT, ilen_out, cudaMemcpyDeviceToDevice, st));
            if (nchunks_out) B200C_CUDA_TRY(c, cudaMemcpyAsync(out.chunk_offsets, d_ooffs, nchunks_out * 8, cudaMemcpyDeviceToDevice, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
        }
    } else {
        // ---- multi-file output: one pass per file over a compressed window (see k_find_cut) ----------------------------------------
        const int comp = m->out_compressor; const int stride = chunk_slot_stride(comp, (int)L);
        const uint64_t nch_total = (ulen_out + L - 1) / L;
        uint8_t* slots; uint32_t *file_len, *seg_raw; uint64_t *woffs, *d_dposf, *d_iposf, *d_cut, *d_ooffs; uint8_t *IOUTF, *d_dout; RunStats* d_fstats;
        B200C_TRY(ws_typed(c, WS_CODEC + 2, (nch_total + 2) * (uint64_t)stride, &slots));
        B200C_TRY(ws_typed(c, WS_CODEC + 3, nch_total + 2, &file_len));
        B200C_TRY(ws_typed(c, WS_CODEC + 4, nch_total + 2, &seg_raw));
        B200C_TRY(ws_typed(c, WS_LCS0, nch_total + 4, &woffs));
        B200C_TRY(ws_typed(c, WS_LCS1, nparts + 2, &d_dposf));
        B200C_TRY(ws_typed(c, WS_LCS2, nparts + 2, &d_iposf));
        B200C_TRY(ws_typed(c, WS_LCS3, 64, &d_cut)); d_fstats = (RunStats*)(d_cut + 8);
        B200C_TRY(ws_typed(c, WS_IOUT + 0, ilen_out + 64, &IOUT));
        B200C_TRY(ws_typed(c, WS_LCS4, ilen_out + 64, &IOUTF));
        B200C_TRY(ws_typed(c, WS_OOFFS, nch_total + 4, &d_ooffs));
        const uint64_t file_bound = b200c_compress_bound(comp, ulen_out, (int)L);
        B200C_TRY(ws_typed(c, WS_DOUT, file_bound + 64, &d_dout));
        res->required_data_cap = res->required_index_cap = res->required_chunk_cap = 0;
        uint64_t jlo = 0, start_b = 0; int f = 0;
        // how much of the stream to compress before looking for the file boundary: the file holds max_sstable_bytes of COMPRESSED chunks, so the
        // window is that divided by the ratio seen so far (the inputs' own ratio for the first file, then the previous file's) plus 8 %; a window
        // that turns out too short is extended below (doubling), nothing is compressed twice
        double est_ratio = 0.5;
        { uint64_t ci = 0, ui = 0; for (int i = 0; i < K; i++) { ci += m->inputs[i].data_len; ui += m->inputs[i].data_length; } if (ui) est_ratio = std::min(1.0, std::max(0.05, (double)ci / (double)ui)); }
        while (jlo < nparts && start_b < ulen_out) {
            B200C_TRY(check_cancel());
            const uint64_t remaining = ulen_out - start_b, rem_chunks = (remaining + L - 1) / L;
            uint64_t want = std::max<uint64_t>(64, (uint64_t)std::min(1e18, (double)m->max_sstable_bytes / est_ratio * 1.08) / L + 8), done = 0, jhi = nparts, status = 2;
            while (status == 2) {
                uint64_t W = std::min(rem_chunks, want);
                if (W > done) B200C_TRY(compress_slots_device(c, comp, UOUT + start_b + done * L, std::min(remaining - done * L, (W - done) * (uint64_t)L), (int)L,
                                                              m->out_max_compressed_len, slots + done * stride, stride, file_len + done, seg_raw + done));
                done = W;
                // bytes flushed before a partition = whole chunks only: a trailing partial chunk of the window is not "flushed"
                uint64_t nfull_known = (W == rem_chunks) ? (remaining / L) : W;
                B200C_TRY(exclusive_scan<uint32_t>(c, file_len, nfull_known, woffs, WS_SCANA, 0));
                B200C_LAUNCH(c, k_find_cut, 1, 1, 0, d_dpos, jlo, nparts, start_b, woffs, (W == rem_chunks) ? ~0ull >> 1 : nfull_known, L, m->max_sstable_bytes, d_cut);
                B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_cut, 16, cudaMemcpyDeviceToHost, st));
                B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                jhi = h[0]; status = h[1];
                if (status == 2) { if (W == rem_chunks) { status = 1; jhi = nparts; } else want *= 2; }
            }
            // the file is partitions [jlo, jhi), bytes [start_b, end_b)
            uint64_t end_b = ulen_out;
            if (jhi < nparts) { B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_dpos + jhi, 8, cudaMemcpyDeviceToHost, st)); B200C_CUDA_TRY(c, cudaStreamSynchronize(st)); end_b = h[0]; }
            const uint64_t flen = end_b - start_b, fchunks = (flen + L - 1) / L, nfull = flen / L, tail = flen % L;
            if (tail && !(end_b == ulen_out && done == rem_chunks))      // the last chunk of the file is shorter than what the window compressed there
                B200C_TRY(compress_slots_device(c, comp, UOUT + start_b + nfull * L, tail, (int)L, m->out_max_compressed_len, slots + nfull * stride, stride, file_len + nfull, seg_raw + nfull));
            uint64_t out_len = 0; uint32_t digest = 0;
            B200C_TRY(pack_digest_device(c, slots, stride, file_len, seg_raw, fchunks, d_dout, file_bound, d_ooffs, &out_len, &digest, WS_CODEC));
            // Index.db of this file: positions relative to the file start
            const uint64_t cnt = jhi - jlo;
            B200C_LAUNCH(c, k_rel_pos, (unsigned)((cnt + 1 + 255) / 256), 256, 0, d_dpos, jlo, jhi, start_b, d_dposf);
            B200C_LAUNCH(c, k_index_sizes, (unsigned)((cnt + 255) / 256), 256, 0, cnt, d_dsize + jlo, d_dposf + jlo, d_ipay + jlo, d_ihead + jlo, d_isize + jlo);
            B200C_TRY(exclusive_scan<uint32_t>(c, d_isize + jlo, cnt, d_iposf + jlo, WS_SCANA + 3, 0));
            B200C_CUDA_TRY(c, cudaMemsetAsync(d_fstats, 0, sizeof(RunStats), st));
            B200C_LAUNCH(c, k_sum_stats, 296, 256, 0, cnt, d_dsize + jlo, d_stmunf + jlo, d_strows + jlo, d_fstats);
            B200C_LAUNCH(c, k_index_simple, (unsigned)((cnt + 255) / 256), 256, 0, dP, cnt, d_contrib, d_opfirst + jlo, d_upos, d_pbase, d_dsize + jlo, d_dposf + jlo,
                         d_nblk + jlo, d_ovf + jlo, d_ihead + jlo, d_iposf + jlo, IOUTF);
            if (!two_pass) B200C_LAUNCH(c, k_index_promoted, (unsigned)((cnt + 127) / 128), 128, 0, dP, cnt, d_contrib, d_opfirst + jlo, d_upos, d_pbase, d_dsize + jlo, d_dposf + jlo,
                                        d_nblk + jlo, d_ovf + jlo, d_ihead + jlo, d_ipay + jlo, d_iposf + jlo, d_ioff + jlo, d_icap + jlo, ISCR, IOUTF);
            ka.dbase = UOUT + start_b; ka.iout = IOUTF; ka.dpos = d_dposf; ka.ipos = d_iposf; ka.jlo = jlo; ka.jhi = jhi;
            B200C_TRY(launch_k4(3));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h, d_iposf + jhi, 8, cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaMemcpyAsync(h + 8, d_fstats, sizeof(RunStats), cudaMemcpyDeviceToHost, st));
            B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
            const uint64_t filen = h[0]; RunStats fs; memcpy(&fs, h + 8, sizeof(fs));
            if (flen && out_len) est_ratio = std::min(1.0, std::max(0.05, (double)out_len / (double)flen));
            res->required_data_cap = std::max<uint64_t>(res->required_data_cap, out_len);
            res->required_index_cap = std::max<uint64_t>(res->required_index_cap, filen);
            res->required_chunk_cap = std::max<uint64_t>(res->required_chunk_cap, fchunks);
            if (fs.partitions_out) {
                if (f >= res->noutputs_cap) { c->err = "more output files than output slots"; rc = B200C_ETOOSMALL; }
                else {
                    b200c_output& o = res->outputs[f];
                    if (out_len > o.data_cap || filen > o.index_cap || fchunks > o.chunk_cap) { c->err = "output buffers too small"; rc = B200C_ETOOSMALL; }
                    else {
                        cudaMemcpyKind k = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
                        if (out_len) B200C_CUDA_TRY(c, cudaMemcpyAsync(o.data, d_dout, out_len, k, st));
                        if (filen) B200C_CUDA_TRY(c, cudaMemcpyAsync(o.index, IOUTF, filen, k, st));
                        if (fchunks) B200C_CUDA_TRY(c, cudaMemcpyAsync(o.chunk_offsets, d_ooffs, fchunks * 8, k, st));
                        B200C_CUDA_TRY(c, cudaStreamSynchronize(st));
                        o.data_len = out_len; o.index_len = filen; o.nchunks = fchunks; o.data_length = flen; o.digest = digest;
                        o.partitions = fs.partitions_out; o.rows = fs.rows_out;
                    }
                    if (want_meta) { const int mrc = file_meta(jlo, jhi, d_iposf, o); if (mrc == B200C_ETOOSMALL) rc = mrc; else B200C_TRY(mrc); }
                }
                f++;
            }
            jlo = jhi; start_b = end_b;
        }
        RunStats rs; B200C_TRY(finish_common(rs));
        res->noutputs = f;
    }
    c->prog_scanned.store(bytes_read); c->prog_stage.store(6);
    res->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    return rc;
}

int64_t b200c_token(int partitioner, const uint8_t* key, uint32_t len) {
    if (partitioner == B200C_PARTITIONER_BYTE_ORDERED) { uint64_t pre = 0; for (uint32_t q = 0; q < 8; q++) pre = (pre << 8) | (q < len ? key[q] : 0); return (int64_t)(pre ^ 0x8000000000000000ull); }
    return murmur3_token(key, len);
}

int b200c_poll(b200c_ctx* c, b200c_progress* p) {
    if (!c || !p) return B200C_EINVAL;
    p->call_seq = c->prog_seq.load(); p->bytes_scanned = c->prog_scanned.load(); p->bytes_total = c->prog_total.load(); p->stage = c->prog_stage.load();
    return B200C_OK;
}
int b200c_poll_inputs(b200c_ctx* c, uint64_t* positions, int n) {
    if (!c || !positions || n < 0) return B200C_EINVAL;
    int k = c->prog_ninputs.load(); if (k > n) k = n;
    for (int i = 0; i < k; i++) positions[i] = c->prog_input_pos[i].load();
    return k;
}
void b200c_cancel(b200c_ctx* c) { if (c) c->cancel.store(1); }
void b200c_cancel_reset(b200c_ctx* c) { if (c) c->cancel.store(0); }

} // extern "C"
