// engine.cuh — context, workspace and launch bookkeeping shared by the C-ABI translation units.
#pragma once
#include <cstdio>
#include <cstring>
#include <string>
#include <atomic>
#include <chrono>
#include <vector>
#include "../../include/b200c.h"
#include "common.cuh"

namespace b200c {

enum { WS_SLOTS = 160, WS_K5_ENT = 150, WS_K1_REC = 151, WS_K1_NSEQ = 152 };      // (slots 0..15: codec calls, 16..: compact.cu's map, 150: K5's hash-chain entries, 151-152: K1's sequence records)

struct WsBuf { void* p = nullptr; size_t cap = 0; };

} // namespace b200c

struct b200c_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    b200c::DevTables* d_tables = nullptr;
    b200c::WsBuf ws[b200c::WS_SLOTS];
    void* h_pinned = nullptr; size_t h_pinned_cap = 0;      // small pinned scratch for scalar read-backs
    std::string err;
    uint64_t launches_call = 0, launches_total = 0;
    double last_ms = 0.0;
    std::atomic<int> cancel{0};
    std::atomic<uint64_t> prog_scanned{0}, prog_total{0};
    std::atomic<int> prog_stage{0}; std::atomic<int> prog_seq{0};
    std::atomic<int> prog_ninputs{0};
    std::atomic<uint64_t> prog_input_pos[B200C_MAX_INPUTS];   // uncompressed bytes of each input consumed so far (b200c_poll_inputs)
    bool timing = false;
    cudaEvent_t ev_stage[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int nstages = 0;
    int k4_attr_set = 0, k4s_attr_set = 0, k4st_attr_set = 0;
    cudaStream_t copy_stream = nullptr;            // host->device staging of the inputs, overlapped with K1 input by input
    cudaEvent_t ev_in[64] = {};
    std::vector<cudaEvent_t> ev_marks;             // timed events of the stage clock (grown on demand)
    cudaEvent_t ev_pool[256] = {};                 // untimed events: OutStream pieces (2 each), token-range staging
    cudaStream_t copy_out = nullptr;               // device->host stream of the outputs (the other copy engine)
    cudaStream_t stream5 = nullptr;                // K5 of streamed piece r runs here, under K1..K3 (and the copies they wait for) of piece r + 1
    std::vector<cudaEvent_t> ev_k5;                // timed event pairs around each piece's K5 on stream5 (stage clock)
};

namespace b200c {

#define B200C_CUDA_TRY(ctx, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e); return B200C_ECUDA; } } while (0)

#define B200C_LAUNCH(ctx, kernel, grid, block, smem, ...) do { \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__); \
    (ctx)->launches_call++; (ctx)->launches_total++; \
    cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { \
        (ctx)->err = std::string(#kernel) + " launch: " + cudaGetErrorString(_e); return B200C_ECUDA; } } while (0)

#define B200C_TRY(expr) do { int _rc = (expr); if (_rc != B200C_OK) return _rc; } while (0)

// workspace slot `slot` with at least `bytes` bytes (+64 bytes of readable slack); contents are NOT preserved on growth
inline int ws_get(b200c_ctx* c, int slot, size_t bytes, void** out) {
    WsBuf& b = c->ws[slot];
    size_t need = bytes + 256;
    if (b.cap < need) {
        if (b.p) { cudaStreamSynchronize(c->stream); if (c->copy_stream) cudaStreamSynchronize(c->copy_stream); if (c->copy_out) cudaStreamSynchronize(c->copy_out); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
        size_t cap = need + need / 8;
        cudaError_t e = cudaMalloc(&b.p, cap);
        if (e != cudaSuccess) { cudaGetLastError(); c->err = "cudaMalloc(" + std::to_string(cap) + "): " + cudaGetErrorString(e); b.p = nullptr; return B200C_ENOMEM; }
        b.cap = cap;
    }
    *out = b.p;
    return B200C_OK;
}
template <typename T> inline int ws_typed(b200c_ctx* c, int slot, size_t count, T** out) {
    void* p; int rc = ws_get(c, slot, count * sizeof(T), &p); *out = (T*)p; return rc;
}

// workspace slot that keeps its first `used` bytes when it has to grow (whole-file arrays of an OutStream)
template <typename T> inline int ws_grow_keep(b200c_ctx* c, int slot, size_t count, size_t used, T** out) {
    WsBuf& b = c->ws[slot];
    size_t need = count * sizeof(T) + 256;
    if (b.cap < need) {
        cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->copy_out);
        void* np = nullptr; size_t cap = need * 2;
        cudaError_t e = cudaMalloc(&np, cap);
        if (e != cudaSuccess) { cudaGetLastError(); c->err = "cudaMalloc(" + std::to_string(cap) + "): " + cudaGetErrorString(e); return B200C_ENOMEM; }
        if (b.p && used) cudaMemcpy(np, b.p, std::min(used * sizeof(T), b.cap), cudaMemcpyDeviceToDevice);
        if (b.p) cudaFree(b.p);
        b.p = np; b.cap = cap;
    }
    *out = (T*)b.p;
    return B200C_OK;
}

inline void timing_begin(b200c_ctx* c) { c->launches_call = 0; cudaEventRecord(c->ev0, c->stream); c->timing = true; }
inline int timing_end(b200c_ctx* c) {
    cudaEventRecord(c->ev1, c->stream);
    B200C_CUDA_TRY(c, cudaEventSynchronize(c->ev1));
    float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms; c->timing = false;
    return B200C_OK;
}

// K5 of one output file fed in pieces (engine.cu)
struct OutStream {
    enum { MAX_PIECES = 96 };
    b200c_ctx* c = nullptr; int comp = 0, L = 0, max_clen = 0, stride = 0, ws_base = 0;
    uint8_t* h_out = nullptr; uint64_t h_cap = 0;           // the caller's Data.db buffer
    uint32_t *file_len = nullptr, *seg_raw = nullptr, *acc = nullptr; uint64_t *d_offs = nullptr, *bases = nullptr;
    uint8_t* img[2] = {nullptr, nullptr}; uint64_t img_cap[2] = {0, 0};
    uint64_t nchunks = 0, ulen = 0, copied = 0; int piece = 0; bool fits = true;
};
int out_stream_begin(OutStream& o, b200c_ctx* c, int comp, int chunk_len, int max_clen, uint8_t* h_out, uint64_t h_cap, int ws_base);
int out_stream_append(OutStream& o, const uint8_t* d_in, uint64_t nbytes);
int out_stream_finish(OutStream& o, uint64_t* out_len, uint32_t* digest, uint64_t** d_offs_out);

// device-wide exclusive scan: out[0..n] (n+1 entries, out[n] = total). TIn = uint32_t or uint64_t. scan_slot0: first of 3 ws slots.
template <typename TIn> int exclusive_scan(b200c_ctx* c, const TIn* in, uint64_t n, uint64_t* out, int scan_slot0, int depth = 0);

} // namespace b200c
