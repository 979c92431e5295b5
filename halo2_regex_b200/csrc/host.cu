// Host-pointer entry points of include/b2r.h: what a drop-in shim around `match_substrs` (reference src/lib.rs:311-315) calls.
//
//   b2r_match_batch_host   the batch is cut into slices of strings; the H2D copy of slice i+1, the kernels of slice i and the
//                          D2H copies of slice i-1 run on three streams (PCIe is full duplex, the copies are the bottleneck).
//                          B2R_OUT_SPARSE_D2H: the zero-dominated columns (substr ids, enable bitmaps, masked chars / ids) are
//                          compacted on the device into (sector index, 32-byte sector) pairs, cross PCIe in that form and are
//                          expanded into the caller's dense buffers by host threads (memset + scatter) — every value is still
//                          computed by the kernels, only the zeros stay home.
//   small batches          (one tile of <= 32 strings, e.g. the reference's one-string call): one H2D copy, one memset, two
//                          kernels, one D2H copy through a pinned staging arena.
//   multi-device handle    b2r_config_new_multi: one process, several GPUs; strings sharded by bytes, one host thread per
//                          device, ONE ncclAllReduce (u64 sum) of the multiplicity block over NVLink (SURVEY 8(b), 8(e)).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types and prototypes only: the library is dlopen'ed (libb2r.so does not link against NCCL)

#include <algorithm>
#include <array>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "config.hpp"
#include "long.cuh"

using namespace b2r;

namespace b2r {

// ---- host worker pool --------------------------------------------------------------------------------------------------
HostPool::HostPool(unsigned n_threads) {
    for (unsigned i = 0; i < (n_threads ? n_threads : 1u); i++) threads_.emplace_back([this] { run(); });
}
HostPool::~HostPool() {
    { std::lock_guard<std::mutex> l(m_); stop_ = true; }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
}
void HostPool::submit(std::function<void()> fn) {
    { std::lock_guard<std::mutex> l(m_); q_.push_back(std::move(fn)); pending_++; }
    cv_.notify_one();
}
void HostPool::wait() {
    std::unique_lock<std::mutex> l(m_);
    done_.wait(l, [this] { return pending_ == 0; });
}
void HostPool::run() {
    for (;;) {
        std::function<void()> fn;
        {
            std::unique_lock<std::mutex> l(m_);
            cv_.wait(l, [this] { return stop_ || !q_.empty(); });
            if (q_.empty()) return;
            fn = std::move(q_.front());
            q_.pop_front();
        }
        fn();
        { std::lock_guard<std::mutex> l(m_); if (--pending_ == 0) done_.notify_all(); }
    }
}

// ---- sparse D2H: device-side compaction of a zero-dominated column -----------------------------------------------------------
// Non-zero 32-byte sectors of the column slice are appended as (sector index, 32 bytes).  A CTA takes 4096 consecutive sectors at
// a time, counts its non-zero ones, reserves their places with ONE atomic and writes them in ascending sector order: the host
// threads that scatter the list into the caller's dense column (and clear it again before the next call) then walk through memory
// in long ascending runs instead of jumping at random (page-table walks and DRAM row misses were most of their time).
// `count` keeps counting past `cap`: the host sees the overflow and copies that column slice densely instead.
constexpr int SPARSIFY_K = 16;           // sectors per thread and pass
__global__ void __launch_bounds__(256) sparsify_kernel(const uint4* __restrict__ col, uint64_t n_sectors, uint32_t* __restrict__ idx, uint4* __restrict__ payload,
                                                       uint32_t cap, unsigned int* count) {
    __shared__ uint32_t s_cnt[SPARSIFY_K * 8];                             // non-zero sectors of (row j, warp w), then their exclusive prefix
    __shared__ uint32_t s_wsum[4], s_base;
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr uint64_t PER_CTA = 256 * SPARSIFY_K;
    for (uint64_t b0 = (uint64_t)blockIdx.x * PER_CTA; b0 < n_sectors; b0 += (uint64_t)gridDim.x * PER_CTA) {
        uint32_t mine = 0;                                                 // bit j: my sector of row j is non-zero
#pragma unroll
        for (int j = 0; j < SPARSIFY_K; j++) {
            const uint64_t s = b0 + (uint64_t)j * 256 + threadIdx.x;
            uint4 a = make_uint4(0, 0, 0, 0), b = a;
            if (s < n_sectors) { a = __ldcg(col + 2 * s); b = __ldcg(col + 2 * s + 1); }
            const bool nz = (a.x | a.y | a.z | a.w | b.x | b.y | b.z | b.w) != 0;
            const unsigned m = __ballot_sync(0xffffffffu, nz);
            if (nz) mine |= 1u << j;
            if (lane == 0) s_cnt[j * 8 + warp] = (uint32_t)__popc(m);
        }
        __syncthreads();
        // exclusive prefix over the SPARSIFY_K * 8 = 128 counts, in (row, warp) order = ascending sector order
        uint32_t v = 0, incl = 0;
        if (threadIdx.x < SPARSIFY_K * 8) {
            v = s_cnt[threadIdx.x];
            incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += t; }
            if (lane == 31) s_wsum[warp] = incl;
        }
        __syncthreads();
        if (threadIdx.x < SPARSIFY_K * 8) {
            uint32_t before = 0;
            for (unsigned w = 0; w < warp; w++) before += s_wsum[w];
            s_cnt[threadIdx.x] = before + incl - v;
            if (threadIdx.x == SPARSIFY_K * 8 - 1) {
                const uint32_t total = before + incl;
                s_base = total ? atomicAdd(count, total) : 0u;
            }
        }
        __syncthreads();
        if (__any_sync(0xffffffffu, mine != 0)) {
            const uint32_t base = s_base;
#pragma unroll 1
            for (int j = 0; j < SPARSIFY_K; j++) {
                const bool nz = (mine >> j) & 1u;
                const unsigned m = __ballot_sync(0xffffffffu, nz);
                if (!nz) continue;
                const uint32_t k = base + s_cnt[j * 8 + warp] + (uint32_t)__popc(m & ((1u << lane) - 1u));
                if (k < cap) {
                    const uint64_t s = b0 + (uint64_t)j * 256 + threadIdx.x;
                    idx[k] = (uint32_t)s;
                    payload[2 * (size_t)k] = __ldcg(col + 2 * s); payload[2 * (size_t)k + 1] = __ldcg(col + 2 * s + 1);   // the second read hits L2
                }
            }
        }
        __syncthreads();                                                   // s_cnt / s_base are reused by the next pass
    }
}

// the sector counts of one slice -> pinned host memory (a store over PCIe instead of a copy: the copy engines are busy with the
// dense columns, and a small copy queued behind them would stall the compute stream)
__global__ void publish_counts_kernel(const unsigned int* __restrict__ dev_cnt, unsigned int* host_cnt, uint32_t n) {
    if (threadIdx.x < n) host_cnt[threadIdx.x] = dev_cnt[threadIdx.x];
}

}  // namespace b2r

namespace {

// hook of a multi-device batch into the per-device pipeline: after the last slice has been finalised the multiplicity block
// is all-reduced; only the first device copies it back
struct MultiHook {
    ncclComm_t comm = nullptr;
    ncclResult_t (*all_reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*error_string)(ncclResult_t) = nullptr;
    bool first = true;                 // this device uploads the caller's counters (accumulate) and copies the result back
    // packed per-string counts: the entries of device k start where those of devices < k end
    struct PkChain* chain = nullptr;
    int index = 0;
    bool last = true;                  // this device writes row_start[N]
};

// The totals a multi-device packed call's devices publish in device order (device k waits for devices < k before it issues its
// entry copies).  A device publishes exactly once, also when its call fails, so that no other device waits forever.
struct PkChain {
    std::mutex m;
    std::condition_variable cv;
    std::vector<char> done;
    std::vector<std::array<uint64_t, B2R_MAX_DEFS>> total;
    explicit PkChain(int n) : done(n, 0), total(n) {}
    void publish(int k, const uint64_t* t) {
        { std::lock_guard<std::mutex> l(m); if (done[k]) return; for (int d = 0; d < B2R_MAX_DEFS; d++) total[k][d] = t[d]; done[k] = 1; }
        cv.notify_all();
    }
    void base(int k, uint64_t* b) {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { for (int q = 0; q < k; q++) if (!done[q]) return false; return true; });
        for (int d = 0; d < B2R_MAX_DEFS; d++) { b[d] = 0; for (int q = 0; q < k; q++) b[d] += total[q][d]; }
    }
};
struct PkPublishOnExit {
    const MultiHook* hook;
    ~PkPublishOnExit() { if (hook && hook->chain) { const uint64_t z[B2R_MAX_DEFS] = {}; hook->chain->publish(hook->index, z); } }
};

unsigned default_host_threads() {
    unsigned hw = std::thread::hardware_concurrency();
    if (!hw) hw = 4;
    unsigned share = 1;                // ranks of a torchrun job share the host cores
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) { const int v = atoi(e); if (v > 1) share = (unsigned)v; }
    // three quarters of the cores, at most 12.  Clearing and scattering one 32-byte sector is one cache miss; a core keeps about a
    // dozen in flight, so the sector rate grows with the threads until they take memory bandwidth from the DMA engines
    // (2^20 x 1 KiB strings, 16-core host, staged sparse mode: 33.9 ms per call with 8 threads, 33.0 with 12; 16 is slower)
    return std::max(2u, std::min(12u, hw * 3 / 4 / share));
}

struct SparseCol {                     // one zero-dominated column of a host batch
    unsigned char* host;               // caller's dense buffer
    unsigned char* dev;                // device column (arena)
    size_t pitch;                      // bytes per string
};

bool is_pinned(const void* h) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, h) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// ---- packed per-string counts: what a slice's lists take, and how many of its entries are stored ----------------------------------
// slots per string of the packed post-pass (string_mult.cu): no list is longer
uint64_t pk_pitch(const b2r_config* c, uint64_t M) {
    uint64_t w = 1;
    for (uint32_t d = 0; d < c->n_defs; d++) w = std::max<uint64_t>(w, std::min<uint64_t>(M, c->packed[d].rows.size()));
    return w;
}

// The entries of ni strings whose lists start at `base` in the caller's area and which are stored under `cap`: the lists of a prefix
// of them (row_start does not decrease), none in part.  rel[k - 1] = row_start[k] - base for 1 <= k <= ni, so rel[ni - 1] is the total.
uint64_t pk_stored(uint64_t base, uint64_t cap, const uint64_t* rel, uint64_t ni) {
    if (!ni || base >= cap) return 0;
    if (base + rel[ni - 1] <= cap) return rel[ni - 1];
    const uint64_t* p = std::upper_bound(rel, rel + ni, cap - base);    // the first list end beyond the capacity
    return p == rel ? 0 : p[-1];
}

// ---- small batches: one tile, one copy each way ------------------------------------------------------------------------------
// Everything the call needs lives in ONE device arena (ws_cols) mirrored by ONE pinned host arena (pin_small):
//   [offsets (n+1) u64 | input bytes | multiplicity block | BatchCounters copy | every requested column]
// the first three parts go up in one copy, everything from the multiplicity block on comes back in one copy.
int host_batch_small(b2r_config* c, BatchEntry entry, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                     const b2r_string_mult_outputs* sm, const b2r_string_mult_packed_outputs* pk, b2r_batch_status* result) {
    cudaStream_t st = c->host_stream;
    const bool trace = c->opt.trace_host;
    const auto wall0 = std::chrono::steady_clock::now();
    auto wall_us = [&] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - wall0).count(); };
    double w_prep = 0, w_up = 0, w_enq = 0, w_sync = 0;
    const uint64_t base = h_offsets[0], nbytes = h_offsets[n] - base;
    const uint64_t rp = ho->row_pitch, bp = ho->bitmap_pitch;
    const bool acc = (ho->flags & B2R_OUT_ACCUMULATE_MULT) != 0;
    size_t need = 0;
    auto slot = [&](size_t bytes, size_t align = 256) { need = align_up(need, align); size_t o = need; need += bytes; return o; };
    const size_t off_offs = slot((n + 1) * 8), off_bytes = slot(nbytes + 16), off_mult = slot(0);
    struct Part { size_t off; void* host; size_t bytes; };
    std::vector<Part> parts;            // device arena offset <-> caller's buffer
    b2r_outputs dout = *ho;
    auto want = [&](void* host, size_t bytes, size_t align = 256) -> size_t { if (!host) return 0; const size_t o = slot(bytes, align); parts.push_back({o, host, bytes}); return o; };
    size_t o_mult[B2R_MAX_DEFS], o_em[B2R_MAX_DEFS];
    for (uint32_t d = 0; d < c->n_defs; d++) {
        o_mult[d] = want(ho->mult[d], c->packed[d].rows.size() * 8, 8);
        o_em[d] = want(ho->endpoint_mult[d], c->packed[d].erows.size() * 16, 8);
    }
    const size_t mult_end = need;
    const size_t off_cnt = slot(sizeof(BatchCounters), 64);
    size_t o_states[B2R_MAX_DEFS], o_sid[B2R_MAX_DEFS], o_se[B2R_MAX_DEFS], o_ee[B2R_MAX_DEFS];
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const size_t w = c->packed[d].state_width;
        o_states[d] = want(ho->states[d], n * rp * w); o_sid[d] = want(ho->substr_ids[d], n * rp);
        o_se[d] = want(ho->start_enable[d], n * bp); o_ee[d] = want(ho->end_enable[d], n * bp);
    }
    const size_t o_mc = want(ho->masked_chars, n * rp), o_ms = want(ho->masked_substr_ids, n * rp);
    const size_t o_st = want(ho->status, n * sizeof(b2r_string_status));
    const size_t o_rec = want(ho->records, n * (size_t)ho->max_records * sizeof(b2r_substr_record));
    const size_t o_cb = want(ho->compact_bytes, n * (size_t)ho->compact_pitch);
    // per-string counts: they come back with the columns; the entry slots go up first (the post-pass leaves unused slots alone)
    bool want_sm = false;
    b2r_string_mult_outputs dsm{};
    size_t o_ent[B2R_MAX_DEFS] = {}, o_nent[B2R_MAX_DEFS] = {}, o_epc[B2R_MAX_DEFS] = {};
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!string_mult_wanted(c, sm, d)) continue;
        want_sm = true;
        o_ent[d] = want(sm->entries[d], n * (size_t)sm->max_entries * sizeof(b2r_row_count));
        o_nent[d] = want(sm->n_entries[d], n * 4);
        o_epc[d] = want(sm->endpoint_counts[d], n * c->packed[d].erows.size() * 8);
    }
    bool want_pk = false;
    for (uint32_t d = 0; d < c->n_defs; d++) want_pk = want_pk || string_mult_packed_wanted(c, pk, d);
    const size_t o_st_scratch = (want_sm || want_pk) && !ho->status ? slot(n * sizeof(b2r_string_status)) : 0;   // the post-pass reads the status
    need = align_up(need, 256);
    // packed per-string counts (b2r_match_batch_host_mult_packed): after the arena's one copy, each part copied back exactly —
    // row_start[1..n] (row_start[0] is 0) and the endpoint counts; the pack kernel stores the entries straight into the pinned
    // arena (one slice: the capacity rule is the caller's), so only stored entries cross
    const size_t pk_begin = need;
    size_t o_pk_rs[B2R_MAX_DEFS] = {}, o_pk_ep[B2R_MAX_DEFS] = {}, o_pk_ent[B2R_MAX_DEFS] = {};
    const uint64_t pk_cap = want_pk ? std::min<uint64_t>(pk->capacity, n * pk_pitch(c, c->max_chars)) : 0;   // n * pitch: every list fits
    for (uint32_t d = 0; d < c->n_defs && want_pk; d++) {
        if (pk->row_start[d]) o_pk_rs[d] = slot((n + 1) * 8, 8);
        if (pk->endpoint_counts[d]) o_pk_ep[d] = slot(n * c->packed[d].erows.size() * 8, 8);
        if (pk->row_start[d] && pk->entries[d] && pk_cap) o_pk_ent[d] = slot(pk_cap * sizeof(b2r_row_count), 8);
    }
    need = align_up(need, 256);
    int rc;
    if ((rc = c->ws_cols.reserve(need))) return rc;
    if ((rc = c->pin_small.reserve(need))) return rc;
    unsigned char* dv = (unsigned char*)c->ws_cols.p;
    unsigned char* hv = (unsigned char*)c->pin_small.p;
    auto dp = [&](void* host, size_t o) -> void* { return host ? dv + o : nullptr; };
    for (uint32_t d = 0; d < c->n_defs; d++) {
        dout.states[d] = dp(ho->states[d], o_states[d]); dout.substr_ids[d] = (uint8_t*)dp(ho->substr_ids[d], o_sid[d]);
        dout.start_enable[d] = (uint8_t*)dp(ho->start_enable[d], o_se[d]); dout.end_enable[d] = (uint8_t*)dp(ho->end_enable[d], o_ee[d]);
        dout.mult[d] = (uint64_t*)dp(ho->mult[d], o_mult[d]); dout.endpoint_mult[d] = (uint64_t*)dp(ho->endpoint_mult[d], o_em[d]);
    }
    dout.masked_chars = (uint8_t*)dp(ho->masked_chars, o_mc); dout.masked_substr_ids = (uint8_t*)dp(ho->masked_substr_ids, o_ms);
    dout.status = (b2r_string_status*)dp(ho->status, o_st); dout.records = (b2r_substr_record*)dp(ho->records, o_rec);
    dout.compact_bytes = (uint8_t*)dp(ho->compact_bytes, o_cb);
    if ((want_sm || want_pk) && !ho->status) dout.status = (b2r_string_status*)(dv + o_st_scratch);
    if (want_sm) {
        dsm.max_entries = sm->max_entries;
        for (uint32_t d = 0; d < c->n_defs; d++) {
            if (!string_mult_wanted(c, sm, d)) continue;
            dsm.entries[d] = (b2r_row_count*)dp(sm->entries[d], o_ent[d]); dsm.n_entries[d] = (uint32_t*)dp(sm->n_entries[d], o_nent[d]);
            dsm.endpoint_counts[d] = (uint32_t*)dp(sm->endpoint_counts[d], o_epc[d]);
        }
    }
    // up: offsets (rebased to the arena), bytes, and the caller's counters when they accumulate
    uint64_t* ho_offs = (uint64_t*)(hv + off_offs);
    const uint64_t shift = base & 15;                                     // keep the strings' alignment inside 16-byte vectors
    for (uint64_t j = 0; j <= n; j++) ho_offs[j] = h_offsets[j] - base + shift;
    if (nbytes) memcpy(hv + off_bytes + shift, h_bytes + base, nbytes);
    size_t up_bytes = off_bytes + shift + nbytes;
    if (acc) {
        for (const Part& p : parts) if (p.off < mult_end) memcpy(hv + p.off, p.host, p.bytes);
        up_bytes = mult_end;
    }
    w_prep = wall_us();
    CUDA_TRY(cudaMemcpyAsync(dv, hv, up_bytes, cudaMemcpyHostToDevice, st));
    for (uint32_t d = 0; d < c->n_defs; d++)
        if (dsm.entries[d]) {
            const size_t bytes = n * (size_t)sm->max_entries * sizeof(b2r_row_count);
            memcpy(hv + o_ent[d], sm->entries[d], bytes);
            CUDA_TRY(cudaMemcpyAsync(dv + o_ent[d], hv + o_ent[d], bytes, cudaMemcpyHostToDevice, st));
            up_bytes += bytes;
        }
    w_up = wall_us();
    dout.flags &= ~(uint32_t)B2R_OUT_SPARSE_D2H;                          // nothing to gain on one tile
    c->counters_copy = (BatchCounters*)(dv + off_cnt);
    rc = entry(c, dv + off_bytes, (const uint64_t*)(dv + off_offs), n, shift + nbytes, &dout, c->max_chars, st);
    c->counters_copy = nullptr;
    if (rc) return rc;
    if (want_sm) {
        void* states[B2R_MAX_DEFS] = {};
        for (uint32_t d = 0; d < c->n_defs; d++) states[d] = c->last.def[d].states;   // the caller's column or the scratch one
        if ((rc = string_mult_impl(c, dv + off_bytes, (const uint64_t*)(dv + off_offs), n, c->max_chars, states, rp, dout.status, &dsm, st, &c->last_launches))) return rc;
    }
    uint64_t pk_d2h = 0;
    if (want_pk) {
        b2r_string_mult_packed_outputs dpk{};
        dpk.capacity = pk_cap;
        void* states[B2R_MAX_DEFS] = {};
        for (uint32_t d = 0; d < c->n_defs; d++) {
            states[d] = c->last.def[d].states;
            if (pk->row_start[d]) dpk.row_start[d] = (uint64_t*)(dv + o_pk_rs[d]);
            if (pk->endpoint_counts[d]) dpk.endpoint_counts[d] = (uint32_t*)(dv + o_pk_ep[d]);
            if (o_pk_ent[d]) dpk.entries[d] = (b2r_row_count*)(hv + o_pk_ent[d]);   // mapped pinned memory: the kernel stores across PCIe
        }
        if ((rc = string_mult_packed_impl(c, dv + off_bytes, (const uint64_t*)(dv + off_offs), n, c->max_chars, states, rp, dout.status, &dpk, nullptr, st,
                                          &c->last_launches))) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(hv + off_mult, dv + off_mult, pk_begin - off_mult, cudaMemcpyDeviceToHost, st));
    for (uint32_t d = 0; d < c->n_defs && want_pk; d++) {
        if (pk->row_start[d]) { CUDA_TRY(cudaMemcpyAsync(hv + o_pk_rs[d] + 8, dv + o_pk_rs[d] + 8, n * 8, cudaMemcpyDeviceToHost, st)); pk_d2h += n * 8; }
        const size_t eb = n * c->packed[d].erows.size() * 8;
        if (pk->endpoint_counts[d]) { CUDA_TRY(cudaMemcpyAsync(hv + o_pk_ep[d], dv + o_pk_ep[d], eb, cudaMemcpyDeviceToHost, st)); pk_d2h += eb; }
    }
    w_enq = wall_us();
    CUDA_TRY(cudaStreamSynchronize(st));
    w_sync = wall_us();
    for (const Part& p : parts) memcpy(p.host, hv + p.off, p.bytes);
    for (uint32_t d = 0; d < c->n_defs && want_pk; d++) {
        if (pk->endpoint_counts[d]) memcpy(pk->endpoint_counts[d], hv + o_pk_ep[d], n * c->packed[d].erows.size() * 8);
        if (!pk->row_start[d]) continue;
        uint64_t* rs = (uint64_t*)(hv + o_pk_rs[d]);
        rs[0] = 0;
        memcpy(pk->row_start[d], rs, (n + 1) * 8);
        if (!o_pk_ent[d]) continue;
        const uint64_t stored = pk_stored(0, pk->capacity, rs + 1, n);
        if (stored) memcpy(pk->entries[d], hv + o_pk_ent[d], stored * sizeof(b2r_row_count));
        pk_d2h += stored * sizeof(b2r_row_count);
    }
    if (trace)
        fprintf(stderr, "[b2r] small batch (%llu strings): staged %.1f us, H2D issued %.1f, kernels + D2H issued %.1f, device done %.1f, copied out %.1f\n", (unsigned long long)n, w_prep,
                w_up, w_enq, w_sync, wall_us());
    c->last_h2d_bytes = up_bytes; c->last_d2h_bytes = pk_begin - off_mult + pk_d2h;
    const BatchCounters* hc = (const BatchCounters*)(hv + off_cnt);
    b2r_batch_status r;
    memset(&r, 0, sizeof r);
    if (hc->any_bad()) {
        rc = launch_diagnose(c->last, hc->first_bad(), c->d_batch_status, st);
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync(&r, c->d_batch_status, sizeof r, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        report_failure(r);
    }
    r.n_overlap_lo = (uint32_t)hc->n_overlap;
    if (result) *result = r;
    return r.code;
}

// ---- the sliced pipeline -------------------------------------------------------------------------------------------------------
// What a host entry point runs on the device: `run` enqueues the kernels of one slice, and `by_bytes` selects the slicing that goes
// with them (see `cuts` below) — the only other difference between b2r_match_batch_host and b2r_match_batch_chunked_host.
struct DeviceEntry {
    BatchEntry run;
    bool by_bytes;                     // slices balanced by bytes at multiples of 4 strings (else by count, at multiples of 32)
};
const DeviceEntry BATCH_ENTRY = {match_batch_impl, false}, CHUNKED_ENTRY = {match_batch_chunked_impl, true};

int host_batch(b2r_config* c, const DeviceEntry& entry, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho, b2r_batch_status* result,
               const MultiHook* hook, const b2r_string_mult_outputs* sm = nullptr, const b2r_string_mult_packed_outputs* pk = nullptr) {
    PkPublishOnExit publish_on_exit{hook};
    if (!c || !ho || (n && !h_offsets)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    int rc = check_outputs(c, ho, false);  // same pitches are used on the device; host pointer alignment is irrelevant
    if (rc) return rc;
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    cudaStream_t st = c->host_stream;
    const uint64_t total = n ? h_offsets[n] : 0;
    const uint64_t base = n ? h_offsets[0] : 0;
    // every offset is checked before anything is enqueued: the kernels read bytes[offsets[j] .. offsets[j+1]) of the staging buffer
    {
        uint64_t bad = 0;                                                 // branch-free first pass (vectorisable), the index only if something is wrong
        for (uint64_t j = 0; j < n; j++) bad |= (uint64_t)(h_offsets[j + 1] < h_offsets[j]);
        if (bad)
            for (uint64_t j = 0; j < n; j++)
                if (h_offsets[j + 1] < h_offsets[j]) { set_error("offsets must be non-decreasing (string %llu)", (unsigned long long)j); return B2R_ERR_INVALID_ARG; }
    }
    const uint64_t nbytes = total - base;
    const uint64_t rp = ho->row_pitch, bp = ho->bitmap_pitch;
    if (!hook && c->opt.small_path && n >= 1 && n <= 32 && n * (rp * (4 + 3 * c->n_defs) + 2 * bp * c->n_defs) + nbytes <= (8u << 20))
        return host_batch_small(c, entry.run, h_bytes, h_offsets, n, ho, sm, pk, result);

    if ((rc = c->ws_bytes.reserve(align_up(nbytes + 16, 256)))) return rc;
    if ((rc = c->ws_offsets.reserve((n + 1) * 8))) return rc;
    const bool sparse = (ho->flags & B2R_OUT_SPARSE_D2H) != 0 && n > 0;
    // device columns, same layout as the host ones
    size_t need = 0;
    auto slot = [&](size_t bytes, size_t align = 256) { need = align_up(need, align); size_t o = need; need += bytes; return o; };
    // stride: bytes per string (0: not per string).  pinned: page-locked destination, the copy is asynchronous; a copy into
    // pageable memory blocks the calling thread until everything queued before it on its stream is done, so those are
    // issued after the last slice instead of inside the pipeline (they would serialise the H2D of slice i+1 behind the
    // D2H of slice i: measured 110 ms instead of 92 ms per 2^20-string batch with three small pageable columns).
    struct Copy { size_t off; void* host; size_t bytes; size_t stride; bool pinned; bool sparse; };
    std::vector<Copy> copies;
    b2r_outputs dout = *ho;
    dout.flags &= ~(uint32_t)B2R_OUT_SPARSE_D2H;
    // the multiplicity counters of every def form one block (a single all-reduce on a multi-device handle)
    size_t off_mult[B2R_MAX_DEFS], off_em[B2R_MAX_DEFS];
    const size_t mult_begin = slot(0);
    const bool copy_mult = !hook || hook->first;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        off_mult[d] = (ho->mult[d] || hook) ? slot(c->packed[d].rows.size() * 8, 8) : 0;
        off_em[d] = (ho->endpoint_mult[d] || hook) ? slot(c->packed[d].erows.size() * 16, 8) : 0;
    }
    const size_t mult_end = need;
    size_t off_states[B2R_MAX_DEFS], off_sid[B2R_MAX_DEFS], off_se[B2R_MAX_DEFS], off_ee[B2R_MAX_DEFS];
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const size_t w = c->packed[d].state_width;
        off_states[d] = ho->states[d] ? slot(n * rp * w) : 0;
        off_sid[d] = ho->substr_ids[d] ? slot(n * rp) : 0;
        off_se[d] = ho->start_enable[d] ? slot(n * bp) : 0;
        off_ee[d] = ho->end_enable[d] ? slot(n * bp) : 0;
    }
    const size_t off_mc = ho->masked_chars ? slot(n * rp) : 0, off_ms = ho->masked_substr_ids ? slot(n * rp) : 0;
    const size_t off_st = ho->status ? slot(n * sizeof(b2r_string_status)) : 0;
    const size_t off_rec = ho->records ? slot(n * (size_t)ho->max_records * sizeof(b2r_substr_record)) : 0;
    const size_t off_cb = ho->compact_bytes ? slot(n * (size_t)ho->compact_pitch) : 0;
    // per-string counts (b2r_match_batch_host_mult): copied back per slice like the status
    bool want_sm = false;
    size_t off_ent[B2R_MAX_DEFS] = {}, off_nent[B2R_MAX_DEFS] = {}, off_epc[B2R_MAX_DEFS] = {};
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!string_mult_wanted(c, sm, d)) continue;
        want_sm = true;
        off_ent[d] = sm->entries[d] ? slot(n * (size_t)sm->max_entries * sizeof(b2r_row_count)) : 0;
        off_nent[d] = sm->n_entries[d] ? slot(n * 4) : 0;
        off_epc[d] = sm->endpoint_counts[d] ? slot(n * c->packed[d].erows.size() * 8) : 0;
    }
    // packed per-string counts (b2r_match_batch_host_mult_packed): the endpoint counts are copied back per slice like the status;
    // each slice packs its lists into its own staging area (lo * pitch on) with row_start relative to the slice (at lo + i)
    bool want_pk = false;
    for (uint32_t d = 0; d < c->n_defs; d++) want_pk = want_pk || string_mult_packed_wanted(c, pk, d);
    const uint64_t pkw = want_pk ? pk_pitch(c, c->max_chars) : 0;
    size_t off_pk_ep[B2R_MAX_DEFS] = {}, off_pk_rs[B2R_MAX_DEFS] = {}, off_pk_ent[B2R_MAX_DEFS] = {};
    for (uint32_t d = 0; d < c->n_defs && want_pk; d++) {
        off_pk_ep[d] = pk->endpoint_counts[d] ? slot(n * c->packed[d].erows.size() * 8) : 0;
        off_pk_rs[d] = pk->row_start[d] ? slot((n + b2r_config::MAX_SLICES + 1) * 8) : 0;
        off_pk_ent[d] = pk->row_start[d] && pk->entries[d] && pk->capacity ? slot(n * pkw * sizeof(b2r_row_count)) : 0;
    }
    const size_t off_st_scratch = (want_sm || want_pk) && !ho->status ? slot(n * sizeof(b2r_string_status)) : 0;   // the post-pass reads the status
    if ((rc = c->ws_cols.reserve(need + 256))) return rc;
    unsigned char* cb = (unsigned char*)c->ws_cols.p;
    auto bind = [&](void* host, size_t off, size_t bytes, size_t stride = 0, bool sp = false) -> void* {
        if (!host) return nullptr;
        copies.push_back({off, host, bytes, stride, is_pinned(host), sp && sparse});
        return cb + off;
    };
    const bool acc = (ho->flags & B2R_OUT_ACCUMULATE_MULT) != 0;
    if (hook && mult_end > mult_begin) CUDA_TRY(cudaMemsetAsync(cb + mult_begin, 0, mult_end - mult_begin, st));   // every slice accumulates into the block
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const size_t w = c->packed[d].state_width;
        dout.states[d] = bind(ho->states[d], off_states[d], n * rp * w, rp * w);
        dout.substr_ids[d] = (uint8_t*)bind(ho->substr_ids[d], off_sid[d], n * rp, rp, true);
        dout.start_enable[d] = (uint8_t*)bind(ho->start_enable[d], off_se[d], n * bp, bp, true);
        dout.end_enable[d] = (uint8_t*)bind(ho->end_enable[d], off_ee[d], n * bp, bp, true);
        if (hook) {   // every device produces every counter; the block is reduced below
            dout.mult[d] = (uint64_t*)(cb + off_mult[d]); dout.endpoint_mult[d] = (uint64_t*)(cb + off_em[d]);
            if (copy_mult && ho->mult[d]) copies.push_back({off_mult[d], ho->mult[d], c->packed[d].rows.size() * 8, 0, false, false});
            if (copy_mult && ho->endpoint_mult[d]) copies.push_back({off_em[d], ho->endpoint_mult[d], c->packed[d].erows.size() * 16, 0, false, false});
        } else {
            dout.mult[d] = (uint64_t*)bind(ho->mult[d], off_mult[d], c->packed[d].rows.size() * 8);
            dout.endpoint_mult[d] = (uint64_t*)bind(ho->endpoint_mult[d], off_em[d], c->packed[d].erows.size() * 16);
        }
        if (acc && copy_mult) {
            if (ho->mult[d]) CUDA_TRY(cudaMemcpyAsync(dout.mult[d], ho->mult[d], c->packed[d].rows.size() * 8, cudaMemcpyHostToDevice, st));
            if (ho->endpoint_mult[d]) CUDA_TRY(cudaMemcpyAsync(dout.endpoint_mult[d], ho->endpoint_mult[d], c->packed[d].erows.size() * 16, cudaMemcpyHostToDevice, st));
        }
    }
    dout.masked_chars = (uint8_t*)bind(ho->masked_chars, off_mc, n * rp, rp, true);
    dout.masked_substr_ids = (uint8_t*)bind(ho->masked_substr_ids, off_ms, n * rp, rp, true);
    dout.status = (b2r_string_status*)bind(ho->status, off_st, n * sizeof(b2r_string_status), sizeof(b2r_string_status));
    dout.records = (b2r_substr_record*)bind(ho->records, off_rec, n * (size_t)ho->max_records * sizeof(b2r_substr_record), (size_t)ho->max_records * sizeof(b2r_substr_record));
    dout.compact_bytes = (uint8_t*)bind(ho->compact_bytes, off_cb, n * (size_t)ho->compact_pitch, (size_t)ho->compact_pitch);
    b2r_string_mult_outputs dsm{};
    if ((want_sm || want_pk) && !ho->status) dout.status = (b2r_string_status*)(cb + off_st_scratch);
    b2r_string_mult_packed_outputs dpk{};
    for (uint32_t d = 0; d < c->n_defs && want_pk; d++) {
        const size_t ps = c->packed[d].erows.size() * 8;
        dpk.endpoint_counts[d] = (uint32_t*)bind(pk->endpoint_counts[d], off_pk_ep[d], n * ps, ps);
        if (pk->row_start[d]) dpk.row_start[d] = (uint64_t*)(cb + off_pk_rs[d]);
        if (off_pk_ent[d]) dpk.entries[d] = (b2r_row_count*)(cb + off_pk_ent[d]);
    }
    if (want_sm) {
        dsm.max_entries = sm->max_entries;
        for (uint32_t d = 0; d < c->n_defs; d++) {
            const size_t es = (size_t)sm->max_entries * sizeof(b2r_row_count), ps = c->packed[d].erows.size() * 8;
            dsm.entries[d] = (b2r_row_count*)bind(sm->entries[d], off_ent[d], n * es, es);
            dsm.n_entries[d] = (uint32_t*)bind(sm->n_entries[d], off_nent[d], n * 4, 4);
            dsm.endpoint_counts[d] = (uint32_t*)bind(sm->endpoint_counts[d], off_epc[d], n * ps, ps);
        }
    }

    // The batch is cut into slices of strings: the H2D copy of slice i+1 and the D2H copy of slice i-1 run on their own
    // streams while the kernels of slice i run (PCIe is full duplex; the copies are the end-to-end bottleneck).
    // inputs: keep the caller's offsets (the kernel adds them to the base pointer, so shift the base instead):
    // d_bytes + offsets[j] must address string j: d_bytes = ws + (base & 15) - base  (16-byte aligned by construction)
    unsigned char* const d_in = (unsigned char*)c->ws_bytes.p + (base & 15);
    const uint8_t* d_bytes = d_in - base;
    const uint64_t* d_offsets = (const uint64_t*)c->ws_offsets.p;
    const bool chunked = entry.by_bytes;
    const bool forced = c->opt.slices >= 1 && c->opt.slices <= b2r_config::MAX_SLICES;   // testing hook
    std::vector<uint64_t> cuts;                                           // slice i: strings [cuts[i], cuts[i + 1])
    int n_slices;
    if (!chunked) {
        n_slices = n >= 16384 ? (n >= (1u << 19) ? 16 : 8) : 1;
        if (forced && n >= 16384) n_slices = c->opt.slices;
        // slice boundaries are multiples of 32 strings: whole tiles per slice, and lo * pitch keeps the 16-byte alignment of every
        // column for any legal pitch (bitmap_pitch is only a multiple of 4)   (small first slices were tried: no gain)
        for (int k = 0; k <= n_slices; k++) cuts.push_back(k >= n_slices ? n : (n * (uint64_t)k / n_slices) & ~uint64_t(31));
    } else {
        // Few long strings: slices balanced by BYTES, so that a batch of a few hundred strings overlaps H2D, kernels and D2H too.
        // A slice holds at least 8 MiB of input (about 0.2 ms of H2D and several times that of D2H at PCIe 5 x16 rates, against
        // some 20 launches of fixed cost per slice) and at least 32 strings (the emit stage gives a warp 32 strings), 16 at most.
        n_slices = (int)std::max<uint64_t>(1, std::min<uint64_t>({(uint64_t)b2r_config::MAX_SLICES, nbytes >> 23, n / 32}));
        if (forced) n_slices = c->opt.slices;
        // Boundaries are multiples of 4 strings.  lo * bitmap_pitch is then a multiple of 16 (bitmap_pitch % 4 == 0), lo * row_pitch
        // too (row_pitch % 16 == 0): every column slice keeps the 16-byte alignment check_outputs asks for and the emit stage's
        // TMA zero-fill needs.  Nothing else depends on the slice base: every store of the emit stage (emit.cuh) stays inside the
        // rows, records, status and compact area of its own string, and its whole-sector stores are chosen at run time from the
        // actual address (bitmap words, status) or only pad a string's own area (records, compact bytes) — so no store reaches a
        // neighbouring slice whose columns may be on their way to the host already.
        cuts.push_back(0);
        for (int k = 1; k < n_slices; k++) {
            const uint64_t target = base + nbytes / n_slices * k + nbytes % n_slices * k / n_slices;
            const uint64_t j = (uint64_t)(std::lower_bound(h_offsets, h_offsets + n + 1, target) - h_offsets);
            cuts.push_back(std::max(cuts.back(), std::min(n, (j + 2) & ~uint64_t(3))));
        }
        cuts.push_back(n);
        cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());    // no empty slices (a forced count larger than the batch)
        if (cuts.size() < 2) cuts.push_back(n);
        n_slices = (int)cuts.size() - 1;
        // the workspaces of every slice, sized for the largest one before anything is enqueued (a buffer that grows between two
        // slices would be freed under the kernels of the previous one)
        uint64_t widest = 0;
        for (int i = 0; i < n_slices; i++) widest = std::max(widest, cuts[i + 1] - cuts[i]);
        if ((rc = chunked_reserve(c, widest, &dout, c->max_chars))) return rc;
    }
    auto cut = [&](int k) { return cuts[k]; };
    // packed counts: the post-pass workspaces, sized for the widest slice before anything is enqueued; pinned: the totals the scan
    // kernel publishes per slice and def, then per def the slice-relative row_start values that come back
    uint64_t* pk_tot = nullptr;
    uint64_t* pk_rel[B2R_MAX_DEFS] = {};
    if (want_pk) {
        uint64_t widest = 0;
        for (int i = 0; i < n_slices; i++) widest = std::max(widest, cut(i + 1) - cut(i));
        b2r_string_mult_packed_outputs shape = dpk;
        shape.capacity = widest * pkw;
        if ((rc = string_mult_packed_reserve(c, widest, c->max_chars, &shape))) return rc;
        if ((rc = c->pin_pk.reserve(((size_t)b2r_config::MAX_SLICES * B2R_MAX_DEFS + (size_t)c->n_defs * (n + 1)) * 8))) return rc;
        pk_tot = (uint64_t*)c->pin_pk.p;
        for (uint32_t d = 0; d < c->n_defs; d++) pk_rel[d] = pk_tot + b2r_config::MAX_SLICES * B2R_MAX_DEFS + d * (n + 1);
    }

    // ---- sparse mode: compaction arenas (device + pinned mirror) and the host threads ---------------------------------------------
    std::vector<const Copy*> scols;
    for (const Copy& cp : copies) if (cp.sparse) scols.push_back(&cp);
    const size_t n_sc = scols.size();
    struct SliceCol { size_t idx_off, pay_off; uint32_t cap; uint64_t n_sectors, bytes; };
    std::vector<SliceCol> sc(n_sc * n_slices);
    size_t sp_need = 0, cnt_off = 0;
    bool reuse = false;
    int arena = 0;
    if (sparse && n_sc) {
        auto sslot = [&](size_t bytes) { sp_need = align_up(sp_need, 256); size_t o = sp_need; sp_need += bytes; return o; };
        cnt_off = sslot(n_sc * n_slices * sizeof(unsigned int));
        for (int i = 0; i < n_slices; i++) {
            const uint64_t ni = cut(i + 1) - cut(i);
            for (size_t k = 0; k < n_sc; k++) {
                SliceCol& s = sc[i * n_sc + k];
                s.bytes = ni * scols[k]->stride;
                s.n_sectors = (s.bytes + 31) / 32;
                if (s.n_sectors > 0xFFFFFFFFull) { set_error("sparse D2H: a slice of more than 2^32 sectors"); return B2R_ERR_UNSUPPORTED; }
                // a sector or two per string, column and KiB of row (rows of about 1 KiB on the batch path); more -> dense copy
                const uint64_t per_string = chunked ? 2 * ((rp + 1023) / 1024) : 2;
                s.cap = (uint32_t)std::min<uint64_t>(s.n_sectors, per_string * ni + 1024);
                if (c->opt.sparse_cap > 0) s.cap = (uint32_t)std::min<uint64_t>(s.n_sectors, (uint64_t)c->opt.sparse_cap);
                s.idx_off = sslot((size_t)s.cap * 4);
                s.pay_off = sslot((size_t)s.cap * 32);
            }
        }
        // the compacted sectors are written by the kernel straight into page-locked host memory (stores over PCIe, no copy to size
        // and issue); two arenas alternate so that the index lists of the previous call survive until they have been used
        arena = c->sparse_memo.arena ^ 1;
        if ((rc = c->ws_sparse.reserve(n_sc * n_slices * sizeof(unsigned int) + 256))) return rc;
        if ((rc = c->pin_sparse[arena].reserve(sp_need + 256))) return rc;
        if (!c->opt.sparse_direct && (rc = c->ws_sparse_arena.reserve(sp_need + 256))) return rc;
        if (!c->pool) c->pool.reset(new HostPool(c->opt.host_threads > 0 ? (unsigned)c->opt.host_threads : default_host_threads()));
        CUDA_TRY(cudaMemsetAsync(c->ws_sparse.p, 0, n_sc * n_slices * sizeof(unsigned int), st));
        // B2R_OUT_SPARSE_REUSE: these are the buffers the previous call filled (same strings per buffer and pitches): only the sectors
        // it scattered are non-zero, and their index lists are still in the pinned arena, where the memo says (its slices need not be
        // this call's: the chunked pipeline cuts by bytes)
        SparseMemo& memo = c->sparse_memo;
        reuse = (ho->flags & B2R_OUT_SPARSE_REUSE) && memo.valid && memo.n == n && memo.rp == rp && memo.bp == bp &&
                memo.sparse_cap == c->opt.sparse_cap && memo.hosts.size() == n_sc && c->pin_sparse[memo.arena].p;
        for (size_t k = 0; reuse && k < n_sc; k++) reuse = memo.hosts[k] == scols[k]->host;
        memo.valid = false;                                               // until this call has completed
        if (reuse && (c->opt.host_debug & 1)) {
        } else if (reuse) {
            const uint32_t piece = 1u << 16;
            for (int i = 0; i < memo.n_slices; i++)
                for (size_t k = 0; k < n_sc; k++) {
                    unsigned char* dst = (unsigned char*)scols[k]->host + memo.cuts[i] * scols[k]->stride;
                    const uint64_t bytes = (memo.cuts[i + 1] - memo.cuts[i]) * scols[k]->stride;
                    if (memo.dense[i * n_sc + k]) { c->pool->submit([dst, bytes] { memset(dst, 0, bytes); }); continue; }
                    const uint32_t cnt = memo.cnt[i * n_sc + k];
                    const uint32_t* idx = (const uint32_t*)((unsigned char*)c->pin_sparse[memo.arena].p + memo.idx_off[i * n_sc + k]);
                    for (uint32_t e0 = 0; e0 < cnt; e0 += piece)
                        c->pool->submit([=] {
                            const uint32_t e1 = std::min(cnt, e0 + piece);
                            for (uint32_t e = e0; e < e1; e++) {   // one cache miss per sector: a dozen in flight towards L1, more towards L2
                                if (e + 48 < e1) __builtin_prefetch(dst + (uint64_t)idx[e + 48] * 32, 0, 1);
                                if (e + 12 < e1) __builtin_prefetch(dst + (uint64_t)idx[e + 12] * 32, 1, 0);
                                const uint64_t o = (uint64_t)idx[e] * 32;
                                memset(dst + o, 0, (size_t)std::min<uint64_t>(32, bytes - o));
                            }
                        });
                }
        } else {
            // the zeros of the caller's dense columns are written here, by the host, while the GPU works
            for (size_t k = 0; k < n_sc; k++) {
                unsigned char* h = (unsigned char*)scols[k]->host;
                const size_t bytes = scols[k]->bytes, piece = 4u << 20;
                for (size_t o = 0; o < bytes; o += piece) c->pool->submit([h, o, bytes, piece] { memset(h + o, 0, std::min(piece, bytes - o)); });
            }
        }
    }
    unsigned int* const d_cnt = (unsigned int*)c->ws_sparse.p;
    unsigned char* const sp_host = (unsigned char*)c->pin_sparse[arena].p;   // unified addressing: the kernels write through the same pointer
    // where sparsify_kernel writes.  Direct mode: pinned host memory, i.e. one PCIe write per 4-byte index and per 32-byte sector
    // (a transaction header for every 32 bytes: 0.25 GB of sectors occupied the link like 0.6 GB).  Staged mode (default): a device
    // arena of the same layout; the host learns the count (published below), then exact-size copies bring index list and sectors over
    const bool staged = sparse && n_sc && !c->opt.sparse_direct;
    unsigned char* const sp_dev = staged ? (unsigned char*)c->ws_sparse_arena.p : sp_host;

    const bool trace = c->opt.trace_host;                                 // timing aid: where the copies sit on the time line
    const auto wall0 = std::chrono::steady_clock::now();
    auto wall_ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count(); };
    double w_enq = 0, w_pay = 0, w_zero = 0, w_scat = 0;
    cudaEvent_t tev[4] = {};
    if (trace) for (auto& e : tev) CUDA_TRY(cudaEventCreate(&e));
    if (trace) CUDA_TRY(cudaEventRecord(tev[0], st));
    CUDA_TRY(cudaEventRecord(c->ev_fork, st));                           // accumulate uploads / earlier work on the compute stream
    CUDA_TRY(cudaStreamWaitEvent(c->in_stream, c->ev_fork, 0));
    CUDA_TRY(cudaStreamWaitEvent(c->out_stream, c->ev_fork, 0));
    uint64_t h2d = 0, d2h = 0;
    if (n) { CUDA_TRY(cudaMemcpyAsync(c->ws_offsets.p, h_offsets, (n + 1) * 8, cudaMemcpyHostToDevice, c->in_stream)); h2d += (n + 1) * 8; }
    std::vector<WalkParams> slice_params(n_slices);
    uint32_t launches = 0;                                                // every kernel of the call, slices and sparse mode
    std::vector<uint64_t> slice_lo(n_slices);
    int n_sm = 148, max_smem = 0;
    device_limits(&n_sm, &max_smem);
    for (int i = 0; i < n_slices; i++) {
        const uint64_t lo = cut(i), hi = cut(i + 1), ni = hi - lo;
        slice_lo[i] = lo;
        const uint64_t b0 = n ? h_offsets[lo] : 0, b1 = n ? h_offsets[hi] : 0;
        if (b1 > b0) { CUDA_TRY(cudaMemcpyAsync(d_in + (b0 - base), h_bytes + b0, b1 - b0, cudaMemcpyHostToDevice, c->in_stream)); h2d += b1 - b0; }
        for (uint32_t d = 0; d < c->n_defs && ni; d++)                  // entry slots the post-pass does not write keep the caller's values
            if (dsm.entries[d]) {
                const size_t es = (size_t)sm->max_entries * sizeof(b2r_row_count);
                CUDA_TRY(cudaMemcpyAsync((unsigned char*)dsm.entries[d] + lo * es, (const unsigned char*)sm->entries[d] + lo * es, ni * es, cudaMemcpyHostToDevice, c->in_stream));
                h2d += ni * es;
            }
        CUDA_TRY(cudaEventRecord(c->ev_in[i], c->in_stream));
        CUDA_TRY(cudaStreamWaitEvent(st, c->ev_in[i], 0));
        b2r_outputs ds = dout;                                           // this slice's rows of every column
        for (uint32_t d = 0; d < c->n_defs; d++) {
            const size_t w = c->packed[d].state_width;
            if (ds.states[d]) ds.states[d] = (unsigned char*)ds.states[d] + lo * rp * w;
            if (ds.substr_ids[d]) ds.substr_ids[d] += lo * rp;
            if (ds.start_enable[d]) ds.start_enable[d] += lo * bp;
            if (ds.end_enable[d]) ds.end_enable[d] += lo * bp;
        }
        if (ds.masked_chars) ds.masked_chars += lo * rp;
        if (ds.masked_substr_ids) ds.masked_substr_ids += lo * rp;
        if (ds.status) ds.status += lo;
        if (ds.records) ds.records += lo * (size_t)ho->max_records;
        if (ds.compact_bytes) ds.compact_bytes += lo * (size_t)ho->compact_pitch;
        if (i > 0 || hook) ds.flags |= B2R_OUT_ACCUMULATE_MULT;          // the multiplicities of the slices add up
        if (entry.by_bytes && ni) {
            // the slice's sparse columns are zeroed by memsets over the whole GPU: emit_kernel would zero them from the warps that
            // own their tiles, and a slice of a few hundred long strings has only a few tiles (2048 x 64 KiB in 16 slices, sparse
            // D2H, B200: 16.5 ms per call with the emit stage's fill, 10.0 ms with the memsets)
            auto zero = [&](void* p, size_t pitch) { return p ? cudaMemsetAsync(p, 0, ni * pitch, st) : cudaSuccess; };
            for (uint32_t d = 0; d < c->n_defs; d++) {
                CUDA_TRY(zero(ds.substr_ids[d], rp)); CUDA_TRY(zero(ds.start_enable[d], bp)); CUDA_TRY(zero(ds.end_enable[d], bp));
            }
            CUDA_TRY(zero(ds.masked_chars, rp)); CUDA_TRY(zero(ds.masked_substr_ids, rp));
            c->sparse_zeroed = true;
        }
        c->counters_copy = c->h_slices + i;                              // finalize_kernel leaves the slice's counters in pinned host memory
        rc = entry.run(c, d_bytes, d_offsets + lo, ni, total, &ds, c->max_chars, st);
        c->counters_copy = nullptr;
        c->sparse_zeroed = false;
        if (rc) return rc;
        if (want_sm && ni) {
            b2r_string_mult_outputs s = dsm;
            void* states[B2R_MAX_DEFS] = {};
            for (uint32_t d = 0; d < c->n_defs; d++) {
                states[d] = c->last.def[d].states;                       // the caller's column or the scratch one, this slice's rows
                if (s.entries[d]) s.entries[d] += lo * sm->max_entries;
                if (s.n_entries[d]) s.n_entries[d] += lo;
                if (s.endpoint_counts[d]) s.endpoint_counts[d] += lo * 2 * c->packed[d].erows.size();
            }
            if ((rc = string_mult_impl(c, d_bytes, d_offsets + lo, ni, c->max_chars, states, rp, ds.status, &s, st, &c->last_launches))) return rc;
        }
        if (want_pk && ni) {
            b2r_string_mult_packed_outputs s{};
            s.capacity = ni * pkw;                                        // the slice's staging holds every list: the caller's capacity is applied below
            void* states[B2R_MAX_DEFS] = {};
            for (uint32_t d = 0; d < c->n_defs; d++) {
                states[d] = c->last.def[d].states;
                if (dpk.row_start[d]) s.row_start[d] = dpk.row_start[d] + lo + i;
                if (dpk.entries[d]) s.entries[d] = dpk.entries[d] + lo * pkw;
                if (dpk.endpoint_counts[d]) s.endpoint_counts[d] = dpk.endpoint_counts[d] + lo * 2 * c->packed[d].erows.size();
            }
            if ((rc = string_mult_packed_impl(c, d_bytes, d_offsets + lo, ni, c->max_chars, states, rp, ds.status, &s, pk_tot + i * B2R_MAX_DEFS, st,
                                              &c->last_launches))) return rc;
        }
        slice_params[i] = c->last;
        launches += c->last_launches;
        if (sparse && ni)
            for (size_t k = 0; k < n_sc; k++) {
                const SliceCol& s = sc[i * n_sc + k];
                const unsigned grid = (unsigned)std::min<uint64_t>((s.n_sectors + 256 * SPARSIFY_K - 1) / (256 * SPARSIFY_K), (uint64_t)n_sm * 8);
                sparsify_kernel<<<grid, 256, 0, st>>>((const uint4*)(cb + scols[k]->off + lo * scols[k]->stride), s.n_sectors, (uint32_t*)(sp_dev + s.idx_off),
                                                      (uint4*)(sp_dev + s.pay_off), s.cap, d_cnt + i * n_sc + k);
                CUDA_TRY(cudaGetLastError());
                launches++;
            }
        if (sparse && n_sc) {
            publish_counts_kernel<<<1, 32, 0, st>>>(d_cnt + i * n_sc, (unsigned int*)(sp_host + cnt_off) + i * n_sc, (uint32_t)n_sc);
            CUDA_TRY(cudaGetLastError());
            launches++;
        }
        CUDA_TRY(cudaEventRecord(c->ev_done[i], st));
        if (trace && i == n_slices - 1) CUDA_TRY(cudaEventRecord(tev[1], c->in_stream));
        // staged sparse mode: the D2H copies of a slice are issued further down, by the loop that has waited for its kernels — the
        // copy engine serves copies in the order they were issued, and the (small) compacted sectors of slice i have to go in FRONT of
        // the state column of slice i, not behind the state columns of every slice (the host threads scatter while the big copies run)
        if (staged) continue;
        CUDA_TRY(cudaStreamWaitEvent(c->out_stream, c->ev_done[i], 0));
        if (trace && i == 0) CUDA_TRY(cudaEventRecord(tev[2], c->out_stream));
        for (const Copy& cp : copies)
            if (cp.stride && cp.pinned && !cp.sparse && ni) {
                CUDA_TRY(cudaMemcpyAsync((unsigned char*)cp.host + lo * cp.stride, cb + cp.off + lo * cp.stride, ni * cp.stride, cudaMemcpyDeviceToHost, c->out_stream));
                d2h += ni * cp.stride;
            }
    }
    w_enq = wall_ms();
    // multi-device handle: the one exchange of the path, NVLink all-reduce of the multiplicity block (SURVEY 8(e))
    if (hook && mult_end > mult_begin) {
        const ncclResult_t nr = hook->all_reduce(cb + mult_begin, cb + mult_begin, (mult_end - mult_begin) / 8, ncclUint64, ncclSum, hook->comm, st);
        if (nr != ncclSuccess) { set_error("ncclAllReduce failed: %s", hook->error_string(nr)); return B2R_ERR_CUDA; }
    }
    // ---- sparse mode: the compacted sectors of slice i are in host memory when ev_done[i] fires; host threads scatter them -----------
    if (sparse && n_sc) {
        const unsigned int* h_cnt = (const unsigned int*)(sp_host + cnt_off);
        std::vector<char> dense(n_sc * n_slices, 0);
        w_pay = wall_ms();
        bool cleared = false;
        bool any_dense = false;
        // the scatter jobs of slice i: its compacted sectors are in the pinned arena (staged mode: once ev_pay[i] has fired)
        auto scatter_slice = [&](int i) {
            // every zero is in place first (reused buffers: the old sectors are cleared): a clear and a scatter may hit the same sector
            if (!cleared) { c->pool->wait(); w_zero = wall_ms(); cleared = true; }
            const uint64_t lo = slice_lo[i], ni = cut(i + 1) - lo;
            if (c->opt.host_debug & 2) return;
            for (size_t k = 0; k < n_sc && ni; k++) {
                const SliceCol& s = sc[i * n_sc + k];
                const uint32_t cnt = h_cnt[i * n_sc + k];
                if (!cnt || dense[i * n_sc + k]) continue;
                unsigned char* dst = (unsigned char*)scols[k]->host + lo * scols[k]->stride;
                const uint32_t* idx = (const uint32_t*)(sp_host + s.idx_off);
                const unsigned char* pay = sp_host + s.pay_off;
                const uint64_t bytes = s.bytes;
                const uint32_t piece = 1u << 15;
                for (uint32_t e0 = 0; e0 < cnt; e0 += piece)
                    c->pool->submit([=] {
                        const uint32_t e1 = std::min(cnt, e0 + piece);
                        for (uint32_t e = e0; e < e1; e++) {
                            if (e + 48 < e1) __builtin_prefetch(dst + (uint64_t)idx[e + 48] * 32, 0, 1);
                            if (e + 12 < e1) __builtin_prefetch(dst + (uint64_t)idx[e + 12] * 32, 1, 0);
                            const uint64_t o = (uint64_t)idx[e] * 32;
                            memcpy(dst + o, pay + (size_t)e * 32, (size_t)std::min<uint64_t>(32, bytes - o));
                        }
                    });
            }
        };
        for (int i = 0; i < n_slices; i++) {
            const uint64_t lo = slice_lo[i], ni = cut(i + 1) - lo;
            CUDA_TRY(cudaEventSynchronize(c->ev_done[i]));
            if (trace) fprintf(stderr, "[b2r]   slice %2d: kernels done %.2f ms", i, wall_ms());
            d2h += n_sc * 4;
            // the host has waited for the slice's kernels, so its copies need no event; staged mode: everything on out_stream, in the
            // order payload -> ev_pay -> dense columns; direct mode: only a dense fallback is copied (pay_stream)
            cudaStream_t ps = staged ? c->out_stream : c->pay_stream;
            bool waited = staged;
            auto pay_wait = [&]() -> int { if (!waited) { CUDA_TRY(cudaStreamWaitEvent(ps, c->ev_done[i], 0)); waited = true; } return 0; };
            if (staged && trace && i == 0) CUDA_TRY(cudaEventRecord(tev[2], c->out_stream));
            for (size_t k = 0; k < n_sc && ni; k++) {
                const SliceCol& s = sc[i * n_sc + k];
                const uint32_t cnt = h_cnt[i * n_sc + k];
                unsigned char* dst = (unsigned char*)scols[k]->host + lo * scols[k]->stride;
                if (cnt > s.cap) {   // not sparse after all: this column slice crosses densely
                    dense[i * n_sc + k] = 1;
                    if ((rc = pay_wait())) return rc;
                    any_dense = true;
                    CUDA_TRY(cudaMemcpyAsync(dst, cb + scols[k]->off + lo * scols[k]->stride, s.bytes, cudaMemcpyDeviceToHost, ps));
                    d2h += s.bytes;
                    continue;
                }
                if (!cnt) continue;
                d2h += (size_t)cnt * 36;
                if (staged) {
                    CUDA_TRY(cudaMemcpyAsync(sp_host + s.idx_off, sp_dev + s.idx_off, (size_t)cnt * 4, cudaMemcpyDeviceToHost, ps));
                    CUDA_TRY(cudaMemcpyAsync(sp_host + s.pay_off, sp_dev + s.pay_off, (size_t)cnt * 32, cudaMemcpyDeviceToHost, ps));
                }
            }
            if (staged) {   // scatter one slice behind the copies
                CUDA_TRY(cudaEventRecord(c->ev_pay[i], ps));
                for (const Copy& cp : copies)
                    if (cp.stride && cp.pinned && !cp.sparse && ni) {
                        CUDA_TRY(cudaMemcpyAsync((unsigned char*)cp.host + lo * cp.stride, cb + cp.off + lo * cp.stride, ni * cp.stride, cudaMemcpyDeviceToHost, ps));
                        d2h += ni * cp.stride;
                    }
                if (i > 0) { CUDA_TRY(cudaEventSynchronize(c->ev_pay[i - 1])); scatter_slice(i - 1); }
            } else scatter_slice(i);
            if (trace) fprintf(stderr, ", sectors of slice %d in host memory %.2f ms, scatter jobs pending %u\n", i - 1, wall_ms(), c->pool->pending());
        }
        if (staged) { CUDA_TRY(cudaEventSynchronize(c->ev_pay[n_slices - 1])); scatter_slice(n_slices - 1); }
        if (any_dense && !staged) CUDA_TRY(cudaStreamSynchronize(c->pay_stream));
        c->pool->wait();
        w_scat = wall_ms();
        SparseMemo& memo = c->sparse_memo;                                // what the next B2R_OUT_SPARSE_REUSE call has to clear
        memo.n = n; memo.rp = rp; memo.bp = bp; memo.n_slices = n_slices; memo.sparse_cap = c->opt.sparse_cap;
        memo.hosts.clear();
        for (size_t k = 0; k < n_sc; k++) memo.hosts.push_back(scols[k]->host);
        memo.cnt.assign(h_cnt, h_cnt + n_sc * n_slices);
        memo.dense = dense;
        memo.cuts = cuts;
        memo.idx_off.clear();
        for (const SliceCol& s : sc) memo.idx_off.push_back(s.idx_off);
        memo.arena = arena;
        memo.valid = true;
    }
    // ---- packed counts: slice i's total is in pinned memory when ev_done[i] fires; its stored entries go to the running offset ------
    uint64_t pk_base[B2R_MAX_DEFS] = {};
    if (want_pk) {
        uint64_t mine[B2R_MAX_DEFS] = {};
        for (int i = 0; i < n_slices; i++) {
            if (cut(i + 1) == cut(i)) continue;
            CUDA_TRY(cudaEventSynchronize(c->ev_done[i]));
            for (uint32_t d = 0; d < c->n_defs; d++) if (dpk.row_start[d]) mine[d] += pk_tot[i * B2R_MAX_DEFS + d];
        }
        if (hook && hook->chain) { hook->chain->publish(hook->index, mine); hook->chain->base(hook->index, pk_base); }
        for (uint32_t d = 0; d < c->n_defs; d++) {
            if (!dpk.row_start[d]) continue;
            uint64_t run = pk_base[d];
            for (int i = 0; i < n_slices; i++) {
                const uint64_t lo = cut(i), ni = cut(i + 1) - lo;
                if (!ni) continue;
                const uint64_t tot = pk_tot[i * B2R_MAX_DEFS + d];
                // row_start[lo + k] - base of the slice, k = 1 .. ni - 1, and the published total as k = ni: 8 bytes per string
                if (ni > 1) CUDA_TRY(cudaMemcpyAsync(pk_rel[d] + lo, dpk.row_start[d] + lo + i + 1, (ni - 1) * 8, cudaMemcpyDeviceToHost, c->out_stream));
                pk_rel[d][lo + ni - 1] = tot;
                d2h += ni * 8;
                if (dpk.entries[d] && run < pk->capacity) {
                    uint64_t stored = tot;
                    if (run + tot > pk->capacity) {                       // the one slice the capacity cuts: its offsets decide
                        CUDA_TRY(cudaStreamSynchronize(c->out_stream));
                        stored = pk_stored(run, pk->capacity, pk_rel[d] + lo, ni);
                    }
                    if (stored) {
                        CUDA_TRY(cudaMemcpyAsync(pk->entries[d] + run, dpk.entries[d] + lo * pkw, stored * sizeof(b2r_row_count), cudaMemcpyDeviceToHost, c->out_stream));
                        d2h += stored * sizeof(b2r_row_count);
                    }
                }
                run += tot;
            }
        }
    }
    for (const Copy& cp : copies)
        if (cp.stride && !cp.pinned && !cp.sparse && n) { CUDA_TRY(cudaMemcpyAsync(cp.host, cb + cp.off, n * cp.stride, cudaMemcpyDeviceToHost, c->out_stream)); d2h += n * cp.stride; }
    for (const Copy& cp : copies)
        if (!cp.stride && cp.bytes) { CUDA_TRY(cudaMemcpyAsync(cp.host, cb + cp.off, cp.bytes, cudaMemcpyDeviceToHost, st)); d2h += cp.bytes; }
    if (trace) CUDA_TRY(cudaEventRecord(tev[3], c->out_stream));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaStreamSynchronize(c->out_stream));
    if (want_pk) {                                                        // row_start = the base of the slice + its relative offsets
        if (!c->pool) c->pool.reset(new HostPool(c->opt.host_threads > 0 ? (unsigned)c->opt.host_threads : default_host_threads()));
        for (uint32_t d = 0; d < c->n_defs; d++) {
            if (!dpk.row_start[d]) continue;
            uint64_t b = pk_base[d];
            for (int i = 0; i < n_slices; i++) {
                const uint64_t lo = cut(i), ni = cut(i + 1) - lo;
                uint64_t* out = pk->row_start[d] + lo;
                const uint64_t* rel = pk_rel[d] + lo;
                c->pool->submit([out, rel, ni, b] { for (uint64_t k = 0; k < ni; k++) out[k] = b + (k ? rel[k - 1] : 0); });
                if (ni) b += rel[ni - 1];
            }
            if (!hook || hook->last) pk->row_start[d][n] = b;
        }
        c->pool->wait();
    }
    if (trace) {
        float h2d_end = 0, d2h_begin = 0, d2h_end = 0;
        cudaEventElapsedTime(&h2d_end, tev[0], tev[1]); cudaEventElapsedTime(&d2h_begin, tev[0], tev[2]); cudaEventElapsedTime(&d2h_end, tev[0], tev[3]);
        fprintf(stderr, "[b2r] host call, %d slices%s: last H2D done at %.2f ms, first D2H starts at %.2f ms, last D2H done at %.2f ms\n", n_slices,
                sparse ? (reuse ? " (sparse D2H, reused buffers)" : " (sparse D2H)") : "", h2d_end, d2h_begin, d2h_end);
        fprintf(stderr, "[b2r]   host wall: everything enqueued %.2f ms, payload copies issued %.2f, host zeroing done %.2f, scatter done %.2f, call done %.2f\n", w_enq, w_pay,
                w_zero, w_scat, wall_ms());
        for (auto& e : tev) cudaEventDestroy(e);
    }
    c->last_h2d_bytes = h2d; c->last_d2h_bytes = d2h + (uint64_t)n_slices * sizeof(BatchCounters);
    if (chunked) c->last_launches = launches;                             // (b2r_match_batch_host keeps reporting its last slice)

    // the batch result: the lowest failing string over all slices (reference: the first panic), overlaps summed
    b2r_batch_status r;
    memset(&r, 0, sizeof r);
    uint64_t n_overlap = 0;
    for (int i = 0; i < n_slices; i++) n_overlap += c->h_slices[i].n_overlap;
    for (int i = 0; i < n_slices; i++) {
        if (!c->h_slices[i].any_bad()) continue;
        rc = launch_diagnose(slice_params[i], c->h_slices[i].first_bad(), c->d_batch_status, st);
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemcpy(&r, c->d_batch_status, sizeof r, cudaMemcpyDeviceToHost));
        r.string_idx += slice_lo[i];
        report_failure(r);
        break;
    }
    r.n_overlap_lo = (uint32_t)n_overlap;
    if (result) *result = r;
    return r.code;
}

}  // namespace

// ---- multi-device handle -------------------------------------------------------------------------------------------------------
namespace b2r {

struct MultiState {
    std::vector<b2r_config*> kids;     // one single-device handle per device
    std::vector<int> devices;
    std::vector<ncclComm_t> comms;
    void* lib = nullptr;               // dlopen("libnccl.so.2")
    decltype(&ncclCommInitAll) comm_init_all = nullptr;
    decltype(&ncclCommDestroy) comm_destroy = nullptr;
    decltype(&ncclAllReduce) all_reduce = nullptr;
    decltype(&ncclGetErrorString) error_string = nullptr;
};

void multi_free(MultiState* m) {
    if (!m) return;
    for (ncclComm_t cm : m->comms) if (cm && m->comm_destroy) m->comm_destroy(cm);
    for (b2r_config* k : m->kids) b2r_config_free(k);
    if (m->lib) dlclose(m->lib);
    delete m;
}

int multi_set_option(MultiState* m, const char* name, const char* value) {
    for (b2r_config* k : m->kids) { const int rc = b2r_config_set_option(k, name, value); if (rc) return rc; }
    return B2R_OK;
}

}  // namespace b2r

namespace {

int multi_host_batch(b2r_config* c, const DeviceEntry& entry, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho, b2r_batch_status* result,
                     const b2r_string_mult_outputs* sm = nullptr, const b2r_string_mult_packed_outputs* pk = nullptr) {
    MultiState* m = c->multi;
    const int nd = (int)m->kids.size();
    if (!ho || (n && !h_offsets)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    for (uint64_t j = 0; j < n; j++)
        if (h_offsets[j + 1] < h_offsets[j]) { set_error("offsets must be non-decreasing (string %llu)", (unsigned long long)j); return B2R_ERR_INVALID_ARG; }
    // contiguous string ranges balanced by bytes, cut at multiples of 32 strings (whole tiles; column alignment) — of 4 strings for
    // the chunked variant, whose slices have the same granularity (host_batch), so that a few long strings still reach every device
    const uint64_t g = entry.by_bytes ? 4 : 32;
    std::vector<uint64_t> cutp(nd + 1, n);
    cutp[0] = 0;
    const uint64_t b0 = n ? h_offsets[0] : 0, total = n ? h_offsets[n] - b0 : 0;
    for (int k = 1; k < nd; k++) {
        const uint64_t target = b0 + total / nd * k + total % nd * k / nd;
        uint64_t j = (uint64_t)(std::lower_bound(h_offsets, h_offsets + n + 1, target) - h_offsets);
        j = std::min(n, (j + g / 2) & ~(g - 1));
        cutp[k] = std::max(j, cutp[k - 1]);
    }
    const uint64_t rp = ho->row_pitch, bp = ho->bitmap_pitch;
    std::vector<int> rcs(nd, 0);
    std::vector<b2r_batch_status> res(nd);
    std::vector<std::string> errs(nd);
    std::vector<std::thread> threads;
    PkChain chain(nd);                                                    // packed counts: device k's entries follow those of devices < k
    for (int k = 0; k < nd; k++)
        threads.emplace_back([&, k] {
            b2r_config* kid = m->kids[k];
            const uint64_t lo = cutp[k], hi = cutp[k + 1];
            b2r_outputs o = *ho;
            for (uint32_t d = 0; d < kid->n_defs; d++) {
                const size_t w = kid->packed[d].state_width;
                if (o.states[d]) o.states[d] = (unsigned char*)o.states[d] + lo * rp * w;
                if (o.substr_ids[d]) o.substr_ids[d] += lo * rp;
                if (o.start_enable[d]) o.start_enable[d] += lo * bp;
                if (o.end_enable[d]) o.end_enable[d] += lo * bp;
            }
            if (o.masked_chars) o.masked_chars += lo * rp;
            if (o.masked_substr_ids) o.masked_substr_ids += lo * rp;
            if (o.status) o.status += lo;
            if (o.records) o.records += lo * (size_t)ho->max_records;
            if (o.compact_bytes) o.compact_bytes += lo * (size_t)ho->compact_pitch;
            b2r_string_mult_outputs s{};                                 // per-string counts: this device's strings, no exchange
            if (sm) {
                s = *sm;
                for (uint32_t d = 0; d < kid->n_defs; d++) {
                    if (s.entries[d]) s.entries[d] += lo * sm->max_entries;
                    if (s.n_entries[d]) s.n_entries[d] += lo;
                    if (s.endpoint_counts[d]) s.endpoint_counts[d] += lo * 2 * kid->packed[d].erows.size();
                }
            }
            b2r_string_mult_packed_outputs q{};                          // the entries' offset is known once devices < k have published
            if (pk) {
                q = *pk;
                for (uint32_t d = 0; d < kid->n_defs; d++) {
                    if (q.row_start[d]) q.row_start[d] += lo;
                    if (q.endpoint_counts[d]) q.endpoint_counts[d] += lo * 2 * kid->packed[d].erows.size();
                }
            }
            MultiHook hook;
            hook.comm = m->comms[k]; hook.all_reduce = m->all_reduce; hook.error_string = m->error_string; hook.first = k == 0;
            hook.chain = pk ? &chain : nullptr; hook.index = k; hook.last = k == nd - 1;
            memset(&res[k], 0, sizeof res[k]);
            static const uint64_t zero_off[1] = {0};
            rcs[k] = host_batch(kid, entry, h_bytes, n ? h_offsets + lo : zero_off, hi - lo, &o, &res[k], &hook, sm ? &s : nullptr, pk ? &q : nullptr);
            if (rcs[k]) errs[k] = get_error();
        });
    for (auto& t : threads) t.join();
    c->last_h2d_bytes = c->last_d2h_bytes = 0; c->last_launches = 0;
    for (int k = 0; k < nd; k++) { c->last_h2d_bytes += m->kids[k]->last_h2d_bytes; c->last_d2h_bytes += m->kids[k]->last_d2h_bytes; c->last_launches += m->kids[k]->last_launches; }
    // the lowest failing string wins (reference: the first panic); infrastructure errors first
    b2r_batch_status r;
    memset(&r, 0, sizeof r);
    uint64_t overlap = 0;
    for (int k = 0; k < nd; k++) overlap += res[k].n_overlap_lo;
    for (int k = 0; k < nd; k++)
        if (rcs[k] && rcs[k] != B2R_ERR_INVALID_TRANSITION && rcs[k] != B2R_ERR_TOO_LONG) { set_error("device %d: %s", m->devices[k], errs[k].c_str()); return rcs[k]; }
    for (int k = 0; k < nd; k++)
        if (rcs[k]) { r = res[k]; r.string_idx += cutp[k]; report_failure(r); break; }
    r.n_overlap_lo = (uint32_t)overlap;
    if (result) *result = r;
    return r.code;
}

}  // namespace

extern "C" {

int b2r_config_new_multi(const b2r_allstr* const* allstr, const b2r_substr* const* const* substrs, const uint32_t* n_substrs, uint32_t n_defs,
                         uint64_t max_chars_size, const int* device_ids, uint32_t n_devices, b2r_config** out) {
    if (!out || !device_ids || n_devices == 0) { set_error("null / empty argument"); return B2R_ERR_INVALID_ARG; }
    for (uint32_t i = 0; i < n_devices; i++)
        for (uint32_t j = 0; j < i; j++)
            if (device_ids[i] == device_ids[j]) { set_error("device %d is listed twice", device_ids[i]); return B2R_ERR_INVALID_ARG; }
    // the parent answers the table queries; the children own the devices
    b2r_config* parent = nullptr;
    int rc = b2r_config_new(allstr, substrs, n_substrs, n_defs, max_chars_size, -1, &parent);
    if (rc) return rc;
    MultiState* m = new (std::nothrow) MultiState;
    if (!m) { b2r_config_free(parent); set_error("out of memory"); return B2R_ERR_INVALID_ARG; }
    parent->multi = m;
    for (uint32_t i = 0; i < n_devices; i++) {
        b2r_config* kid = nullptr;
        rc = b2r_config_new(allstr, substrs, n_substrs, n_defs, max_chars_size, device_ids[i], &kid);
        if (rc) { b2r_config_free(parent); return rc; }
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        if (!kid->opt.host_threads) kid->opt.host_threads = (int)std::max(2u, std::min(8u, hw / 2 / n_devices));
        m->kids.push_back(kid);
        m->devices.push_back(device_ids[i]);
    }
    // NCCL is resolved at run time: a process that already carries a libnccl.so.2 (PyTorch's) shares it
    m->lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!m->lib) { set_error("b2r_config_new_multi: libnccl.so.2 cannot be loaded (%s); the multi-device handle has no other exchange path", dlerror()); b2r_config_free(parent); return B2R_ERR_UNSUPPORTED; }
    m->comm_init_all = (decltype(m->comm_init_all))dlsym(m->lib, "ncclCommInitAll");
    m->comm_destroy = (decltype(m->comm_destroy))dlsym(m->lib, "ncclCommDestroy");
    m->all_reduce = (decltype(m->all_reduce))dlsym(m->lib, "ncclAllReduce");
    m->error_string = (decltype(m->error_string))dlsym(m->lib, "ncclGetErrorString");
    if (!m->comm_init_all || !m->comm_destroy || !m->all_reduce || !m->error_string) { set_error("libnccl.so.2 lacks a required symbol"); b2r_config_free(parent); return B2R_ERR_UNSUPPORTED; }
    m->comms.assign(n_devices, nullptr);
    const ncclResult_t nr = m->comm_init_all(m->comms.data(), (int)n_devices, device_ids);
    if (nr != ncclSuccess) { set_error("ncclCommInitAll failed: %s", m->error_string(nr)); m->comms.clear(); b2r_config_free(parent); return B2R_ERR_CUDA; }
    *out = parent;
    return B2R_OK;
}

uint32_t b2r_config_num_devices(const b2r_config* c) { return !c ? 0 : c->multi ? (uint32_t)c->multi->kids.size() : c->device >= 0 ? 1u : 0u; }

int b2r_match_batch_host(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                         b2r_batch_status* result) {
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (c->multi) return multi_host_batch(c, BATCH_ENTRY, h_bytes, h_offsets, n, ho, result);
    return host_batch(c, BATCH_ENTRY, h_bytes, h_offsets, n, ho, result, nullptr);
}

int b2r_match_batch_chunked_host(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                                 b2r_batch_status* result) {
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (c->multi) return multi_host_batch(c, CHUNKED_ENTRY, h_bytes, h_offsets, n, ho, result);
    return host_batch(c, CHUNKED_ENTRY, h_bytes, h_offsets, n, ho, result, nullptr);
}

}  // extern "C"

namespace {

int host_batch_mult(b2r_config* c, const DeviceEntry& entry, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                    const b2r_string_mult_outputs* sm, b2r_batch_status* result) {
    // the arguments are checked first (the same answer on any handle), then the device
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (!ho || !sm) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    const int rc = check_string_mult(c, sm);
    if (rc) return rc;
    if (!c->multi && c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    if (c->multi) return multi_host_batch(c, entry, h_bytes, h_offsets, n, ho, result, sm);
    return host_batch(c, entry, h_bytes, h_offsets, n, ho, result, nullptr, sm);
}

int host_batch_mult_packed(b2r_config* c, const DeviceEntry& entry, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                           const b2r_string_mult_packed_outputs* pk, b2r_batch_status* result) {
    // the arguments are checked first (the same answer on any handle), then the device
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (!ho || !pk) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    const int rc = check_string_mult_packed(c, pk);
    if (rc) return rc;
    if (!c->multi && c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    if (c->multi) return multi_host_batch(c, entry, h_bytes, h_offsets, n, ho, result, nullptr, pk);
    return host_batch(c, entry, h_bytes, h_offsets, n, ho, result, nullptr, nullptr, pk);
}

}  // namespace

extern "C" {

int b2r_match_batch_host_mult(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                              const b2r_string_mult_outputs* sm, b2r_batch_status* result) {
    return host_batch_mult(c, BATCH_ENTRY, h_bytes, h_offsets, n, ho, sm, result);
}

int b2r_match_batch_chunked_host_mult(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                                      const b2r_string_mult_outputs* sm, b2r_batch_status* result) {
    return host_batch_mult(c, CHUNKED_ENTRY, h_bytes, h_offsets, n, ho, sm, result);
}

int b2r_match_batch_host_mult_packed(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                                     const b2r_string_mult_packed_outputs* pk, b2r_batch_status* result) {
    return host_batch_mult_packed(c, BATCH_ENTRY, h_bytes, h_offsets, n, ho, pk, result);
}

int b2r_match_batch_chunked_host_mult_packed(b2r_config* c, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n, const b2r_outputs* ho,
                                             const b2r_string_mult_packed_outputs* pk, b2r_batch_status* result) {
    return host_batch_mult_packed(c, CHUNKED_ENTRY, h_bytes, h_offsets, n, ho, pk, result);
}

int b2r_match_substrs(b2r_config* c, const uint8_t* characters, uint64_t len, const b2r_outputs* h_out, b2r_batch_status* result) {
    if (!c || !h_out) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    const uint64_t offsets[2] = {0, len};
    b2r_config* one = c->multi ? c->multi->kids[0] : c;                   // one string: one device
    return host_batch(one, BATCH_ENTRY, characters, offsets, 1, h_out, result, nullptr);
}

int b2r_last_host_bytes(const b2r_config* c, uint64_t* h2d_bytes, uint64_t* d2h_bytes) {
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (h2d_bytes) *h2d_bytes = c->last_h2d_bytes;
    if (d2h_bytes) *d2h_bytes = c->last_d2h_bytes;
    return B2R_OK;
}

// Host-pointer variant of the long-string path: the string goes up in one copy, the columns come back in one copy each.
int b2r_match_long_host(b2r_config* c, const uint8_t* h_bytes, uint64_t len, const b2r_outputs* ho, b2r_batch_status* result) {
    if (!c || !ho || (!h_bytes && len)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    if (c->multi) c = c->multi->kids[0];
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    const uint64_t M = len + 1;
    int rc = check_outputs(c, ho, false, M);
    if (rc) return rc;
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    cudaStream_t st = c->host_stream;
    if ((rc = c->ws_bytes.reserve(align_up(len + 16, 256)))) return rc;
    const uint64_t rp = ho->row_pitch, bp = ho->bitmap_pitch;
    size_t need = 0;
    auto slot = [&](size_t bytes) { size_t o = need; need += align_up(bytes, 256); return o; };
    struct Copy { size_t off; void* host; size_t bytes; };
    std::vector<Copy> copies;
    std::vector<size_t> offs;
    b2r_outputs dout = *ho;
    auto want = [&](void* host, size_t bytes) -> size_t {
        if (!host) { offs.push_back(0); return 0; }
        const size_t o = slot(bytes);
        copies.push_back({o, host, bytes});
        offs.push_back(o);
        return o;
    };
    // first pass: sizes; second pass (after the reserve): device pointers
    for (uint32_t d = 0; d < c->n_defs; d++) {
        want(ho->states[d], rp * c->packed[d].state_width); want(ho->substr_ids[d], rp); want(ho->start_enable[d], bp); want(ho->end_enable[d], bp);
        want(ho->mult[d], c->packed[d].rows.size() * 8); want(ho->endpoint_mult[d], c->packed[d].erows.size() * 16);
    }
    want(ho->masked_chars, rp); want(ho->masked_substr_ids, rp); want(ho->status, sizeof(b2r_string_status));
    want(ho->records, (size_t)ho->max_records * sizeof(b2r_substr_record)); want(ho->compact_bytes, (size_t)ho->compact_pitch);
    if ((rc = c->ws_cols.reserve(need + 256))) return rc;
    unsigned char* cb = (unsigned char*)c->ws_cols.p;
    size_t k = 0;
    auto dev = [&](void* host) -> void* { const size_t o = offs[k++]; return host ? cb + o : nullptr; };
    for (uint32_t d = 0; d < c->n_defs; d++) {
        dout.states[d] = dev(ho->states[d]); dout.substr_ids[d] = (uint8_t*)dev(ho->substr_ids[d]);
        dout.start_enable[d] = (uint8_t*)dev(ho->start_enable[d]); dout.end_enable[d] = (uint8_t*)dev(ho->end_enable[d]);
        dout.mult[d] = (uint64_t*)dev(ho->mult[d]); dout.endpoint_mult[d] = (uint64_t*)dev(ho->endpoint_mult[d]);
        if (ho->flags & B2R_OUT_ACCUMULATE_MULT) {
            if (ho->mult[d]) CUDA_TRY(cudaMemcpyAsync(dout.mult[d], ho->mult[d], c->packed[d].rows.size() * 8, cudaMemcpyHostToDevice, st));
            if (ho->endpoint_mult[d]) CUDA_TRY(cudaMemcpyAsync(dout.endpoint_mult[d], ho->endpoint_mult[d], c->packed[d].erows.size() * 16, cudaMemcpyHostToDevice, st));
        }
    }
    dout.masked_chars = (uint8_t*)dev(ho->masked_chars); dout.masked_substr_ids = (uint8_t*)dev(ho->masked_substr_ids);
    dout.status = (b2r_string_status*)dev(ho->status); dout.records = (b2r_substr_record*)dev(ho->records);
    dout.compact_bytes = (uint8_t*)dev(ho->compact_bytes);
    dout.flags &= ~(uint32_t)B2R_OUT_SPARSE_D2H;
    if (len) CUDA_TRY(cudaMemcpyAsync(c->ws_bytes.p, h_bytes, len, cudaMemcpyHostToDevice, st));
    if ((rc = b2r_match_long(c, (const uint8_t*)c->ws_bytes.p, len, &dout, st))) return rc;
    uint64_t d2h = 0;
    for (const Copy& cp : copies) { CUDA_TRY(cudaMemcpyAsync(cp.host, cb + cp.off, cp.bytes, cudaMemcpyDeviceToHost, st)); d2h += cp.bytes; }
    c->last_h2d_bytes = len; c->last_d2h_bytes = d2h;
    return b2r_batch_result(c, st, result);
}

}  // extern "C"
