// The handle behind `b2r_config` and the helpers shared by api.cu (device-pointer entry points) and host.cu (host-pointer
// entry points: staging, sliced copy pipeline, sparse D2H, the small-batch path, the multi-device handle).  Internal.
#pragma once
#include <cuda_runtime.h>

#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/b2r.h"
#include "defs.hpp"
#include "kernels.cuh"

struct b2r_allstr { b2r::AllstrDef def; };
struct b2r_substr { b2r::SubstrDef def; };

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            b2r::set_error("%s failed: %s", #expr, cudaGetErrorString(_e));              \
            return B2R_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

namespace b2r {

struct DevBuf {                       // device allocation that only grows
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t n) {
        if (n <= cap) return B2R_OK;
        if (p) CUDA_TRY(cudaFree(p));
        p = nullptr; cap = 0;
        CUDA_TRY(cudaMalloc(&p, n));
        cap = n;
        return B2R_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinBuf {                       // page-locked host allocation that only grows
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t n) {
        if (n <= cap) return B2R_OK;
        if (p) CUDA_TRY(cudaFreeHost(p));
        p = nullptr; cap = 0;
        CUDA_TRY(cudaHostAlloc(&p, n, cudaHostAllocPortable | cudaHostAllocMapped));   // unified addressing: kernels may write it directly
        cap = n;
        return B2R_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct DevDef {
    uint8_t* byte_class = nullptr;
    uint32_t* trans = nullptr;
    uint32_t* hot = nullptr;     // walk table [C][P] (walk.cuh)
    uint32_t *row_bin = nullptr, *erow_start_bin = nullptr, *erow_end_bin = nullptr;
    uint32_t *sorted_bins = nullptr, *sorted_rows = nullptr;   // rows >= 1 ordered by bin ch*S + cur (string_mult.cu: bin -> row by binary search)
    unsigned long long *hist = nullptr, *ep_start = nullptr, *ep_end = nullptr;  // inside cfg->scratch
};

// Host worker threads of one handle (sparse D2H mode: zeroing and scattering the caller's dense columns).
class HostPool {
public:
    explicit HostPool(unsigned n_threads);
    ~HostPool();
    void submit(std::function<void()> fn);
    void wait();                      // until every submitted task has finished
    unsigned size() const { return (unsigned)threads_.size(); }
    unsigned pending() { std::lock_guard<std::mutex> l(m_); return (unsigned)pending_; }   // tasks submitted and not finished (trace output)

private:
    void run();
    std::vector<std::thread> threads_;
    std::deque<std::function<void()>> q_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    size_t pending_ = 0;
    bool stop_ = false;
};

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct MultiState;                    // host.cu: the children of a multi-device handle and their NCCL communicators

// What the last sparse-D2H call scattered into which host buffers (B2R_OUT_SPARSE_REUSE: the next call on the same buffers clears
// exactly those sectors instead of zeroing the whole columns).  The sector index lists themselves stay in the pinned arena.
struct SparseMemo {
    bool valid = false;
    uint64_t n = 0, rp = 0, bp = 0;
    int n_slices = 0, sparse_cap = 0, arena = 0;   // arena: which of the two pinned arenas holds the index lists
    std::vector<const void*> hosts;   // caller's buffer of every sparse column
    std::vector<uint32_t> cnt;        // [slice][column] sectors scattered
    std::vector<char> dense;          // [slice][column] 1: that column slice was copied densely
    std::vector<uint64_t> cuts;       // slice i: strings [cuts[i], cuts[i + 1])
    std::vector<size_t> idx_off;      // [slice][column] where its sector index list lies in the pinned arena
};

}  // namespace b2r

struct b2r_config {
    int device = -1;             // -1: host-only handle (table queries), no matching
    uint64_t max_chars = 0;
    uint32_t n_defs = 0;
    b2r::PackedDef packed[B2R_MAX_DEFS];
    b2r::DevDef dev[B2R_MAX_DEFS];
    void* tables = nullptr;      // one allocation holding every constant table
    uint8_t* d_bin_of_byte = nullptr;   // compact multiplicity bins (kernels.cuh): byte -> column, column -> byte; inside `tables`
    uint8_t* d_bin_byte = nullptr;
    uint32_t bin_cols = 256;
    void* scratch = nullptr;     // BatchCounters + hist + endpoint counters, zeroed per batch
    size_t scratch_bytes = 0;
    b2r_batch_status* d_batch_status = nullptr;
    // testing / tuning hooks: read ONCE from the environment when the handle is created (B2R_TABLE_MODE, B2R_HIST_MODE, B2R_DEBUG,
    // B2R_SPREAD_FILL, B2R_FUSE, B2R_SLICES, B2R_TRACE_HOST, B2R_HIST_CACHE_LOG2), changed later only through b2r_config_set_option
    struct Options {
        int force_table_mode = -1;    // repl|plain|plain16|global
        int force_hist_mode = -1;     // smem|global
        uint32_t debug = 0;           // timing experiments only: emit skips 1 zero-fill, 2 scan, 4 final-state loads, 8 status
        uint32_t spread_fill = 1;
        int stagger_ns = -1;          // start offset between the warps of a walk CTA (-1 = default, see plan in api.cu)
        int fuse = -1;                // 1: walk_kernel runs the emit stage itself; 0: emit_kernel as its own launch (it also zero-fills); 2: emit_kernel as its
                                      // own launch, but the walk zero-fills; -1: 1 for one def with replicated tables, else 2
        int slices = 0;               // host entry point: slices per batch (0 = default)
        bool trace_host = false;
        int hist_cache_log2 = 0;      // 0 = default
        int host_threads = 0;         // sparse D2H mode: host worker threads (0 = default)
        int small_path = 1;           // 0: small batches take the sliced pipeline too (testing hook)
        int long_fused = 1;           // 0: the long-string path computes the chunk maps with the general multi-kernel pass (testing hook)
        long long chunked_max_maps = 0;   // chunked batch: bytes of slot transition vectors per pass (0 = 1 GiB; testing hook)
        int sparse_cap = 0;           // sparse D2H mode: sectors per column slice before the dense fallback (0 = default; testing hook)
        int host_debug = 0;           // timing experiments only: 1 = skip the host-side clearing, 2 = skip the host-side scatter (results are wrong)
        int sparse_direct = 0;        // sparse D2H mode: 1 = the kernel stores the compacted sectors straight into pinned host memory (36-byte
                                      // PCIe writes); 0 = it compacts into device memory and exact-size copies follow once the host has the count
    } opt;
    b2r::DevBuf ws_fmask;                  // granule flags (walk -> emit)
    b2r::DevBuf ws_long;                   // long-string path: chunk offsets, transition-vector tree, entry states, flag summary
    b2r::DevBuf ws_states[B2R_MAX_DEFS];   // state column of a def the caller did not ask for (emit reads it)
    b2r::DevBuf ws_smult;                  // per-string counters of strings longer than one string_mult segment (string_mult.cu)
    b2r::DevBuf ws_smpk;                   // packed per-string counts: running totals, list lengths and slots of one pass (string_mult.cu)
    b2r::WalkParams last = {};
    bool have_last = false;
    uint32_t last_launches = 0;
    bool timing = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // before walk, after walk, after emit, after finalize
    // staging for the host-pointer entry points
    b2r::DevBuf ws_bytes, ws_offsets, ws_cols, ws_sparse, ws_sparse_arena;
    b2r::PinBuf pin_sparse[2], pin_small;
    b2r::PinBuf pin_pk;                    // packed per-string counts: slice totals and slice-relative row_start values on their way back
    cudaStream_t host_stream = nullptr;
    cudaStream_t in_stream = nullptr, out_stream = nullptr;   // host entry point: H2D / D2H copies overlapping the kernels
    cudaStream_t pay_stream = nullptr;                        // sparse D2H mode: the compacted sectors of a slice
    b2r::BatchCounters* counters_copy = nullptr;              // small-batch path: finalize_kernel leaves a copy of the batch counters here
    bool sparse_zeroed = false;                               // chunked host pipeline: the sparse columns are zero already (emit_kernel skips its fill)
    static constexpr int MAX_SLICES = 16;
    cudaEvent_t ev_in[MAX_SLICES] = {}, ev_done[MAX_SLICES] = {}, ev_pay[MAX_SLICES] = {};
    b2r::BatchCounters* h_slices = nullptr;    // pinned: the counters of every slice of a host batch
    cudaEvent_t ev_fork = nullptr;
    std::unique_ptr<b2r::HostPool> pool;       // created by the first sparse-mode call
    uint64_t last_h2d_bytes = 0, last_d2h_bytes = 0;   // bytes the last host call moved over PCIe
    b2r::SparseMemo sparse_memo;
    b2r::MultiState* multi = nullptr;          // non-null: a multi-device handle (b2r_config_new_multi); `device` = its first device
};

namespace b2r {

// api.cu
int check_outputs(const b2r_config* c, const b2r_outputs* o, bool check_ptrs, uint64_t M = 0);
void fill_walk_params(const b2r_config* c, WalkParams& p, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                      const b2r_outputs* o, uint64_t max_chars);
int enqueue_finalize(b2r_config* c, const b2r_outputs* o, uint64_t n, uint64_t max_chars, cudaStream_t st);
int match_batch_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes, const b2r_outputs* o,
                     uint64_t max_chars, cudaStream_t st);
// b2r_match_batch_chunked behind its argument checks; the same signature as match_batch_impl, so that the host pipeline can run either
int match_batch_chunked_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes, const b2r_outputs* o,
                             uint64_t max_chars, cudaStream_t st);
using BatchEntry = decltype(&match_batch_impl);
// grows the workspaces a match_batch_chunked_impl call over n strings uses (ws_fmask, ws_states of the defs `o` has no state column
// for, ws_long) to their size for n; a call over at most n strings then reserves nothing
int chunked_reserve(b2r_config* c, uint64_t n, const b2r_outputs* o, uint64_t max_chars);
void report_failure(const b2r_batch_status& r);      // sets the thread's error text for a failed string (reference panic text)
// string_mult.cu: the argument checks of the per-string outputs (host: pointers into host memory, states / status may be NULL),
// and the post-pass over n strings whose state columns and status the match kernels have written (device pointers; `states` =
// the columns they used, scratch ones included).  Adds its kernels to *launches.
int check_string_mult(const b2r_config* c, const b2r_string_mult_outputs* sm);
bool string_mult_wanted(const b2r_config* c, const b2r_string_mult_outputs* sm, uint32_t d);
int string_mult_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t max_chars, void* const* states,
                     uint64_t row_pitch, const b2r_string_status* status, const b2r_string_mult_outputs* sm, cudaStream_t st, uint32_t* launches);
// the packed layout: argument checks, the workspace of a call over at most n strings (reserved before a host pipeline enqueues
// its first slice), and the post-pass itself.  row_start is written relative to the call's first string; with host_total
// (pinned, [n_defs]) the call's total per def is also stored there by a kernel, readable once the stream has passed the call.
bool string_mult_packed_wanted(const b2r_config* c, const b2r_string_mult_packed_outputs* pk, uint32_t d);
int check_string_mult_packed(const b2r_config* c, const b2r_string_mult_packed_outputs* pk);
int string_mult_packed_reserve(b2r_config* c, uint64_t n, uint64_t max_chars, const b2r_string_mult_packed_outputs* pk);
int string_mult_packed_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t max_chars, void* const* states,
                            uint64_t row_pitch, const b2r_string_status* status, const b2r_string_mult_packed_outputs* pk, uint64_t* host_total,
                            cudaStream_t st, uint32_t* launches);
// host.cu
void multi_free(MultiState* m);
int multi_set_option(MultiState* m, const char* name, const char* value);

}  // namespace b2r
