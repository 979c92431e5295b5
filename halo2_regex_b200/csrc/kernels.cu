// Small kernels (multiplicity finalisation, failure diagnosis) and the launch planning / dispatch of walk_kernel and
// emit_kernel.  The two big kernels live in walk.cuh / emit.cuh and are instantiated per number of defs in walk_inst.cu.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "emit.cuh"
#include "walk.cuh"

namespace b2r {

// ---- multiplicity finalisation: dense (byte,state) bins -> table rows (reference order, src/table.rs:101-122) ----
__global__ void finalize_kernel(const __grid_constant__ FinalizeParams p) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t nth = gridDim.x * blockDim.x;
    if (p.counters_copy && tid == 0) *p.counters_copy = *p.counters;
    for (uint32_t d = 0; d < p.n_defs; d++) {
        const auto& f = p.def[d];
        if (f.mult) {
            for (uint32_t r = tid; r < f.n_rows; r += nth) {
                const unsigned long long v = (r == 0) ? p.counters->pad_rows : f.hist[f.row_bin[r]];
                f.mult[r] = (p.accumulate ? f.mult[r] : 0ull) + v;
            }
        }
        if (f.endpoint_mult && tid == 0) {   // a handful of rows
            unsigned long long tot_s = 0, tot_e = 0;
            for (uint32_t r = 1; r < f.n_erows; r++) {
                const unsigned long long vs = f.erow_start_bin[r] != 0xFFFFFFFFu ? f.ep_start[f.erow_start_bin[r]] : 0ull;
                const unsigned long long ve = f.erow_end_bin[r] != 0xFFFFFFFFu ? f.ep_end[f.erow_end_bin[r]] : 0ull;
                tot_s += vs; tot_e += ve;
                f.endpoint_mult[r] = (p.accumulate ? f.endpoint_mult[r] : 0ull) + vs;
                f.endpoint_mult[f.n_erows + r] = (p.accumulate ? f.endpoint_mult[f.n_erows + r] : 0ull) + ve;
            }
            // every other row of the batch looks up (0, dummy, dummy) = endpoint row 0
            f.endpoint_mult[0] = (p.accumulate ? f.endpoint_mult[0] : 0ull) + (p.n_rows_total - tot_s);
            f.endpoint_mult[f.n_erows] = (p.accumulate ? f.endpoint_mult[f.n_erows] : 0ull) + (p.n_rows_total - tot_e);
        }
    }
}

// ---- diagnose: details of the failing string for the batch status (one thread) ------------------------------------
__global__ void diagnose_kernel(const __grid_constant__ WalkParams p, uint64_t j, b2r_batch_status* out) {
    b2r_batch_status r = diagnose_string(p, j);
    r.n_overlap_lo = (uint32_t)p.counters->n_overlap;
    *out = r;
}

// ---- launch planning ---------------------------------------------------------------------------------------------------
int device_limits(int* n_sm, int* max_smem) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { set_error("cudaGetDevice failed"); return B2R_ERR_CUDA; }
    cudaDeviceGetAttribute(n_sm, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    return B2R_OK;
}

static constexpr int MIN_WARPS_REPL16 = 10; // 16-bit replicated tables: taken when at least this many warps fit next to them
static constexpr int MIN_WARPS_REPL = 12;  // below this the replicated tables are not worth the lost occupancy (measured on the two-def set)

// Picks where the walk tables and the multiplicity bins live.  Preference: replicated tables + shared bins with as many
// warps as possible; then a single copy of the tables; then global tables.  Bins go to shared memory whenever they fit.
static int plan_walk_tables(WalkParams& p, bool wide, int force_table_mode, int force_hist_mode, int hist_cache_log2);

int plan_walk(WalkParams& p, bool wide, int force_table_mode, int force_hist_mode, int hist_cache_log2) {
    p.cls_repl = 0;
    int rc = plan_walk_tables(p, wide, force_table_mode, force_hist_mode, hist_cache_log2);
    if (rc) return rc;
    // single-copy tables in shared memory: the byte -> class lookup (one per byte, shared by all defs) is still made conflict-free by
    // replicating the 256-entry class table once per lane (32 KB) — when every warp still fits next to it
    if ((p.table_mode == TABLE_PLAIN || p.table_mode == TABLE_PLAIN16) && p.n_tiles > 8) {
        int n_sm = 0, max_smem = 0;
        if ((rc = device_limits(&n_sm, &max_smem))) return rc;
        p.cls_repl = 1;
        if (walk_smem_bytes(p, wide ? 2 : 1, WALK_MAX_THREADS / 32) > (size_t)max_smem) p.cls_repl = 0;
    }
    return B2R_OK;
}

static int plan_walk_tables(WalkParams& p, bool wide, int force_table_mode, int force_hist_mode, int hist_cache_log2) {
    int n_sm = 0, max_smem = 0;
    int rc = device_limits(&n_sm, &max_smem);
    if (rc) return rc;
    const uint32_t sb = wide ? 2 : 1;
    auto fits_k = [&](uint32_t tm, uint32_t hm, int warps) {
        p.table_mode = tm; p.hist_mode = hm;
        if (tm != TABLE_GLOBAL) {
            const uint32_t stride = walk_stride(tm);
            for (uint32_t d = 0; d < p.n_defs; d++)
                if ((uint64_t)p.def[d].padded_states * stride > 65536u || (tm == TABLE_REPL16 && p.def[d].padded_states > 512u)) return false;   // the entry's low bits hold next*stride (pair-packed: (next >> 1) << 7 in 16 bits)
        }
        uint64_t bins = 0;
        for (uint32_t d = 0; d < p.n_defs; d++) bins += (uint64_t)(p.def[d].num_states + 1) * walk_bin_cols(p) * 4u;
        if (hm == HIST_SMEM && (wide || bins > (uint64_t)max_smem)) return false;
        uint64_t tabs = 0;
        if (tm != TABLE_GLOBAL)
            for (uint32_t d = 0; d < p.n_defs; d++) tabs += (uint64_t)p.def[d].num_classes * p.def[d].padded_states * walk_stride(tm);
        if (tabs > (uint64_t)max_smem) return false;
        return walk_smem_bytes(p, sb, warps) <= (size_t)max_smem;
    };
    // HIST_GLOBAL: the largest bin cache (4096 .. 256 slots per def) that leaves room for the warps
    auto fits = [&](uint32_t tm, uint32_t hm, int warps) {
        const uint32_t top = (hist_cache_log2 >= 8 && hist_cache_log2 <= 14) ? (uint32_t)hist_cache_log2 : 12u;   // tuning hook (B2R_HIST_CACHE_LOG2)
        for (p.hist_cache_log2 = top; p.hist_cache_log2 >= 8; p.hist_cache_log2--)
            if (fits_k(tm, hm, warps)) return true;
        p.hist_cache_log2 = 8;
        return false;
    };
    // preference: replicated tables + shared bins; a single copy of 16-bit entries; bins behind the cache; a single copy of
    // 32-bit entries; global tables.  A placement is taken when at least `need` warps fit next to it.
    // (single copy: the 16-bit entries win at every size measured — two entries per bank word halve the conflicts and
    //  the footprint: 3-def set 28.9 % -> 31.9 % of HBM peak, 2-def 40.1 -> 43.3, 1023-state DFA 2.2x)
    const uint32_t P16 = TABLE_PLAIN16, P32 = TABLE_PLAIN;
    // (TABLE_REPL16 is not in the fall-back order below: it is taken by the rule above, or when asked for)
    const uint32_t order[][2] = {{TABLE_REPL, HIST_SMEM}, {P16, HIST_SMEM}, {TABLE_REPL, HIST_GLOBAL}, {P16, HIST_GLOBAL},
                                 {P32, HIST_SMEM}, {P32, HIST_GLOBAL}, {TABLE_GLOBAL, HIST_GLOBAL}, {TABLE_REPL16, HIST_SMEM}, {TABLE_REPL16, HIST_GLOBAL}};
    // a handful of tiles (the reference's one-string call): one CTA walks them, and staging 100 KB of replicated tables for it costs
    // more than the bank conflicts of a few warps — a single copy of the tables
    if (p.n_tiles <= 8 && force_table_mode < 0 && force_hist_mode < 0 && !p.segment_mode)
        for (const uint32_t tm : {P32, P16})
            if (fits(tm, HIST_SMEM, 4)) return B2R_OK;
    // two or three small DFAs whose 32-bit replicated tables do not fit: 16-bit replicated tables next to compact bins, if enough warps
    // still fit to hide the latency of the chains
    if (force_table_mode < 0 && force_hist_mode < 0 && p.n_defs >= 2 && p.n_defs <= 3 && !wide && !fits(TABLE_REPL, HIST_SMEM, 4) &&
        fits(TABLE_REPL16, HIST_SMEM, MIN_WARPS_REPL16))
        return B2R_OK;
    for (const auto& o : order) {
        if (force_table_mode >= 0 && (uint32_t)force_table_mode != o[0]) continue;   // testing hooks: honoured when they fit
        if (force_hist_mode >= 0 && (uint32_t)force_hist_mode != o[1]) continue;
        if (fits(o[0], o[1], 4)) return B2R_OK;
    }
    for (const int need : {MIN_WARPS_REPL, 4})
        for (const auto& o : order) {
            if (o[0] == TABLE_GLOBAL && need != 4) continue;                       // global tables: the last resort
            if (o[0] == TABLE_REPL16 && force_table_mode != (int)TABLE_REPL16) continue;
            if (fits(o[0], o[1], o[0] == TABLE_REPL ? MIN_WARPS_REPL : need)) return B2R_OK;
        }
    set_error("walk_kernel: no table placement fits in shared memory");
    return B2R_ERR_UNSUPPORTED;
}

template <int D, bool CH>
int launch_walk_d(const WalkParams& p, bool wide, size_t smem, int grid, int block, cudaStream_t st);
template <> int launch_walk_d<1, false>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<2, false>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<3, false>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<4, false>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<1, true>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<2, true>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<3, true>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <> int launch_walk_d<4, true>(const WalkParams&, bool, size_t, int, int, cudaStream_t);
template <int D>
int launch_emit_d(const WalkParams& p, bool wide, size_t smem, int grid, cudaStream_t st);
template <> int launch_emit_d<1>(const WalkParams&, bool, size_t, int, cudaStream_t);
template <> int launch_emit_d<2>(const WalkParams&, bool, size_t, int, cudaStream_t);
template <> int launch_emit_d<3>(const WalkParams&, bool, size_t, int, cudaStream_t);
template <> int launch_emit_d<4>(const WalkParams&, bool, size_t, int, cudaStream_t);

int launch_walk(const WalkParams& p, bool wide, void* stream, LaunchInfo* chosen) {
    int n_sm = 0, max_smem = 0;
    int rc = device_limits(&n_sm, &max_smem);
    if (rc) return rc;
    const uint32_t sb = wide ? 2 : 1;
    int warps = WALK_MAX_THREADS / 32;
    while (warps > 1 && walk_smem_bytes(p, sb, warps) > (size_t)max_smem) warps--;
    size_t smem = walk_smem_bytes(p, sb, warps);
    if (smem > (size_t)max_smem) { set_error("walk_kernel: %zu bytes of shared memory needed, %d available", smem, max_smem); return B2R_ERR_UNSUPPORTED; }
    // persistent: one CTA per SM.  A batch of fewer tiles than the SMs have warps is spread over ALL SMs with fewer warps per
    // CTA (the long-string path: 2048 tiles -> 147 CTAs of 14 warps instead of 128 of 16; every warp still walks one tile)
    if ((long long)p.n_tiles < (long long)n_sm * warps) {
        const int per = (int)((p.n_tiles + n_sm - 1) / n_sm);
        warps = per < 4 ? (warps < 4 ? warps : 4) : per;                   // at least four warps: they also stage the tables
        smem = walk_smem_bytes(p, sb, warps);
    }
    const long long ctas = ((long long)p.n_tiles + warps - 1) / warps;
    const int grid = (int)(ctas < n_sm ? (ctas > 0 ? ctas : 1) : n_sm);
    if (chosen) { chosen->grid = grid; chosen->block = warps * 32; chosen->smem_bytes = smem; }
    cudaStream_t st = (cudaStream_t)stream;
    const bool ch = p.chunk_k != 0;
    switch (p.n_defs) {
        case 1: return ch ? launch_walk_d<1, true>(p, wide, smem, grid, warps * 32, st) : launch_walk_d<1, false>(p, wide, smem, grid, warps * 32, st);
        case 2: return ch ? launch_walk_d<2, true>(p, wide, smem, grid, warps * 32, st) : launch_walk_d<2, false>(p, wide, smem, grid, warps * 32, st);
        case 3: return ch ? launch_walk_d<3, true>(p, wide, smem, grid, warps * 32, st) : launch_walk_d<3, false>(p, wide, smem, grid, warps * 32, st);
        case 4: return ch ? launch_walk_d<4, true>(p, wide, smem, grid, warps * 32, st) : launch_walk_d<4, false>(p, wide, smem, grid, warps * 32, st);
    }
    set_error("unsupported number of defs %u", p.n_defs);
    return B2R_ERR_UNSUPPORTED;
}

int launch_emit(const WalkParams& p, bool wide, void* stream, LaunchInfo* chosen) {
    int n_sm = 0, max_smem = 0;
    int rc = device_limits(&n_sm, &max_smem);
    if (rc) return rc;
    const size_t smem = ((emit_smem_bytes(p) + 15u) & ~15u) + emit_scratch_bytes(p, wide ? 2 : 1);   // tables + endpoint counters, granule scratch
    const int wpc = EMIT_THREADS / 32;
    int per_sm = 2048 / EMIT_THREADS;
    { const int by_smem = (int)((size_t)max_smem / (smem + EMIT_ZERO_BYTES + 1024)); if (by_smem < per_sm) per_sm = by_smem < 1 ? 1 : by_smem; }   // + the static zero buffer
    const long long want = ((long long)p.n_tiles + wpc - 1) / wpc;   // one warp per tile of 32 strings
    long long grid = (long long)n_sm * per_sm;
    if (grid > want) grid = want > 0 ? want : 1;
    if (chosen) { chosen->grid = (int)grid; chosen->block = EMIT_THREADS; chosen->smem_bytes = smem; }
    cudaStream_t st = (cudaStream_t)stream;
    switch (p.n_defs) {
        case 1: return launch_emit_d<1>(p, wide, smem, (int)grid, st);
        case 2: return launch_emit_d<2>(p, wide, smem, (int)grid, st);
        case 3: return launch_emit_d<3>(p, wide, smem, (int)grid, st);
        case 4: return launch_emit_d<4>(p, wide, smem, (int)grid, st);
    }
    set_error("unsupported number of defs %u", p.n_defs);
    return B2R_ERR_UNSUPPORTED;
}

int launch_finalize(const FinalizeParams& p, void* stream) {
    finalize_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("finalize_kernel launch: %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    return B2R_OK;
}

int launch_diagnose(const WalkParams& p, uint64_t string_idx, b2r_batch_status* d_out, void* stream) {
    diagnose_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(p, string_idx, d_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("diagnose_kernel launch: %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    return B2R_OK;
}

}  // namespace b2r
