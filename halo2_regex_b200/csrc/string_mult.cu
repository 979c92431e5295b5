// Per-string lookup multiplicities (include/b2r.h, b2r_string_mult): a post-pass over the state columns the match kernels wrote.
//
// Row i < len of def d looks up table row row(bytes[i], states[d][i]), a bijection from the bin ch*S + cur onto the rows >= 1
// (defs.cpp, row_bin); rows i >= len look up row 0.  The endpoint rows follow from the packed transition entry of (byte, state).
// So once the walk has written the states there is no dependent chain left: every position is independent, and counting one
// string is a histogram over its distinct bins.
//
//   string_mult_kernel          one warp per segment (<= SEG positions of one string): bins counted in a per-warp open-addressing
//                               table in shared memory (warp-aggregated: lanes holding the same bin add once), then each distinct
//                               bin mapped to its row by binary search in the sorted (bin, row) table of the handle.  A string of
//                               one segment is sorted by row in the warp (bitonic) and written out; a longer string adds its
//                               distinct rows into a dense per-string workspace of u32 counters.
//   string_mult_compact_kernel  one CTA per string of several segments: the workspace row counters -> ascending entries.
//
// Packed layout (b2r_string_mult_packed): the two kernels above write every list whole into a slot workspace, then per pass
//   string_mult_scan_kernel     one CTA per def: exclusive prefix of the list lengths -> row_start, carried across passes in device memory
//   string_mult_pack_kernel     one warp per string: a list that fits below the capacity moves from its slots to entries + row_start[j]
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "config.hpp"

namespace b2r {
namespace {

constexpr uint32_t SEG = 4096;            // positions per work unit: 2^20 x 1 KiB and 2^17 x 4 KiB strings are one unit each
constexpr uint32_t EMPTY = 0xFFFFFFFFu;
constexpr int MAX_WARPS = 4;              // warps per CTA (fewer when the tables of a large DFA take the shared memory): small CTAs pack the SM
constexpr int COMPACT_THREADS = 256;
constexpr uint64_t WS_CAP = 256ull << 20; // bytes of per-string counters per pass (strings longer than SEG)

struct SmDef {
    const uint8_t* byte_class;
    const uint32_t* trans;                // [num_classes][S] packed entries (defs.hpp)
    const uint32_t* sorted_bins;          // [T - 1] ascending
    const uint32_t* sorted_rows;          // [T - 1] the row of each
    const uint32_t *erow_start_bin, *erow_end_bin;   // [E] (0xFFFFFFFF: shadowed row, receives 0)
    uint32_t S, n_rows, n_erows, sid_offset;
    const void* states;                   // this pass's first string
    b2r_row_count* entries;
    uint32_t* n_entries;
    uint32_t* ep;                         // [n][2E]
    uint32_t* ws_rows;                    // several segments: [n][T] row counters
    uint32_t* ws_ep;                      //                   [n][2E]
};

struct SmParams {
    const uint8_t* bytes;
    const uint64_t* offsets;              // of this pass's first string
    const b2r_string_status* status;      // of this pass's first string
    uint64_t n, row_pitch;
    uint32_t M, units_per_string, n_defs, wide, max_entries, slots_log2, ep_words;
    SmDef def[B2R_MAX_DEFS];
};

__device__ __forceinline__ uint32_t bin_to_row(const SmDef& f, uint32_t bin) {
    uint32_t lo = 0, hi = f.n_rows - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(f.sorted_bins + mid) < bin) lo = mid + 1; else hi = mid;
    }
    return (lo < f.n_rows - 1 && __ldg(f.sorted_bins + lo) == bin) ? __ldg(f.sorted_rows + lo) : EMPTY;
}

__device__ __forceinline__ uint32_t find_erow(const uint32_t* bins, uint32_t n, uint32_t bin) {
    for (uint32_t r = 1; r < n; r++) if (__ldg(bins + r) == bin) return r;
    return EMPTY;
}

// The table has at least twice as many slots as a segment of a string of at most M - 1 bytes has distinct bins.  The probe count is
// bounded all the same: state columns that are not the ones the match wrote (a contract violation) give wrong counts, never a hang.
__device__ __forceinline__ void insert(uint32_t* keys, uint32_t* cnts, uint32_t key, uint32_t add, uint32_t log2) {
    const uint32_t mask = (1u << log2) - 1u;
    uint32_t h = (key * 2654435761u) >> (32 - log2);
    for (uint32_t probe = 0; probe <= mask; probe++) {
        uint32_t k = ((volatile uint32_t*)keys)[h];
        if (k == EMPTY) { k = atomicCAS(keys + h, EMPTY, key); if (k == EMPTY) k = key; }
        if (k == key) { atomicAdd(cnts + h, add); return; }
        h = (h + 1) & mask;
    }
}

// Strings that count nothing: flagged invalid or too long by the match call, or longer than M - 1 for the M of THIS call (a post-pass
// given a smaller M than the match used, e.g. the handle's M after b2r_match_long) — the same rule the match applies to its own M
__device__ __forceinline__ bool skipped(const SmParams& p, uint64_t j, uint64_t& len) {
    len = p.offsets[j + 1] - p.offsets[j];                                // decreasing offsets wrap to a huge length: skipped as well
    return (p.status[j].flags & (B2R_ST_INVALID_TRANSITION | B2R_ST_TOO_LONG)) != 0 || len >= (uint64_t)p.M;
}

__global__ void string_mult_kernel(const __grid_constant__ SmParams p) {
    extern __shared__ uint32_t smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t slots = 1u << p.slots_log2;
    uint32_t* const keys = smem + warp * (2 * slots + p.ep_words);
    uint32_t* const cnts = keys + slots;
    uint32_t* const ep = cnts + slots;
    const unsigned below = (1u << lane) - 1u;
    const uint64_t n_units = p.n * p.units_per_string;
    for (uint64_t u = (uint64_t)blockIdx.x * n_warps + warp; u < n_units; u += (uint64_t)gridDim.x * n_warps) {
        const uint64_t j = u / p.units_per_string;
        const uint32_t s = (uint32_t)(u % p.units_per_string);
        uint64_t len;
        if (skipped(p, j, len)) {                                         // counts nothing (the reference panics on such a string)
            if (s == 0)
                for (uint32_t d = 0; d < p.n_defs; d++) {
                    const SmDef& f = p.def[d];
                    if (f.n_entries && lane == 0) f.n_entries[j] = 0;
                    if (f.ep) for (uint32_t r = lane; r < 2 * f.n_erows; r += 32) f.ep[j * 2 * f.n_erows + r] = 0;
                }
            continue;
        }
        const uint64_t off = p.offsets[j];
        const uint64_t lo = (uint64_t)s * SEG;
        if (s > 0 && lo >= len) continue;                                 // segment 0 always runs: an empty string has its row-0 entry
        const uint64_t hi = len < lo + SEG ? len : lo + SEG;
        const bool multi = len > SEG;
        const uint8_t* const b = p.bytes + off;
        for (uint32_t d = 0; d < p.n_defs; d++) {
            const SmDef& f = p.def[d];
            if (!f.n_entries && !f.ep) continue;
            const uint32_t S = f.S, E = f.n_erows;
            for (uint32_t i = lane; i < slots; i += 32) { keys[i] = EMPTY; cnts[i] = 0; }
            for (uint32_t i = lane; i < 2 * E; i += 32) ep[i] = 0;
            __syncwarp();
            const uint8_t* const st8 = (const uint8_t*)f.states + j * p.row_pitch;
            const uint16_t* const st16 = (const uint16_t*)f.states + j * p.row_pitch;
            for (uint64_t i0 = lo; i0 < hi; i0 += 32) {
                const uint64_t i = i0 + lane;
                const uint32_t key = i < hi ? (uint32_t)__ldg(b + i) * S + (p.wide ? (uint32_t)__ldg(st16 + i) : (uint32_t)__ldg(st8 + i)) : EMPTY;
                const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
                if (key != EMPTY && lane == (uint32_t)__ffs(peers) - 1u) insert(keys, cnts, key, (uint32_t)__popc(peers), p.slots_log2);
            }
            __syncwarp();
            // the distinct bins to the front of the table, in place (slot k of the list is never after the slot it came from, and every
            // lane has read its slot before anyone writes), then bins -> rows (and endpoint rows) over the list only: the binary searches
            // are dependent loads, so they run on full warps
            uint32_t n_list = 0;
            for (uint32_t s0 = 0; s0 < slots; s0 += 32) {
                const uint32_t k = keys[s0 + lane], c = cnts[s0 + lane];
                __syncwarp();
                const unsigned m = __ballot_sync(0xFFFFFFFFu, k != EMPTY);
                if (k != EMPTY) { const uint32_t at = n_list + (uint32_t)__popc(m & below); keys[at] = k; cnts[at] = c; }
                n_list += (uint32_t)__popc(m);
            }
            __syncwarp();
            for (uint32_t t = lane; t < n_list; t += 32) {
                const uint32_t k = keys[t], c = cnts[t];
                const uint32_t row = bin_to_row(f, k);
                if (f.ep) {
                    const uint32_t ch = k / S, st = k - ch * S;
                    const uint32_t e = __ldg(f.trans + (size_t)__ldg(f.byte_class + ch) * S + st);
                    const uint32_t sub = ((e & ENT_SID_MASK) >> ENT_SID_SHIFT) - f.sid_offset;
                    if (e & ENT_IS_START) { const uint32_t r = find_erow(f.erow_start_bin, E, sub * S + st); if (r != EMPTY) atomicAdd(ep + r, c); }
                    if (e & ENT_IS_END) { const uint32_t r = find_erow(f.erow_end_bin, E, sub * S + (e & ENT_NEXT_MASK)); if (r != EMPTY) atomicAdd(ep + E + r, c); }
                }
                if (multi) { if (row != EMPTY && f.n_entries) atomicAdd(f.ws_rows + j * f.n_rows + row, c); }
                else keys[t] = row;                                       // (every bin of an unflagged string has its row)
            }
            __syncwarp();
            if (multi) {
                if (f.ep) for (uint32_t r = lane; r < 2 * E; r += 32) if (ep[r]) atomicAdd(f.ws_ep + j * 2 * E + r, ep[r]);
                __syncwarp();
                continue;
            }
            if (f.n_entries) {
                // bitonic sort of the list by row (pads sort last); n_list <= slots / 2
                uint32_t P = 1;
                while (P < n_list) P <<= 1;
                for (uint32_t i = n_list + lane; i < P; i += 32) keys[i] = EMPTY;
                __syncwarp();
                for (uint32_t k = 2; k <= P; k <<= 1)
                    for (uint32_t h = k >> 1; h > 0; h >>= 1) {
                        for (uint32_t i = lane; i < P; i += 32) {
                            const uint32_t x = i ^ h;
                            if (x > i) {
                                const uint32_t a = keys[i], bb = keys[x];
                                if ((a > bb) == ((i & k) == 0)) { keys[i] = bb; keys[x] = a; const uint32_t t = cnts[i]; cnts[i] = cnts[x]; cnts[x] = t; }
                            }
                        }
                        __syncwarp();
                    }
                if (lane == 0) f.n_entries[j] = n_list + 1;
                if (f.entries) {
                    b2r_row_count* const out = f.entries + j * p.max_entries;
                    const uint32_t ne = n_list + 1 < p.max_entries ? n_list + 1 : p.max_entries;
                    for (uint32_t t = lane; t < ne; t += 32)
                        *reinterpret_cast<uint2*>(out + t) = t == 0 ? make_uint2(0u, p.M - (uint32_t)len) : make_uint2(keys[t - 1], cnts[t - 1]);
                }
            }
            if (f.ep) {
                uint32_t ts = 0, te = 0;
                for (uint32_t r = 1 + lane; r < E; r += 32) { ts += ep[r]; te += ep[E + r]; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { ts += __shfl_xor_sync(0xFFFFFFFFu, ts, o); te += __shfl_xor_sync(0xFFFFFFFFu, te, o); }
                uint32_t* const out = f.ep + j * 2 * E;
                for (uint32_t r = lane; r < 2 * E; r += 32)
                    out[r] = r == 0 ? p.M - ts : r == E ? p.M - te : ep[r];    // every other row of the string looks up endpoint row 0
            }
            __syncwarp();
        }
    }
}

// one CTA per string longer than SEG: its dense row counters in ascending row order -> entries
__global__ void __launch_bounds__(COMPACT_THREADS) string_mult_compact_kernel(const __grid_constant__ SmParams p) {
    __shared__ uint32_t s_warp[COMPACT_THREADS / 32];
    __shared__ uint32_t s_tot[2];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t j = blockIdx.x; j < p.n; j += gridDim.x) {
        uint64_t len;
        if (skipped(p, j, len) || len <= SEG) continue;                  // written by string_mult_kernel
        for (uint32_t d = 0; d < p.n_defs; d++) {
            const SmDef& f = p.def[d];
            if (f.n_entries) {
                const uint32_t* const w = f.ws_rows + j * f.n_rows;
                b2r_row_count* const out = f.entries ? f.entries + j * p.max_entries : nullptr;
                uint32_t base = 1;                                        // entry 0: row 0
                for (uint32_t r0 = 1; r0 < f.n_rows; r0 += COMPACT_THREADS) {
                    const uint32_t r = r0 + threadIdx.x;
                    const uint32_t v = r < f.n_rows ? w[r] : 0u;
                    const unsigned m = __ballot_sync(0xFFFFFFFFu, v != 0);
                    if (lane == 0) s_warp[warp] = (uint32_t)__popc(m);
                    __syncthreads();
                    uint32_t before = 0, total = 0;
                    for (uint32_t k = 0; k < COMPACT_THREADS / 32; k++) { if (k < warp) before += s_warp[k]; total += s_warp[k]; }
                    const uint32_t at = base + before + (uint32_t)__popc(m & ((1u << lane) - 1u));
                    if (v && out && at < p.max_entries) *reinterpret_cast<uint2*>(out + at) = make_uint2(r, v);
                    base += total;
                    __syncthreads();
                }
                if (threadIdx.x == 0) {
                    f.n_entries[j] = base;
                    if (out && p.max_entries) *reinterpret_cast<uint2*>(out) = make_uint2(0u, p.M - (uint32_t)len);
                }
            }
            if (f.ep) {
                const uint32_t E = f.n_erows;
                const uint32_t* const w = f.ws_ep + j * 2 * E;
                uint32_t* const out = f.ep + j * 2 * E;
                if (threadIdx.x == 0) { s_tot[0] = 0; s_tot[1] = 0; }
                __syncthreads();
                for (uint32_t r = threadIdx.x; r < 2 * E; r += COMPACT_THREADS)
                    if (r != 0 && r != E) { out[r] = w[r]; if (w[r]) atomicAdd(&s_tot[r >= E], w[r]); }
                __syncthreads();
                if (threadIdx.x == 0) { out[0] = p.M - s_tot[0]; out[E] = p.M - s_tot[1]; }
                __syncthreads();
            }
        }
    }
}

// ---- packed layout (b2r_string_mult_packed): count into slots, then scan the counts and pack the lists back to back -------------
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 8;             // counts per thread and tile: 8192 strings per tile, 128 tiles for 2^20 strings
constexpr int PACK_THREADS = 256;

struct PkDef {
    const uint32_t* counts;               // this pass's strings: distinct rows (string_mult_kernel's n_entries)
    const b2r_row_count* slots;           // [np][slot_pitch], or NULL: offsets only
    b2r_row_count* entries;               // the caller's packed area
    uint64_t* row_start;                  // of the CALL's string 0: this pass writes [j0, j0 + np]
};

struct PkParams {
    uint64_t np, j0, capacity, slot_pitch;
    uint64_t* carry;                      // [n_defs] entries of the earlier passes (device memory: no host round trip between passes)
    uint64_t* host_total;                 // [n_defs] pinned host memory, or NULL: the running total after this pass
    uint32_t n_defs;
    PkDef def[B2R_MAX_DEFS];
};

// one CTA per def: the exclusive prefix of the pass's counts in tiles of SCAN_THREADS * SCAN_ITEMS, carried across tiles in a
// register and across passes in `carry`.  One CTA streams 2^20 counts in well under a millisecond, against tens of milliseconds
// of counting before it: a multi-CTA scan would buy nothing worth its second kernel
__global__ void __launch_bounds__(SCAN_THREADS) string_mult_scan_kernel(const __grid_constant__ PkParams p) {
    __shared__ uint64_t s_warp[SCAN_THREADS / 32];
    const PkDef& f = p.def[blockIdx.x];
    if (!f.row_start) return;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t carry = p.carry[blockIdx.x];
    uint64_t* const out = f.row_start + p.j0;
    constexpr uint64_t TILE = (uint64_t)SCAN_THREADS * SCAN_ITEMS;
    for (uint64_t t0 = 0; t0 < p.np; t0 += TILE) {
        const uint64_t first = t0 + (uint64_t)threadIdx.x * SCAN_ITEMS;
        uint32_t v[SCAN_ITEMS];
        uint64_t mine = 0;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = first + k < p.np ? f.counts[first + k] : 0u; mine += v[k]; }
        uint64_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint64_t x = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= (uint32_t)o) incl += x; }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint64_t before = 0, tile = 0;
        for (uint32_t w = 0; w < SCAN_THREADS / 32; w++) { const uint64_t x = s_warp[w]; if (w < warp) before += x; tile += x; }
        uint64_t at = carry + before + incl - mine;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) { if (first + k < p.np) out[first + k] = at; at += v[k]; }
        carry += tile;
        __syncthreads();                                                  // s_warp is reused by the next tile
    }
    if (threadIdx.x == 0) {
        out[p.np] = carry;                                                // the next pass overwrites it with the same value
        p.carry[blockIdx.x] = carry;
        if (p.host_total) p.host_total[blockIdx.x] = carry;
    }
}

// one warp per (def, string): a list that fits whole below `capacity` moves from its slots to entries + row_start[j], 8 bytes a lane
__global__ void __launch_bounds__(PACK_THREADS) string_mult_pack_kernel(const __grid_constant__ PkParams p) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_units = p.np * p.n_defs;
    for (uint64_t u = ((uint64_t)blockIdx.x * PACK_THREADS + threadIdx.x) >> 5; u < n_units; u += ((uint64_t)gridDim.x * PACK_THREADS) >> 5) {
        const PkDef& f = p.def[u / p.np];
        const uint64_t j = u % p.np;
        if (!f.slots) continue;
        const uint32_t cnt = f.counts[j];
        const uint64_t start = f.row_start[p.j0 + j];
        if (!cnt || start + cnt > p.capacity) continue;                  // no string is stored in part
        const uint2* src = reinterpret_cast<const uint2*>(f.slots + j * p.slot_pitch);
        uint2* dst = reinterpret_cast<uint2*>(f.entries + start);
        for (uint32_t t = lane; t < cnt; t += 32) dst[t] = __ldcs(src + t);
    }
}

}  // namespace

bool string_mult_wanted(const b2r_config* c, const b2r_string_mult_outputs* sm, uint32_t d) {
    return sm && d < c->n_defs && (sm->entries[d] || sm->n_entries[d] || sm->endpoint_counts[d]);
}

int check_string_mult(const b2r_config* c, const b2r_string_mult_outputs* sm) {
    if (!sm) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (sm->entries[d] && !sm->n_entries[d]) { set_error("def %u: entries without n_entries", d); return B2R_ERR_INVALID_ARG; }
        if (sm->entries[d] && sm->max_entries == 0) { set_error("def %u: entries with max_entries = 0", d); return B2R_ERR_INVALID_ARG; }
    }
    for (uint32_t d = 0; d < c->n_defs; d++)
        if ((reinterpret_cast<uintptr_t>(sm->entries[d]) & 7) || (reinterpret_cast<uintptr_t>(sm->n_entries[d]) & 3) ||
            (reinterpret_cast<uintptr_t>(sm->endpoint_counts[d]) & 3)) {
            set_error("def %u: entries must be 8-byte aligned, n_entries and endpoint_counts 4-byte aligned", d);
            return B2R_ERR_ALIGNMENT;
        }
    return B2R_OK;
}

int string_mult_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t M, void* const* states,
                     uint64_t row_pitch, const b2r_string_status* status, const b2r_string_mult_outputs* sm, cudaStream_t st, uint32_t* launches) {
    bool any = false;
    for (uint32_t d = 0; d < c->n_defs; d++) any = any || string_mult_wanted(c, sm, d);
    if (!n || !any) return B2R_OK;
    SmParams p;
    memset(&p, 0, sizeof p);
    p.bytes = d_bytes; p.row_pitch = row_pitch; p.M = (uint32_t)M; p.n_defs = c->n_defs; p.max_entries = sm->max_entries;
    p.units_per_string = M - 1 > SEG ? (uint32_t)((M - 1 + SEG - 1) / SEG) : 1u;
    const bool multi = p.units_per_string > 1;
    uint64_t max_t = 1, per_str = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!string_mult_wanted(c, sm, d)) continue;
        const PackedDef& pd = c->packed[d];
        p.wide = p.wide || pd.state_width == 2;
        max_t = std::max<uint64_t>(max_t, pd.rows.size());
        p.ep_words = std::max<uint32_t>(p.ep_words, 2 * (uint32_t)pd.erows.size());
        per_str += (pd.rows.size() + 2 * pd.erows.size()) * 4;
    }
    // a segment has at most min(SEG, M - 1, T - 1) distinct bins: a table of twice that keeps the probes short and holds the sorted list
    const uint64_t max_distinct = std::max<uint64_t>(1, std::min<uint64_t>({(uint64_t)SEG, M - 1, max_t - 1}));
    p.slots_log2 = 6;
    while ((1ull << p.slots_log2) < 2 * max_distinct) p.slots_log2++;
    p.ep_words = (p.ep_words + 3) & ~3u;
    const size_t per_warp = ((size_t)2 * (1u << p.slots_log2) + p.ep_words) * 4;
    int n_sm = 0, max_smem = 0, rc;
    if ((rc = device_limits(&n_sm, &max_smem))) return rc;
    const int warps = (int)std::min<size_t>(MAX_WARPS, (size_t)max_smem / per_warp);
    if (warps < 1) { set_error("string_mult: %zu bytes of shared memory per warp needed, %d available", per_warp, max_smem); return B2R_ERR_UNSUPPORTED; }
    const size_t smem = per_warp * warps;
    CUDA_TRY(cudaFuncSetAttribute(string_mult_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, string_mult_kernel, warps * 32, smem));
    per_sm = std::max(per_sm, 1);
    const uint64_t cap = c->opt.chunked_max_maps > 0 ? (uint64_t)c->opt.chunked_max_maps : WS_CAP;
    const uint64_t per_pass = multi ? std::min<uint64_t>(n, std::max<uint64_t>(1, cap / std::max<uint64_t>(per_str, 1))) : n;
    if (multi && (rc = c->ws_smult.reserve(per_pass * per_str))) return rc;
    for (uint64_t j0 = 0; j0 < n; j0 += per_pass) {
        const uint64_t np = std::min(per_pass, n - j0);
        p.n = np; p.offsets = d_offsets + j0; p.status = status + j0;
        size_t ws_off = 0;
        for (uint32_t d = 0; d < c->n_defs; d++) {
            SmDef& f = p.def[d];
            memset(&f, 0, sizeof f);
            if (!string_mult_wanted(c, sm, d)) continue;
            const PackedDef& pd = c->packed[d];
            f.byte_class = c->dev[d].byte_class; f.trans = c->dev[d].trans;
            f.sorted_bins = c->dev[d].sorted_bins; f.sorted_rows = c->dev[d].sorted_rows;
            f.erow_start_bin = c->dev[d].erow_start_bin; f.erow_end_bin = c->dev[d].erow_end_bin;
            f.S = pd.num_states; f.n_rows = (uint32_t)pd.rows.size(); f.n_erows = (uint32_t)pd.erows.size(); f.sid_offset = pd.substr_id_offset;
            f.states = (const unsigned char*)states[d] + j0 * row_pitch * (p.wide ? 2 : 1);
            f.entries = sm->entries[d] ? sm->entries[d] + j0 * sm->max_entries : nullptr;
            f.n_entries = sm->n_entries[d] ? sm->n_entries[d] + j0 : nullptr;
            f.ep = sm->endpoint_counts[d] ? sm->endpoint_counts[d] + j0 * 2 * f.n_erows : nullptr;
            if (multi) {
                unsigned char* ws = (unsigned char*)c->ws_smult.p;
                f.ws_rows = (uint32_t*)(ws + ws_off); ws_off += np * f.n_rows * 4;
                f.ws_ep = (uint32_t*)(ws + ws_off); ws_off += np * 2 * f.n_erows * 4;
            }
        }
        if (multi) CUDA_TRY(cudaMemsetAsync(c->ws_smult.p, 0, ws_off, st));
        const uint64_t want = (np * p.units_per_string + warps - 1) / warps;
        const int grid = (int)std::min<uint64_t>(want, (uint64_t)n_sm * per_sm);
        string_mult_kernel<<<grid, warps * 32, smem, st>>>(p);
        CUDA_TRY(cudaGetLastError());
        (*launches)++;
        if (multi) {
            string_mult_compact_kernel<<<(int)std::min<uint64_t>(np, (uint64_t)n_sm * 8), COMPACT_THREADS, 0, st>>>(p);
            CUDA_TRY(cudaGetLastError());
            (*launches)++;
        }
    }
    return B2R_OK;
}

// ---- packed layout ----------------------------------------------------------------------------------------------------------------
bool string_mult_packed_wanted(const b2r_config* c, const b2r_string_mult_packed_outputs* pk, uint32_t d) {
    return pk && d < c->n_defs && (pk->entries[d] || pk->row_start[d] || pk->endpoint_counts[d]);
}

int check_string_mult_packed(const b2r_config* c, const b2r_string_mult_packed_outputs* pk) {
    if (!pk) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    for (uint32_t d = 0; d < c->n_defs; d++)
        if (pk->entries[d] && !pk->row_start[d]) { set_error("def %u: entries without row_start", d); return B2R_ERR_INVALID_ARG; }
    for (uint32_t d = 0; d < c->n_defs; d++)
        if ((reinterpret_cast<uintptr_t>(pk->entries[d]) & 7) || (reinterpret_cast<uintptr_t>(pk->row_start[d]) & 7) ||
            (reinterpret_cast<uintptr_t>(pk->endpoint_counts[d]) & 3)) {
            set_error("def %u: entries and row_start must be 8-byte aligned, endpoint_counts 4-byte aligned", d);
            return B2R_ERR_ALIGNMENT;
        }
    return B2R_OK;
}

namespace {

// How a packed call over n strings runs: the counting kernels write each string's list into `pitch` = max_d min(M, T_d) slots
// (never truncated) and its length into a u32, for `per_pass` strings at a time; scan and pack follow each pass
struct PkShape {
    bool scan = false;                    // some def wants offsets (else: endpoint counts only, one slot-less string_mult_impl call)
    uint64_t pitch = 0, per_pass = 0, ws_bytes = 0;
    size_t counts_off[B2R_MAX_DEFS] = {}, slots_off[B2R_MAX_DEFS] = {};
};

constexpr size_t PK_CARRY_BYTES = 256;    // [n_defs] u64 running totals at the front of ws_smpk

PkShape pk_shape(const b2r_config* c, const b2r_string_mult_packed_outputs* pk, uint64_t n, uint64_t M) {
    PkShape s;
    uint64_t per_str = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!pk->row_start[d]) continue;
        s.scan = true;
        per_str += 4;
        if (pk->entries[d] && pk->capacity) s.pitch = std::max<uint64_t>(s.pitch, std::min<uint64_t>(M, c->packed[d].rows.size()));
    }
    if (!s.scan) return s;
    for (uint32_t d = 0; d < c->n_defs; d++) if (pk->row_start[d] && pk->entries[d] && pk->capacity) per_str += s.pitch * 8;
    const uint64_t cap = c->opt.chunked_max_maps > 0 ? (uint64_t)c->opt.chunked_max_maps : WS_CAP;
    s.per_pass = std::max<uint64_t>(1, std::min<uint64_t>(n, cap / per_str));
    size_t off = PK_CARRY_BYTES;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!pk->row_start[d]) continue;
        s.counts_off[d] = off; off += align_up(s.per_pass * 4, 256);
        if (pk->entries[d] && pk->capacity) { s.slots_off[d] = off; off += align_up(s.per_pass * s.pitch * 8, 256); }
    }
    s.ws_bytes = off;
    return s;
}

// the slot-call outputs that a packed call hands to string_mult_impl (pointers into ws_smpk; endpoint counts: the caller's)
b2r_string_mult_outputs pk_slot_outputs(const b2r_config* c, const b2r_string_mult_packed_outputs* pk, const PkShape& s, uint64_t j0) {
    b2r_string_mult_outputs sm{};
    sm.max_entries = (uint32_t)std::max<uint64_t>(1, s.pitch);
    unsigned char* ws = (unsigned char*)c->ws_smpk.p;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (pk->row_start[d]) sm.n_entries[d] = (uint32_t*)(ws + s.counts_off[d]);
        if (pk->row_start[d] && pk->entries[d] && pk->capacity) sm.entries[d] = (b2r_row_count*)(ws + s.slots_off[d]);
        if (pk->endpoint_counts[d]) sm.endpoint_counts[d] = pk->endpoint_counts[d] + j0 * 2 * c->packed[d].erows.size();
    }
    return sm;
}

}  // namespace

int string_mult_packed_reserve(b2r_config* c, uint64_t n, uint64_t M, const b2r_string_mult_packed_outputs* pk) {
    const PkShape s = pk_shape(c, pk, n, M);
    int rc;
    if (s.scan && (rc = c->ws_smpk.reserve(s.ws_bytes))) return rc;
    // the per-string counters of strings longer than one segment, as string_mult_impl sizes them for a pass of per_pass strings
    if (M - 1 > SEG) {
        const b2r_string_mult_outputs sm = s.scan ? pk_slot_outputs(c, pk, s, 0) : b2r_string_mult_outputs{};
        uint64_t per_str = 0;
        for (uint32_t d = 0; d < c->n_defs; d++)
            if (string_mult_wanted(c, &sm, d) || pk->endpoint_counts[d]) per_str += (c->packed[d].rows.size() + 2 * c->packed[d].erows.size()) * 4;
        const uint64_t cap = c->opt.chunked_max_maps > 0 ? (uint64_t)c->opt.chunked_max_maps : WS_CAP;
        const uint64_t m = s.scan ? s.per_pass : n;
        if (per_str && (rc = c->ws_smult.reserve(std::min<uint64_t>(m, std::max<uint64_t>(1, cap / per_str)) * per_str))) return rc;
    }
    return B2R_OK;
}

int string_mult_packed_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t M, void* const* states,
                            uint64_t row_pitch, const b2r_string_status* status, const b2r_string_mult_packed_outputs* pk, uint64_t* host_total,
                            cudaStream_t st, uint32_t* launches) {
    bool any = false;
    for (uint32_t d = 0; d < c->n_defs; d++) any = any || string_mult_packed_wanted(c, pk, d);
    if (!any) return B2R_OK;
    if (!n) {                                                             // row_start = {0}
        for (uint32_t d = 0; d < c->n_defs; d++) if (pk->row_start[d]) CUDA_TRY(cudaMemsetAsync(pk->row_start[d], 0, 8, st));
        if (host_total) for (uint32_t d = 0; d < c->n_defs; d++) host_total[d] = 0;
        return B2R_OK;
    }
    const PkShape s = pk_shape(c, pk, n, M);
    if (!s.scan) {                                                        // endpoint counts only: the slot call does it all
        const b2r_string_mult_outputs sm = pk_slot_outputs(c, pk, s, 0);
        return string_mult_impl(c, d_bytes, d_offsets, n, M, states, row_pitch, status, &sm, st, launches);
    }
    int rc;
    if ((rc = string_mult_packed_reserve(c, n, M, pk))) return rc;
    int n_sm = 0, max_smem = 0;
    if ((rc = device_limits(&n_sm, &max_smem))) return rc;
    unsigned char* const ws = (unsigned char*)c->ws_smpk.p;
    PkParams p;
    memset(&p, 0, sizeof p);
    p.capacity = pk->capacity; p.slot_pitch = s.pitch; p.carry = (uint64_t*)ws; p.host_total = host_total; p.n_defs = c->n_defs;
    bool pack = false;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        PkDef& f = p.def[d];
        if (!pk->row_start[d]) continue;
        f.counts = (const uint32_t*)(ws + s.counts_off[d]);
        f.row_start = pk->row_start[d];
        if (pk->entries[d] && pk->capacity) { f.slots = (const b2r_row_count*)(ws + s.slots_off[d]); f.entries = pk->entries[d]; pack = true; }
    }
    CUDA_TRY(cudaMemsetAsync(p.carry, 0, c->n_defs * sizeof(uint64_t), st));
    for (uint64_t j0 = 0; j0 < n; j0 += s.per_pass) {
        const uint64_t np = std::min(s.per_pass, n - j0);
        const b2r_string_mult_outputs sm = pk_slot_outputs(c, pk, s, j0);
        void* sh[B2R_MAX_DEFS] = {};
        for (uint32_t d = 0; d < c->n_defs; d++)
            if (states[d]) sh[d] = (unsigned char*)states[d] + j0 * row_pitch * c->packed[d].state_width;
        if ((rc = string_mult_impl(c, d_bytes, d_offsets + j0, np, M, sh, row_pitch, status + j0, &sm, st, launches))) return rc;
        p.np = np; p.j0 = j0;
        string_mult_scan_kernel<<<c->n_defs, SCAN_THREADS, 0, st>>>(p);
        CUDA_TRY(cudaGetLastError());
        (*launches)++;
        if (pack) {
            const uint64_t warps = np * c->n_defs;
            const int grid = (int)std::min<uint64_t>((warps + PACK_THREADS / 32 - 1) / (PACK_THREADS / 32), (uint64_t)n_sm * 16);
            string_mult_pack_kernel<<<grid, PACK_THREADS, 0, st>>>(p);
            CUDA_TRY(cudaGetLastError());
            (*launches)++;
        }
    }
    return B2R_OK;
}

}  // namespace b2r

using namespace b2r;

extern "C" int b2r_string_mult(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes, uint64_t max_chars_size,
                               const b2r_outputs* o, const b2r_string_mult_outputs* sm, void* cuda_stream) {
    // the arguments are checked first (the same answer on any handle), then the device
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (!o || !sm || (n && !d_offsets) || (n && !d_bytes && total_bytes)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    const uint64_t M = max_chars_size ? max_chars_size : c->max_chars;
    if (M > 0xFFFFFFF0ull) { set_error("max_chars_size out of range"); return B2R_ERR_INVALID_ARG; }
    int rc = check_string_mult(c, sm);
    if (rc) return rc;
    bool any = false;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!string_mult_wanted(c, sm, d)) continue;
        any = true;
        if (!o->states[d]) { set_error("def %u: per-string counts need the state column the match call wrote", d); return B2R_ERR_INVALID_ARG; }
    }
    if (any && !o->status) { set_error("per-string counts need the status column the match call wrote"); return B2R_ERR_INVALID_ARG; }
    if ((rc = check_outputs(c, o, false, M))) return rc;
    if (c->multi) { set_error("b2r_string_mult takes device pointers of one device: a multi-device handle has no such call (use b2r_match_batch_host_mult)"); return B2R_ERR_INVALID_ARG; }
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    c->last_launches = 0;
    return string_mult_impl(c, d_bytes, d_offsets, n, M, o->states, o->row_pitch, o->status, sm, (cudaStream_t)cuda_stream, &c->last_launches);
}

extern "C" int b2r_string_mult_packed(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                                      uint64_t max_chars_size, const b2r_outputs* o, const b2r_string_mult_packed_outputs* pk, void* cuda_stream) {
    // the checks of b2r_string_mult, in the same order
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    if (!o || !pk || (n && !d_offsets) || (n && !d_bytes && total_bytes)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    const uint64_t M = max_chars_size ? max_chars_size : c->max_chars;
    if (M > 0xFFFFFFF0ull) { set_error("max_chars_size out of range"); return B2R_ERR_INVALID_ARG; }
    int rc = check_string_mult_packed(c, pk);
    if (rc) return rc;
    bool any = false;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!string_mult_packed_wanted(c, pk, d)) continue;
        any = true;
        if (!o->states[d]) { set_error("def %u: per-string counts need the state column the match call wrote", d); return B2R_ERR_INVALID_ARG; }
    }
    if (any && !o->status) { set_error("per-string counts need the status column the match call wrote"); return B2R_ERR_INVALID_ARG; }
    if ((rc = check_outputs(c, o, false, M))) return rc;
    if (c->multi) { set_error("b2r_string_mult_packed takes device pointers of one device: a multi-device handle has no such call (use b2r_match_batch_host_mult_packed)"); return B2R_ERR_INVALID_ARG; }
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    c->last_launches = 0;
    return string_mult_packed_impl(c, d_bytes, d_offsets, n, M, o->states, o->row_pitch, o->status, pk, nullptr, (cudaStream_t)cuda_stream, &c->last_launches);
}
