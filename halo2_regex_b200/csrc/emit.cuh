// Emit stage: everything the reference derives from the state sequence, for one tile of 32 consecutive strings per warp.
//
// Inputs: the strings, their state columns and granule flags (walk.cuh).  Outputs: per-def substr ids (src/lib.rs:825-845),
// start_enable / end_enable bitmaps (:482-513), the endpoint-lookup multiplicities (:235-284), masked_chars /
// masked_substr_ids (:740-764), substring records + compact bytes, the accept flag (:427-457) and the status record.
//
// Rule of the memory traffic: never write PART of a sector that was completely written earlier (L2 streams full sectors
// out early; a later partial write costs a DRAM read-modify-write).  Hence, per tile,
//   fill  (warp)          the tile's rows of every sparse column are contiguous: blanket zero-fill, coalesced 16-byte stores;
//   scan  (lane = string) each lane walks the flagged granules of ITS string in order: it rewrites the complete 32-byte
//                         sector of the substr-id columns (values and zeros merged in registers), collects the bitmap
//                         words, counts endpoint lookups and streams the boundaries of the mask algebra below, which
//                         yields the masked segments, their records and compact bytes;
//   masks (lane = string) rewrites the complete sectors of masked_chars / masked_substr_ids that a masked segment touches.
// A row's packed entries are looked up again from (byte, state): one lookup replaces the reference's HashSet probes and
// `contains` scans and gives substr id, is_start, is_end(next row).
//
// Masks.  With b_1 < b_2 < ... the rows where the id sum changes AND is_start_sum|is_end_sum is set, the forward scan
//         (src/lib.rs:598-645) sets start_mask at b_k when is_start_sum[b_k] and resets it when only is_end_sum[b_k]; the
//         backward scan (:663-714) sets end_mask for the rows before b_{k+1} when is_end_sum[b_{k+1}] and resets it when
//         only is_start_sum[b_{k+1}].  Hence mask = 1 exactly on [b_k, b_{k+1}) with is_start at b_k and is_end at b_{k+1}.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "defs.hpp"
#include "kernels.cuh"

namespace b2r {

constexpr uint32_t NO_POS = 0xFFFFFFFFu;
constexpr int EMIT_THREADS = 256;
constexpr int EMIT_NSEG = 4;       // masked segments per string kept in registers; further ones take the patch path

__device__ __forceinline__ uint32_t ent_sid(uint32_t e) { return (e >> ENT_SID_SHIFT) & 0xFFu; }

// Failure details of string j in the reference's order: derive_states walks def 0 over the whole string first, then
// def 1, ... (src/lib.rs:806-821), so the panic belongs to the LOWEST def index that fails, at its first failing byte.
static __device__ __noinline__ b2r_batch_status diagnose_string(const WalkParams& p, uint64_t j) {
    b2r_batch_status r = {};
    r.string_idx = j;
    const uint64_t off = p.offsets[j], end = p.offsets[j + 1];
    if (end < off || end - off > (uint64_t)(p.max_chars - 1) || end > p.total_bytes) {
        r.code = B2R_ERR_TOO_LONG; r.pos = NO_POS;
        return r;
    }
    for (uint32_t d = 0; d < p.n_defs && r.code == 0; d++) {
        uint32_t s = p.def[d].first_state;
        for (uint64_t i = off; i < end; i++) {
            const uint32_t c = p.bytes[i];
            const uint32_t e = p.def[d].trans[(uint32_t)p.def[d].byte_class[c] * p.def[d].num_states + s];
            if (e & ENT_INVALID) {
                r.code = B2R_ERR_INVALID_TRANSITION; r.pos = (uint32_t)(i - off); r.state = s; r.byte = (uint8_t)c; r.def = (uint8_t)d;
                break;
            }
            s = e & ENT_NEXT_MASK;
        }
    }
    return r;
}

// the reference panics (src/lib.rs:817) / the string does not fit: mark the string, remember the lowest failing index
static __device__ __noinline__ void kill_string(const WalkParams& p, uint64_t idx) {
    atomicMax(&p.counters->first_bad_inv, ~(unsigned long long)idx);
    if (p.status) {
        const b2r_batch_status r = diagnose_string(p, idx);
        b2r_string_status st = {};
        st.flags = (r.code == B2R_ERR_TOO_LONG) ? B2R_ST_TOO_LONG : B2R_ST_INVALID_TRANSITION;
        st.err_pos = (r.code == B2R_ERR_TOO_LONG) ? NO_POS : r.pos; st.err_state = r.state; st.err_byte = r.byte; st.err_def = r.def;
        p.status[idx] = st;
    }
}

// warp-cooperative zero-fill of a contiguous region; base 16-byte aligned, bytes a multiple of 4
__device__ __forceinline__ void emit_zero_region(uint8_t* base, uint64_t bytes, int lane) {
    if (!base) return;
    const uint32_t nv = (uint32_t)(bytes / 16);
    uint4* q = reinterpret_cast<uint4*>(base) + lane;
    const uint4 z = make_uint4(0, 0, 0, 0);
    uint32_t v = lane;
    for (; v + 96 < nv; v += 128, q += 128) { q[0] = z; q[32] = z; q[64] = z; q[96] = z; }
    for (; v < nv; v += 32, q += 32) q[0] = z;
    for (uint64_t o = (uint64_t)nv * 16 + (uint64_t)lane * 4; o < bytes; o += 128) *reinterpret_cast<uint32_t*>(base + o) = 0u;
}

// per-CTA view of the lookup tables (shared memory when they fit, else global) and the endpoint counters
template <int D>
struct EmitTables {
    const uint8_t* cls[D];
    const uint32_t* trans[D];
    uint32_t* ep_s[D];          // shared-memory endpoint counters: [0,K*S) start lookups, [K*S,2*K*S) end lookups; null = global
};

// per-lane running sums published once at the end of the kernel
struct EmitTotals {
    unsigned long long pad_rows = 0;
    uint32_t n_ok = 0, n_overlap = 0;
};

// Overflow path (a string with more than EMIT_NSEG masked segments): rows [a,b) of string j are masked
// (src/lib.rs:740-764), b <= len: masked_chars / masked_substr_ids byte by byte, the compact bytes and one record per
// maximal run of a constant id sum.  Lane-private.  Returns the updated (n_rec, n_cmp).
template <int D, typename ST>
static __device__ __noinline__ uint2 emit_segment(const WalkParams& p, const EmitTables<D> tb, uint64_t j, const uint8_t* src, uint32_t a, uint32_t b,
                                                  uint32_t n_rec, uint32_t n_cmp) {
    uint8_t* const mc = p.masked_chars ? p.masked_chars + j * p.row_pitch : nullptr;
    uint8_t* const ms = p.masked_substr_ids ? p.masked_substr_ids + j * p.row_pitch : nullptr;
    uint8_t* const cb = p.compact_bytes ? p.compact_bytes + j * (uint64_t)p.compact_pitch : nullptr;
    auto record = [&](uint32_t start, uint32_t len, uint32_t sid, uint32_t coff) {
        if (p.records && n_rec < p.max_records) {
            b2r_substr_record r; r.start = start; r.len = len; r.substr_id = sid; r.compact_off = coff;
            p.records[j * p.max_records + n_rec] = r;
        }
        n_rec++;
    };
    uint32_t run_start = a, run_sum = 0;
    for (uint32_t i = a; i < b; i++) {
        const uint32_t c = __ldg(src + i);
        uint32_t sum = 0;
#pragma unroll
        for (int d = 0; d < D; d++) {
            const uint32_t S = p.def[d].num_states;
            const uint32_t s = (uint32_t)__ldcg(reinterpret_cast<const ST*>(p.def[d].states) + j * p.row_pitch + i);
            if (s < S) sum += ent_sid(tb.trans[d][(uint32_t)tb.cls[d][c] * S + s]);
        }
        if (mc) mc[i] = (uint8_t)c;
        if (ms) ms[i] = (uint8_t)sum;
        const uint32_t k = n_cmp + (i - a);
        if (cb && k < p.compact_pitch) cb[k] = (uint8_t)c;
        if (i == a) run_sum = sum;
        else if (sum != run_sum) {                                       // records: maximal runs of a constant id sum
            record(run_start, i - run_start, run_sum, n_cmp + (run_start - a));
            run_start = i; run_sum = sum;
        }
    }
    record(run_start, b - run_start, run_sum, n_cmp + (run_start - a));
    return make_uint2(n_rec, n_cmp + (b - a));
}

// 16 rows of one string in registers: the bytes and the states of every def.
// SG (the stand-alone emit kernel): the granule is mirrored in a shared-memory scratch of the thread (vector v at gs + v * EMIT_SG_PITCH:
// the bytes, then the states of every def), so that a row chosen at run time costs one LDS instead of a chain of selects — the per-row
// loops of the scan are what that kernel spends its instructions on.
constexpr uint32_t EMIT_SG_PITCH = 256 * 16;   // EMIT_THREADS * 16 bytes: vector v of thread t lives at v * pitch + t * 16
template <int D, typename ST, bool SG = false>
struct Granule {
    uint32_t w[4];
    uint32_t sv[D][4 * sizeof(ST)];
    uint32_t n;                    // rows that are characters (1..16)
    uint32_t gs;                   // SG: shared-memory address of this thread's vector 0

    __device__ __forceinline__ void mirror() {
        if (!SG) return;
        auto sts = [](uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t q) { asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(q) : "memory"); };
        sts(gs, w[0], w[1], w[2], w[3]);
#pragma unroll
        for (int d = 0; d < D; d++) {
            sts(gs + (1 + d * (int)sizeof(ST)) * EMIT_SG_PITCH, sv[d][0], sv[d][1], sv[d][2], sv[d][3]);
            if (sizeof(ST) == 2) {
                constexpr int H = 4 * (sizeof(ST) - 1);
                sts(gs + (2 + d * (int)sizeof(ST)) * EMIT_SG_PITCH, sv[d][H], sv[d][H + 1], sv[d][H + 2], sv[d][H + 3]);
            }
        }
    }

    // granule g of string j (src = its first byte, L its length); 16*g < L
    // stash_g / stash_s: a granule of this string kept in shared memory by the walk (fused mode): vector v at stash_s + 512*v,
    // v = 0 the bytes, then the states of every def
    __device__ __forceinline__ void load(const WalkParams& p, uint64_t j, const uint8_t* src, uint32_t L, uint32_t g, uint32_t stash_g, uint32_t stash_s) {
        const uint32_t base = 16 * g;
        n = L - base < 16 ? L - base : 16;
        if (g == stash_g) {
            auto lds = [](uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v; };
            const uint4 b = lds(stash_s);
            w[0] = b.x; w[1] = b.y; w[2] = b.z; w[3] = b.w;
#pragma unroll
            for (int d = 0; d < D; d++) {
                const uint4 a = lds(stash_s + (1 + d * sizeof(ST)) * 512);
                sv[d][0] = a.x; sv[d][1] = a.y; sv[d][2] = a.z; sv[d][3] = a.w;
                if (sizeof(ST) == 2) { const uint4 b2 = lds(stash_s + (2 + d * sizeof(ST)) * 512); sv[d][4 * (sizeof(ST) - 1)] = b2.x; sv[d][4 * (sizeof(ST) - 1) + 1] = b2.y; sv[d][4 * (sizeof(ST) - 1) + 2] = b2.z; sv[d][4 * (sizeof(ST) - 1) + 3] = b2.w; }
            }
            mirror();
            return;
        }
        // 16 bytes from an arbitrary address: two aligned 16-byte loads shifted into place; the second one is only
        // touched when the bytes needed reach into it
        const uintptr_t addr = reinterpret_cast<uintptr_t>(src + base);
        const uint32_t sh = (uint32_t)(addr & 15);
        const uint4* q = reinterpret_cast<const uint4*>(addr - sh);
        const uint4 v0 = __ldg(q);
        uint4 v1 = make_uint4(0, 0, 0, 0);
        if (sh + n > 16) v1 = __ldg(q + 1);
        const uint32_t x[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        uint32_t y[7], z[5];
#pragma unroll
        for (int k = 0; k < 7; k++) y[k] = (sh & 4) ? x[k + 1] : x[k];
#pragma unroll
        for (int k = 0; k < 5; k++) z[k] = (sh & 8) ? y[k + 2] : y[k];
#pragma unroll
        for (int k = 0; k < 4; k++) w[k] = __funnelshift_r(z[k], z[k + 1], (sh & 3) * 8);
#pragma unroll
        for (int d = 0; d < D; d++) {   // written by the walk (possibly by this very kernel): L2-coherent loads
            const uint4* sp = reinterpret_cast<const uint4*>(reinterpret_cast<const ST*>(p.def[d].states) + j * p.row_pitch + base);
            const uint4 a = __ldcg(sp);
            sv[d][0] = a.x; sv[d][1] = a.y; sv[d][2] = a.z; sv[d][3] = a.w;
            if (sizeof(ST) == 2) { const uint4 b2 = __ldcg(sp + 1); sv[d][4 * (sizeof(ST) - 1)] = b2.x; sv[d][4 * (sizeof(ST) - 1) + 1] = b2.y; sv[d][4 * (sizeof(ST) - 1) + 2] = b2.z; sv[d][4 * (sizeof(ST) - 1) + 3] = b2.w; }
        }
        mirror();
    }
    // compile-time row index
    __device__ __forceinline__ uint32_t byte_at(int r) const { return (w[r >> 2] >> (8 * (r & 3))) & 0xFFu; }
    __device__ __forceinline__ uint32_t state_at(int d, int r) const {
        return sizeof(ST) == 1 ? (sv[d][r >> 2] >> (8 * (r & 3))) & 0xFFu : (sv[d][(r >> 1) % (4 * sizeof(ST))] >> (16 * (r & 1))) & 0xFFFFu;
    }
    // run-time row index
    __device__ __forceinline__ uint32_t byte_dyn(uint32_t r) const {
        if (SG) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(gs + r)); return v; }
        const uint32_t q = r < 8 ? (r < 4 ? w[0] : w[1]) : (r < 12 ? w[2] : w[3]);
        return (q >> (8 * (r & 3))) & 0xFFu;
    }
    __device__ __forceinline__ uint32_t state_dyn(int d, uint32_t r) const {
        if (SG) {
            uint32_t v;
            if (sizeof(ST) == 1) asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(gs + (1 + d) * EMIT_SG_PITCH + r));
            else asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(gs + (1 + 2 * d + (r >> 3)) * EMIT_SG_PITCH + (r & 7u) * 2u));
            return v;
        }
        if (sizeof(ST) == 1) {
            const uint32_t q = r < 8 ? (r < 4 ? sv[d][0] : sv[d][1]) : (r < 12 ? sv[d][2] : sv[d][3]);
            return (q >> (8 * (r & 3))) & 0xFFu;
        }
        constexpr int H = 4 * (sizeof(ST) - 1);                           // 4 for 2-byte states (0 keeps the 1-byte instantiation in bounds)
        const uint32_t lo = r < 4 ? (r < 2 ? sv[d][0] : sv[d][1]) : (r < 6 ? sv[d][2] : sv[d][3]);
        const uint32_t hi = r < 12 ? (r < 10 ? sv[d][H] : sv[d][H + 1]) : (r < 14 ? sv[d][H + 2] : sv[d][H + 3]);
        return ((r < 8 ? lo : hi) >> (16 * (r & 1))) & 0xFFFFu;
    }
};

// The string a lane works on, and what the scan learns about it.
template <int D, typename ST, bool SG = false>
struct LaneString {
    const WalkParams& p;
    const EmitTables<D>& tb;
    uint64_t j;
    const uint8_t* src;
    uint32_t L;
    uint32_t stash_g, stash_s;  // granule kept in shared memory by the walk (fused mode), NO_POS = none
    uint32_t gs = 0;            // SG: this thread's granule scratch (Granule::gs)
    // results of the scan
    uint32_t seg_a[EMIT_NSEG], seg_b[EMIT_NSEG], n_seg;   // masked segments [a,b), in order; n_seg may exceed EMIT_NSEG
    uint32_t n_rec, n_cmp;
    bool overlap, invalid;
    // streaming state of the scan
    bool prev_valid, prev_is;   // last boundary: is_start_sum set there
    uint32_t prev_pos;
    uint32_t next_row;          // last examined row + 1; NO_POS = none yet / gap closed
    uint32_t carry_s, carry_ie; // id sum of row next_row-1, is_end_sum[next_row] (0 after a gap)
    uint32_t bw_t, sw[D], ew[D]; // bitmap words being assembled: rows [32*bw_t, 32*bw_t+32)
    // Whole-sector stores of the records and compact bytes (SECTORS) and of the bitmaps (HOLD), DESIGN 4.2: one def only.  The
    // stand-alone emit kernel of three defs, bound by its instructions, took 0.63 -> 0.98 ms with the extra stores, and the held
    // bitmap words made the walk kernels of several defs spill.  The one-def stand-alone emit kernel keeps bitmap word stores
    // (the same bytes; its walk counterpart is the fused kernel, where the sectors pay).  Whatever the choice, the fused and the
    // stand-alone emit stage of a def set write the same bytes: the batch and chunked paths are compared tensor for tensor.
    static constexpr bool SECTORS = D == 1;
    static constexpr bool HOLD = SECTORS && !SG;
    uint32_t hn, hk, hv[D][4];  // bitmap words held for the sectors of the span bw_t >> 3 (fold_bitmap_words)
    uint32_t cbv[2];            // compact_pitch <= 8: the compact bytes, collected by write_masks, stored by store_compact

    __device__ __forceinline__ LaneString(const WalkParams& p_, const EmitTables<D>& tb_, uint64_t j_, const uint8_t* src_, uint32_t L_)
        : p(p_), tb(tb_), j(j_), src(src_), L(L_), stash_g(NO_POS), stash_s(0) { cbv[0] = 0; cbv[1] = 0; }

    __device__ __forceinline__ uint32_t entry(int d, uint32_t c, uint32_t s) const {
        const uint32_t S = p.def[d].num_states;
        return s < S ? tb.trans[d][(uint32_t)tb.cls[d][c] * S + s] : ENT_INVALID;   // state S = the trap state of the walk
    }
    // can a transition out of state s carry a substr id (or is s the trap state)?  One bit per state, packed by defs.cpp.
    __device__ __forceinline__ bool state_is_hot(int d, uint32_t s) const {
        if (s >= 64u) return true;
        const uint32_t m = s < 32u ? p.def[d].hot_states[0] : p.def[d].hot_states[1];
        return (m >> (s & 31u)) & 1u;
    }

    // ---- scan ----------------------------------------------------------------------------------------------------------
    // PATCH: the string has more masked segments than the registers hold; this second scan only emits them one by one
    template <bool PATCH>
    __device__ __forceinline__ void boundary(uint32_t pos, bool b_is, bool b_ie) {
        if (prev_valid && prev_is && b_ie) {                             // [prev_pos, pos) is masked
            if (PATCH) {
                const uint2 r = emit_segment<D, ST>(p, tb, j, src, prev_pos, pos, n_rec, n_cmp);
                n_rec = r.x; n_cmp = r.y;
            }
#pragma unroll
            for (int k = 0; k < EMIT_NSEG; k++)
                if (n_seg == (uint32_t)k) { seg_a[k] = prev_pos; seg_b[k] = pos; }
            n_seg++;
        }
        prev_valid = true; prev_pos = pos; prev_is = b_is;
    }
    // the rows from next_row on are not examined (id sum 0 in every def, or past the end of the string); row next_row can
    // still be a boundary: the id sum drops to 0 there and is_end_sum[next_row] comes from the row before
    template <bool PATCH>
    __device__ __forceinline__ void close_gap() {
        if (next_row != NO_POS && carry_s != 0 && carry_ie != 0) {
            if (carry_ie > 1) overlap = true;
            boundary<PATCH>(next_row, false, true);
        }
        next_row = NO_POS; carry_s = 0; carry_ie = 0;
    }
    // Bitmap words leave as whole sectors: the fill zeroed every sector long ago, so a word stored on its own would be a partial
    // write of a sector that may have left L2.  The words of the 256-row span bw_t >> 3 that have a bit in some column are held
    // (at most two: hk = their indices k0 | k1 << 3, hv = their values) and go out as one 32-byte sector per column when the scan
    // leaves the span.  A third such word stores the sector at once and itself, and any later word of the span, word by word.
    // Rows that are not 32-byte aligned take word stores throughout.
    __device__ __forceinline__ bool bitmap_sectors(const uint8_t* col) const {
        return (p.bitmap_pitch & 31) == 0 && (reinterpret_cast<uintptr_t>(col) & 31) == 0;
    }
    __device__ __forceinline__ void store_bitmap_sector(uint8_t* col, uint32_t v0, uint32_t v1) {
        if (!col || (v0 | v1) == 0) return;
        uint8_t* const sec = col + j * p.bitmap_pitch + 32ull * (bw_t >> 3);
        const uint32_t k0 = hk & 7u, k1 = hn > 1 ? hk >> 3 : 8u;   // v1 == 0 unless two words are held
        if (bitmap_sectors(col)) {
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; k++) w[k] = ((uint32_t)k == k0 ? v0 : 0u) | ((uint32_t)k == k1 ? v1 : 0u);
            reinterpret_cast<uint4*>(sec)[0] = make_uint4(w[0], w[1], w[2], w[3]);
            reinterpret_cast<uint4*>(sec)[1] = make_uint4(w[4], w[5], w[6], w[7]);
        } else {
            if (v0) reinterpret_cast<uint32_t*>(sec)[k0] = v0;
            if (v1) reinterpret_cast<uint32_t*>(sec)[k1] = v1;
        }
    }
    __device__ __forceinline__ void store_bitmap_held() {
#pragma unroll
        for (int d = 0; d < D; d++) {
            store_bitmap_sector(p.def[d].start_enable, hv[d][0], hn > 1 ? hv[d][1] : 0u);
            store_bitmap_sector(p.def[d].end_enable, hv[d][2], hn > 1 ? hv[d][3] : 0u);
        }
    }
    // the word being assembled is complete
    __device__ __forceinline__ void fold_bitmap_words() {
        uint32_t any = 0;
#pragma unroll
        for (int d = 0; d < D; d++) any |= sw[d] | ew[d];
        if (any) {
            if (HOLD && hn < 2) {
#pragma unroll
                for (int d = 0; d < D; d++) {
                    if (hn == 0) { hv[d][0] = sw[d]; hv[d][2] = ew[d]; } else { hv[d][1] = sw[d]; hv[d][3] = ew[d]; }
                }
                hk |= (bw_t & 7u) << (3 * hn);
                hn++;
            } else {
                if (HOLD && hn == 2) { store_bitmap_held(); hn = 3; }
#pragma unroll
                for (int d = 0; d < D; d++) {
                    if (sw[d] && p.def[d].start_enable) *reinterpret_cast<uint32_t*>(p.def[d].start_enable + j * p.bitmap_pitch + 4 * bw_t) = sw[d];
                    if (ew[d] && p.def[d].end_enable) *reinterpret_cast<uint32_t*>(p.def[d].end_enable + j * p.bitmap_pitch + 4 * bw_t) = ew[d];
                }
            }
        }
#pragma unroll
        for (int d = 0; d < D; d++) { sw[d] = 0; ew[d] = 0; }
    }
    __device__ __forceinline__ void flush_bitmap_span() {
        if (bw_t == NO_POS) return;
        fold_bitmap_words();
        if (HOLD && (hn == 1 || hn == 2)) store_bitmap_held();
        hn = 0; hk = 0;
    }
    // flagged granule g; partner_flagged: the other granule of its 32-row window is flagged too (and writes itself)
    template <bool PATCH>
    __device__ __forceinline__ void scan_granule(uint32_t g, bool partner_flagged) {
        Granule<D, ST, SG> gr;
        gr.gs = gs;
        gr.load(p, j, src, L, g, stash_g, stash_s);
        // pass 1, unrolled, all lanes in step: rows whose state can start a transition with a substr id (or is the trap state)
        uint32_t hot = 0;
#pragma unroll
        for (int r = 0; r < 16; r++) {
#pragma unroll
            for (int d = 0; d < D; d++)
                if (state_is_hot(d, gr.state_at(d, r))) hot |= 1u << r;
        }
        hot &= (1u << gr.n) - 1u;                                        // rows past the end of the string are not characters
        // pass 2, one loop body shared by all lanes: each lane handles ITS next candidate row
        uint32_t sidv[D][4];
#pragma unroll
        for (int d = 0; d < D; d++) sidv[d][0] = sidv[d][1] = sidv[d][2] = sidv[d][3] = 0;
        if (!PATCH && (g >> 1) != bw_t) {
            if (bw_t != NO_POS && (g >> 4) == (bw_t >> 3)) fold_bitmap_words(); else flush_bitmap_span();
            bw_t = g >> 1;
        }
        while (hot) {
            const uint32_t r = (uint32_t)__ffs((int)hot) - 1u;
            hot &= hot - 1;
            const uint32_t i = 16 * g + r;
            const uint32_t c = gr.byte_dyn(r);
            uint32_t sum = 0, is_sum = 0, ie_next = 0;
            bool any = false;
#pragma unroll
            for (int d = 0; d < D; d++) {
                const uint32_t S = p.def[d].num_states;
                const uint32_t st = gr.state_dyn(d, r);
                const uint32_t e = entry(d, c, st);
                if (e & ENT_INVALID) { invalid = true; continue; }
                const uint32_t sid = ent_sid(e);
                if (!sid) continue;
                any = true;
                sum += sid;
                if (!PATCH) {
                    const uint32_t v = sid << (8 * (r & 3));
                    if ((r >> 2) == 0) sidv[d][0] |= v; else if ((r >> 2) == 1) sidv[d][1] |= v; else if ((r >> 2) == 2) sidv[d][2] |= v; else sidv[d][3] |= v;
                }
                if (e & ENT_IS_START) {                                  // start_enable; endpoint lookup src/lib.rs:235-258
                    is_sum++;
                    if (!PATCH) {
                        sw[d] |= 1u << (i & 31);
                        const uint32_t bin = (sid - p.def[d].sid_offset) * S + st;
                        if (tb.ep_s[d]) atomicAdd(tb.ep_s[d] + bin, 1u); else atomicAdd(p.def[d].ep_start + bin, 1ull);
                    }
                }
                if (e & ENT_IS_END) {                                    // end_enable; endpoint lookup src/lib.rs:260-284
                    ie_next++;
                    if (!PATCH) {
                        ew[d] |= 1u << (i & 31);
                        const uint32_t bin = (sid - p.def[d].sid_offset) * S + (e & ENT_NEXT_MASK);
                        if (tb.ep_s[d]) atomicAdd(tb.ep_s[d] + p.def[d].num_substrs * S + bin, 1u); else atomicAdd(p.def[d].ep_end + bin, 1ull);
                    }
                }
            }
            if (!any) continue;                                          // id sum 0 in every def: like a row of an unflagged granule
            if (next_row != i) close_gap<PATCH>();
            if (is_sum > 1 || carry_ie > 1) overlap = true;
            if (sum != carry_s && (is_sum | carry_ie)) boundary<PATCH>(i, is_sum != 0, carry_ie != 0);
            carry_s = sum; carry_ie = ie_next; next_row = i + 1;
        }
        if (!PATCH) {
            // the complete sector of the substr-id columns: my 16 bytes, and zeros for the partner unless it writes itself
            const uint32_t base = 16 * g, pbase = 16 * (g ^ 1u);
            const bool partner = !partner_flagged && (uint64_t)pbase + 16 <= p.row_pitch;
#pragma unroll
            for (int d = 0; d < D; d++) {
                if (!p.def[d].substr_ids) continue;
                uint8_t* const row = p.def[d].substr_ids + j * p.row_pitch;
                *reinterpret_cast<uint4*>(row + base) = make_uint4(sidv[d][0], sidv[d][1], sidv[d][2], sidv[d][3]);
                if (partner) *reinterpret_cast<uint4*>(row + pbase) = make_uint4(0, 0, 0, 0);
            }
        }
    }
    __device__ __forceinline__ void scan_begin() {
        n_seg = 0; n_rec = 0; n_cmp = 0; overlap = false; invalid = false;
        prev_valid = false; prev_is = false; prev_pos = 0;
        next_row = NO_POS; carry_s = 0; carry_ie = 0;
        bw_t = NO_POS;
#pragma unroll
        for (int d = 0; d < D; d++) { sw[d] = 0; ew[d] = 0; }
        hn = 0; hk = 0;
    }
    template <bool PATCH>
    __device__ __forceinline__ void scan_end() {
        if (!invalid) { close_gap<PATCH>(); if (!PATCH) flush_bitmap_span(); }
        // an invalid string: the words finished before the failing row still go out, as word stores would have written them
        // (the stand-alone emit kernel does), so that both emit paths leave the same bytes
        else if (!PATCH && HOLD && (hn == 1 || hn == 2)) store_bitmap_held();
    }
    // fw0 / fw1: granule flags 0..63 of this string; further words come from the flag buffer `flags`
    template <bool PATCH>
    __device__ __forceinline__ void scan(uint32_t fw0, uint32_t fw1, const uint32_t* flags) {
        scan_begin();
        for (uint32_t w = 0; w < p.fm_words && !invalid; w++) {
            const uint32_t fw = w == 0 ? fw0 : w == 1 ? fw1 : __ldcg(flags + (size_t)w * p.n_strings + j);
            uint32_t bits = fw;
            while (bits && !invalid) {
                const uint32_t g = (uint32_t)__ffs((int)bits) - 1u;
                bits &= bits - 1;
                scan_granule<PATCH>(w * 32 + g, (fw >> (g ^ 1u)) & 1u);
            }
        }
        scan_end<PATCH>();
    }

    // ---- masks ---------------------------------------------------------------------------------------------------------
    // The masked segments (at most EMIT_NSEG, in order): the complete sectors of masked_chars / masked_substr_ids they
    // touch, the compact bytes, and one record per maximal run of a constant id sum (src/lib.rs:740-764).
    __device__ __forceinline__ void write_masks() {
        uint8_t* const mc = p.masked_chars ? p.masked_chars + j * p.row_pitch : nullptr;
        uint8_t* const ms = p.masked_substr_ids ? p.masked_substr_ids + j * p.row_pitch : nullptr;
        uint8_t* const cb = p.compact_bytes ? p.compact_bytes + j * (uint64_t)p.compact_pitch : nullptr;
        uint32_t cur_t = NO_POS;                                         // window being assembled
        uint32_t mcv[8], msv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { mcv[k] = 0; msv[k] = 0; }
        auto flush = [&]() {
            if (cur_t == NO_POS) return;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint64_t o = 32ull * cur_t + 16ull * h;
                if (o + 16 > p.row_pitch) continue;                      // the last window of a row can be half
                if (mc) *reinterpret_cast<uint4*>(mc + o) = make_uint4(mcv[4 * h], mcv[4 * h + 1], mcv[4 * h + 2], mcv[4 * h + 3]);
                if (ms) *reinterpret_cast<uint4*>(ms + o) = make_uint4(msv[4 * h], msv[4 * h + 1], msv[4 * h + 2], msv[4 * h + 3]);
            }
#pragma unroll
            for (int k = 0; k < 8; k++) { mcv[k] = 0; msv[k] = 0; }
        };
        uint32_t run_start = 0, run_sum = 0, run_coff = 0;
        bool in_run = false;
        auto close_run = [&](uint32_t end) {
            if (!in_run) return;
            if (p.records && n_rec < p.max_records) {
                b2r_substr_record r; r.start = run_start; r.len = end - run_start; r.substr_id = run_sum; r.compact_off = run_coff;
                p.records[j * p.max_records + n_rec] = r;
            }
            n_rec++; in_run = false;
        };
#pragma unroll
        for (int k = 0; k < EMIT_NSEG; k++) {
            if ((uint32_t)k >= n_seg) continue;
            const uint32_t a = seg_a[k], b = seg_b[k];
            for (uint32_t g = a >> 4; g <= (b - 1) >> 4; g++) {
                if ((g >> 1) != cur_t) { flush(); cur_t = g >> 1; }
                Granule<D, ST, SG> gr;
                gr.gs = gs;
                gr.load(p, j, src, L, g, stash_g, stash_s);
                const uint32_t lo = a > 16 * g ? a - 16 * g : 0u, hi = b < 16 * g + 16 ? b - 16 * g : 16u;
                for (uint32_t r = lo; r < hi; r++) {
                    const uint32_t i = 16 * g + r;
                    const uint32_t c = gr.byte_dyn(r);
                    uint32_t sum = 0;
#pragma unroll
                    for (int d = 0; d < D; d++) {
                        const uint32_t e = entry(d, c, gr.state_dyn(d, r));
                        sum += (e & ENT_INVALID) ? 0u : ent_sid(e);
                    }
                    const uint32_t q = (i >> 2) & 7u, sh = 8 * (i & 3u);
#pragma unroll
                    for (int w = 0; w < 8; w++)
                        if (q == (uint32_t)w) { mcv[w] |= c << sh; msv[w] |= sum << sh; }
                    if (cb && n_cmp < p.compact_pitch) {
                        if (SECTORS && p.compact_pitch <= 8) { if (n_cmp < 4) cbv[0] |= c << (8 * n_cmp); else cbv[1] |= c << (8 * (n_cmp - 4)); }
                        else cb[n_cmp] = (uint8_t)c;
                    }
                    if (!in_run || sum != run_sum || i == a) {          // a new segment always starts a new run (the id sum changes at a boundary)
                        close_run(i);
                        in_run = true; run_start = i; run_sum = sum; run_coff = n_cmp;
                    }
                    n_cmp++;
                }
            }
            close_run(b);
        }
        flush();
        // the last record ends in the first half of a sector: zeros in the second half, so that the sector leaves L2 whole
        if (SECTORS && p.records && n_rec > 0 && n_rec < p.max_records) {
            b2r_substr_record* const r = p.records + j * p.max_records + n_rec;
            if ((reinterpret_cast<uintptr_t>(r) & 31) == 16) *reinterpret_cast<uint4*>(r) = make_uint4(0, 0, 0, 0);
        }
        // a compact area of more than 8 bytes that is not full: zeros up to its end (areas of at most 8: store_compact)
        if (SECTORS && cb && p.compact_pitch > 8 && n_cmp > 0 && n_cmp < p.compact_pitch) {
            for (uint32_t k = n_cmp; k < p.compact_pitch;) {
                const uintptr_t a = reinterpret_cast<uintptr_t>(cb + k);
                if ((a & 15) == 0 && k + 16 <= p.compact_pitch) { *reinterpret_cast<uint4*>(cb + k) = make_uint4(0, 0, 0, 0); k += 16; }
                else if ((a & 3) == 0 && k + 4 <= p.compact_pitch) { *reinterpret_cast<uint32_t*>(cb + k) = 0u; k += 4; }
                else { cb[k] = 0; k++; }
            }
        }
    }
    // compact_pitch <= 8: the string's whole compact area at once (the bytes write_masks collected, zeros after them).  Called by
    // all lanes of a warp together, for neighbouring strings, so that the areas of four or more strings leave as whole sectors.
    __device__ __forceinline__ void store_compact() {
        uint8_t* const cb = p.compact_bytes + j * (uint64_t)p.compact_pitch;
        if (p.compact_pitch == 8 && (reinterpret_cast<uintptr_t>(cb) & 7) == 0) *reinterpret_cast<uint2*>(cb) = make_uint2(cbv[0], cbv[1]);
        else
            for (uint32_t k = 0; k < p.compact_pitch; k++) cb[k] = (uint8_t)((k < 4 ? cbv[0] : cbv[1]) >> (8 * (k & 3)));
    }
};

// Warp-cooperative emitter for one tile of 32 consecutive strings.
template <int D, typename ST, bool SG = false>
struct TileEmitter {
    const WalkParams& p;
    const EmitTables<D>& tb;
    const int lane;
    uint32_t gs = 0;            // SG: this thread's granule scratch in shared memory

    __device__ __forceinline__ TileEmitter(const WalkParams& p_, const EmitTables<D>& tb_, int lane_) : p(p_), tb(tb_), lane(lane_) {}

    // Lane = string.  off / Ll / live: the lane's string (live = in range and not too long); fw0 / fw1: its granule flags
    // 0..63 (further words are read from p.fmask); fin[]: its final states; filled: the caller has zeroed the tile's rows.
    __device__ __forceinline__ void run_tile(uint64_t tile_base, bool valid, bool live, uint64_t off, uint32_t Ll, uint32_t fw0, uint32_t fw1,
                                             const uint32_t* fin, EmitTotals& tot, bool filled, uint32_t stash_g = NO_POS, uint32_t stash_s = 0) {
        constexpr uint32_t FULL = 0xffffffffu;
        const uint64_t N = p.n_strings;
        const uint32_t M = p.max_chars;
        const uint64_t rp = p.row_pitch, bp = p.bitmap_pitch;
        const uint64_t jl = tile_base + lane;
        const uint64_t rows_here = N - tile_base < 32 ? N - tile_base : 32;

        // ---- fill (warp): the tile's rows of a column are contiguous ----------------------------------------------------
        if (!filled && !(p.debug & 1)) {
#pragma unroll
            for (int d = 0; d < D; d++) {
                emit_zero_region(p.def[d].substr_ids ? p.def[d].substr_ids + tile_base * rp : nullptr, rows_here * rp, lane);
                emit_zero_region(p.def[d].start_enable ? p.def[d].start_enable + tile_base * bp : nullptr, rows_here * bp, lane);
                emit_zero_region(p.def[d].end_enable ? p.def[d].end_enable + tile_base * bp : nullptr, rows_here * bp, lane);
            }
            emit_zero_region(p.masked_chars ? p.masked_chars + tile_base * rp : nullptr, rows_here * rp, lane);
            emit_zero_region(p.masked_substr_ids ? p.masked_substr_ids + tile_base * rp : nullptr, rows_here * rp, lane);
        }
        __syncwarp();                                                    // the zeros are ordered before the values below

        // ---- scan + masks (lane = string) ---------------------------------------------------------------------------------
        uint32_t r_nrec = 0, r_ncmp = 0, r_flags = 0;
        bool patch = false;
        LaneString<D, ST, SG> ls(p, tb, jl, p.bytes + off, Ll);
        ls.stash_g = stash_g; ls.stash_s = stash_s; ls.gs = gs;
        if (live && !(p.debug & 2) && (p.fm_words > 2 || (fw0 | fw1) != 0)) {
            ls.template scan<false>(fw0, fw1, p.fmask);
            if (ls.invalid) r_flags = B2R_ST_INVALID_TRANSITION;
            else {
                if (ls.overlap) r_flags = B2R_ST_OVERLAP;
                patch = ls.n_seg > EMIT_NSEG;
                if (!patch) { ls.write_masks(); r_nrec = ls.n_rec; r_ncmp = ls.n_cmp; }
            }
        }
#pragma unroll
        for (int d = 0; d < D; d++)
            if (live && fin[d] >= p.def[d].num_states) r_flags = B2R_ST_INVALID_TRANSITION;   // the last character had no transition
        // ---- more masked segments than the registers hold: emit them one by one, byte by byte (rare) --------------------------
        if (__any_sync(FULL, patch)) {
            __syncwarp();
            if (patch) { ls.template scan<true>(fw0, fw1, p.fmask); r_nrec = ls.n_rec; r_ncmp = ls.n_cmp; }
        }
        if (LaneString<D, ST, SG>::SECTORS) {
            __syncwarp();
            if (p.compact_bytes && p.compact_pitch <= 8 && valid && !patch) ls.store_compact();
        }
        // two defs flagging one row: the string has no records (include/b2r.h), so no counts and no truncation flags either
        if (r_flags & B2R_ST_OVERLAP) { r_nrec = 0; r_ncmp = 0; }

        // ---- accept rule (src/lib.rs:427-457), status records (lane = string) --------------------------------------------
        if (valid && !(p.debug & 8)) {
            if (!live || (r_flags & B2R_ST_INVALID_TRANSITION)) kill_string(p, jl);
            else {
                uint32_t flags = r_flags;
#pragma unroll
                for (int d = 0; d < D; d++)
                    if (fin[d] == p.def[d].accepted_state) flags |= B2R_ST_ACCEPTED(d);
                if (p.records && r_nrec > p.max_records) flags |= B2R_ST_RECORDS_TRUNCATED;
                if (p.compact_bytes && r_ncmp > p.compact_pitch) flags |= B2R_ST_COMPACT_TRUNCATED;
                if (p.status) {   // 32 bytes per string: two 16-byte stores when the array is 16-byte aligned (2 x 32 sectors per warp, not 8 x 32)
                    if ((reinterpret_cast<uintptr_t>(p.status) & 15) == 0) {
                        uint4* q = reinterpret_cast<uint4*>(p.status + jl);
                        q[0] = make_uint4(flags, NO_POS, 0u, 0u);        // flags, err_pos, err_state, err_byte/err_def/reserved0
                        q[1] = make_uint4(r_nrec, r_ncmp, 0u, 0u);       // n_records, n_compact, reserved1[2]
                    } else {
                        b2r_string_status st = {};
                        st.flags = flags; st.err_pos = NO_POS; st.n_records = r_nrec; st.n_compact = r_ncmp;
                        p.status[jl] = st;
                    }
                }
                tot.pad_rows += M - Ll; tot.n_ok++; tot.n_overlap += (r_flags & B2R_ST_OVERLAP) ? 1u : 0u;
            }
        }
        __syncwarp();
    }

    // stand-alone entry: everything about the tile's strings comes from global memory
    __device__ __forceinline__ void run_tile_from_memory(uint64_t tile, EmitTotals& tot, bool filled) {
        const uint64_t N = p.n_strings;
        const uint32_t M = p.max_chars;
        const uint64_t tile_base = tile * 32;
        const uint64_t jl = tile_base + lane;
        const bool valid = jl < N;
        uint64_t off = 0, end = 0;
        if (valid) { off = p.offsets[jl]; end = p.offsets[jl + 1]; }
        const bool too_long = valid && (end < off || end - off > (uint64_t)(M - 1) || end > p.total_bytes);   // SURVEY 8(a) row 6: len must be <= M-1
        const bool live = valid && !too_long;
        const uint32_t Ll = live ? (uint32_t)(end - off) : 0u;
        uint32_t fw0 = 0, fw1 = 0;
        if (live && p.fm_words > 0) fw0 = __ldcg(p.fmask + jl);
        if (live && p.fm_words > 1) fw1 = __ldcg(p.fmask + N + jl);
        uint32_t fin[D];
#pragma unroll
        for (int d = 0; d < D; d++)
            fin[d] = (live && !(p.debug & 4)) ? (uint32_t)__ldcg(reinterpret_cast<const ST*>(p.def[d].states) + jl * p.row_pitch + Ll) : 0xFFFFFFFEu;
        run_tile(tile_base, valid, live, live ? off : 0ull, Ll, fw0, fw1, fin, tot, filled);
    }
};

// shared memory of the emitter: endpoint counters, then (optionally) the lookup tables.
__host__ __device__ inline uint32_t emit_smem_bytes(const WalkParams& p) {
    uint32_t n = (p.ep_smem_bytes + 15u) & ~15u;
    if (p.emit_smem_tables)
        for (uint32_t d = 0; d < p.n_defs; d++) n += ((p.def[d].num_classes * p.def[d].num_states * 4u + 256u) + 15u) & ~15u;
    return n;
}
// the stand-alone emit kernel appends the granule scratch of its threads (Granule<.., SG = true>) behind the tables
__host__ __device__ inline uint32_t emit_scratch_bytes(const WalkParams& p, uint32_t state_bytes) { return (1u + p.n_defs * state_bytes) * EMIT_SG_PITCH; }
// Every thread of the CTA calls this, followed by a __syncthreads().
template <int D>
__device__ __forceinline__ void emit_tables_init(const WalkParams& p, unsigned char* esmem, EmitTables<D>& tb) {
    uint32_t off = 0;
#pragma unroll
    for (int d = 0; d < D; d++) {
        tb.ep_s[d] = p.ep_smem_bytes ? reinterpret_cast<uint32_t*>(esmem + off) : nullptr;
        if (p.ep_smem_bytes) off += 2u * p.def[d].num_substrs * p.def[d].num_states * 4u;
    }
    off = (off + 15u) & ~15u;
    for (uint32_t i = threadIdx.x; i < off / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(esmem)[i] = 0;
#pragma unroll
    for (int d = 0; d < D; d++) {
        if (p.emit_smem_tables) {
            const uint32_t n = p.def[d].num_classes * p.def[d].num_states;
            uint32_t* const t = reinterpret_cast<uint32_t*>(esmem + off);
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) t[i] = p.def[d].trans[i];
            uint8_t* const c = esmem + off + n * 4;
            for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) c[i] = p.def[d].byte_class[i];
            off += ((n * 4 + 256u) + 15u) & ~15u;
            tb.trans[d] = t; tb.cls[d] = c;
        } else {
            tb.trans[d] = p.def[d].trans; tb.cls[d] = p.def[d].byte_class;
        }
    }
}

// publish the per-lane totals and the CTA's endpoint counters; every thread of the CTA calls this
template <int D>
__device__ __forceinline__ void emit_publish(const WalkParams& p, const EmitTables<D>& tb, const EmitTotals& tot) {
    unsigned long long psum = tot.pad_rows;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
    const uint32_t nok = __reduce_add_sync(0xffffffffu, tot.n_ok), nov = __reduce_add_sync(0xffffffffu, tot.n_overlap);
    if ((threadIdx.x & 31) == 0) {
        if (psum) atomicAdd(&p.counters->pad_rows, psum);
        if (nov) atomicAdd(&p.counters->n_overlap, (unsigned long long)nov);
        if (nok) atomicAdd(&p.counters->n_ok_strings, (unsigned long long)nok);
    }
    __syncthreads();
#pragma unroll
    for (int d = 0; d < D; d++) {
        if (!tb.ep_s[d]) continue;
        const uint32_t ks = p.def[d].num_substrs * p.def[d].num_states;
        for (uint32_t i = threadIdx.x; i < 2 * ks; i += blockDim.x) {
            const uint32_t v = tb.ep_s[d][i];
            if (v) atomicAdd((i < ks ? p.def[d].ep_start + i : p.def[d].ep_end + (i - ks)), (unsigned long long)v);
        }
    }
}

// Zero-fill of one tile's rows of every sparse column with TMA bulk stores (shared zero buffer -> global), lane-strided; the
// caller commits the bulk group.  The rows of a tile are contiguous in every column.  zero_s: EMIT_ZERO_BYTES of zeros.
constexpr uint32_t EMIT_ZERO_BYTES = 4096;
template <int D>
__device__ __forceinline__ void emit_issue_tile_fill(const WalkParams& p, uint64_t tile, int lane, uint32_t zero_s) {
    const uint64_t tile_base = tile * 32;
    const uint64_t rows_here = p.n_strings - tile_base < 32 ? p.n_strings - tile_base : 32;
    const uint64_t cbytes = rows_here * p.row_pitch, bbytes = rows_here * p.bitmap_pitch;
    uint32_t first = 0;
    auto region = [&](uint8_t* ptr, uint64_t bytes) {
        if (!ptr) return;
        const uint32_t bulk_bytes = (uint32_t)(bytes & ~15ull);            // bitmap regions of a partial tile can end on a 4-byte boundary
        const uint32_t n_ops = (bulk_bytes + EMIT_ZERO_BYTES - 1) / EMIT_ZERO_BYTES;
        for (uint32_t op = ((uint32_t)lane + 32u - (first & 31u)) & 31u; op < n_ops; op += 32) {
            const uint32_t o = op * EMIT_ZERO_BYTES;
            const uint32_t nb = bulk_bytes - o < EMIT_ZERO_BYTES ? bulk_bytes - o : EMIT_ZERO_BYTES;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(ptr + o), "r"(zero_s), "r"(nb) : "memory");
        }
        for (uint64_t o = bulk_bytes + (uint64_t)lane * 4; o < bytes; o += 128) *reinterpret_cast<uint32_t*>(ptr + o) = 0u;
        first += n_ops;
    };
#pragma unroll
    for (int d = 0; d < D; d++) {
        region(p.def[d].substr_ids ? p.def[d].substr_ids + tile_base * p.row_pitch : nullptr, cbytes);
        region(p.def[d].start_enable ? p.def[d].start_enable + tile_base * p.bitmap_pitch : nullptr, bbytes);
        region(p.def[d].end_enable ? p.def[d].end_enable + tile_base * p.bitmap_pitch : nullptr, bbytes);
    }
    region(p.masked_chars ? p.masked_chars + tile_base * p.row_pitch : nullptr, cbytes);
    region(p.masked_substr_ids ? p.masked_substr_ids + tile_base * p.row_pitch : nullptr, cbytes);
}

// The emit stage as its own kernel (the walk ran first; B2R_FUSE=0, and the default for three or more defs: there the fused kernel's
// code no longer fits the instruction caches — 34 % of its warp samples were instruction-fetch stalls — and walk + emit as two
// kernels take 4.0 instead of 4.7 ms per 2^20 strings).  Tiles are handed out by an atomic counter.  The zero-fill of the NEXT tile
// (TMA bulk stores, asynchronous) is in flight while the current tile is scanned: fill and scan overlap instead of adding up.
template <int D, typename ST>
__global__ void __launch_bounds__(EMIT_THREADS) emit_kernel(const __grid_constant__ WalkParams p) {
    extern __shared__ __align__(16) unsigned char esmem[];
    __shared__ __align__(128) unsigned char zero_buf[EMIT_ZERO_BYTES];
    const int lane = threadIdx.x & 31;
    EmitTables<D> tb;
    emit_tables_init<D>(p, esmem, tb);
    const bool fill = !p.prefilled && !(p.debug & 1);
    for (uint32_t i = threadIdx.x * 16; i < EMIT_ZERO_BYTES; i += blockDim.x * 16) *reinterpret_cast<uint4*>(zero_buf + i) = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // zero buffer -> visible to the TMA (async proxy)
    __syncthreads();
    const uint32_t zero_s = (uint32_t)__cvta_generic_to_shared(zero_buf);

    TileEmitter<D, ST, true> em(p, tb, lane);
    em.gs = (uint32_t)__cvta_generic_to_shared(esmem) + ((emit_smem_bytes(p) + 15u) & ~15u) + threadIdx.x * 16u;
    EmitTotals tot;
    auto fetch = [&]() -> unsigned long long {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(&p.counters->emit_tile_counter, 1ull);
        return __shfl_sync(0xffffffffu, t, 0);
    };
    unsigned long long t = fetch();
    if (fill && t < p.n_tiles) emit_issue_tile_fill<D>(p, t, lane, zero_s);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    while (t < p.n_tiles) {
        const unsigned long long t_next = fetch();
        if (fill && t_next < p.n_tiles) emit_issue_tile_fill<D>(p, t_next, lane, zero_s);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group 1;" ::: "memory");      // the zeros of tile t are in place (mine ...
        __syncwarp();                                                    // ... and those of the other lanes)
        em.run_tile_from_memory(t, tot, /*filled=*/true);
        t = t_next;
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    emit_publish<D>(p, tb, tot);
}

}  // namespace b2r
