// walk_kernel — stage 1 of the batch path: the DFA walk (reference derive_states, src/lib.rs:804-823).
//
// One LANE per string, one WARP per tile of 32 strings, persistent CTAs (one per SM), tiles handed out by an atomic
// counter.  The kernel produces
//   - the state column of every def (rows 0..len-1 = s_i, row len = final state, later rows = dummy, src/lib.rs:404-418),
//   - one flag bit per 16-row granule and string: "some row in here has a non-zero substr id or an invalid transition"
//     (everything the reference derives beyond the state column lives in such rows; emit.cuh re-derives it from the
//     state column, only inside flagged granules),
//   - the multiplicity bins of the transition lookup (src/lib.rs:207-233): one count per (byte, state) row.
// There is no data-dependent branch in the hot loop.
//
// Tables.  The sparse lookup text was packed by defs.cpp into byte classes + a [class][state] next-state table.  In
// shared memory every entry is REPLICATED ONCE PER BANK (TABLE_REPL): entry (class k, state s) of lane l lives at
//   tab + (k*P + s)*128 + l*4,
// so a warp's 32 lookups (32 different strings, arbitrary bytes and states) never conflict: one wavefront per lookup
// instead of ~3.4 for randomly banked addresses.  The byte -> class table is replicated the same way and, for a single
// def, holds the ABSOLUTE shared address of (class row, state 0, this lane).  An entry is
//   [31:16] next state   [15:2] next state * stride / 4   [0] rare
// so the dependent chain per byte is   LOP3 (entry & 0xFFFC | class row)  ->  LDS.
// When the replicated tables do not fit, the same code runs with stride 4 (TABLE_PLAIN, one copy, bank conflicts), and
// when even that does not fit the table stays in global memory (TABLE_GLOBAL, template parameter).
//
// I/O.  cp.async 16-byte copies (zero-filled past the string end) stage chunk k+1 of the 32 strings into a padded,
// double-buffered tile while chunk k is walked; each lane reads ITS string with conflict-free LDS.128.  States go back
// through a padded tile and out as coalesced 16-byte stores, one full 32-byte sector per row and chunk.
//
// Multiplicities.  One shared-memory atomic per byte into bins [state][byte] (bank = byte mod 32), flushed once per
// CTA with 64-bit global atomics.  (HIST_GLOBAL: straight to the global bins; only for tables too large for shared memory.)
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "defs.hpp"
#include "emit.cuh"
#include "kernels.cuh"
#include "long.cuh"

namespace b2r {

constexpr int WALK_MAX_THREADS = 512;
constexpr int WALK_DCH = 32;                       // positions per staged chunk
constexpr int WALK_PITCH = WALK_DCH + 16;          // input tile row pitch (bytes): 3 x 16 B keeps per-lane LDS.128 conflict-free
constexpr uint32_t WALK_ZERO_BYTES = 4096;         // shared zero buffer, source of the TMA bulk zero-fills (fused emit stage)

// ---- PTX helpers -------------------------------------------------------------------------------------------------------
// prmt (default mode): selector nibble 0-7 picks a byte of {a (0-3), b (4-7)}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t saddr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void red_shared_inc(uint32_t saddr) { asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(saddr) : "memory"); }
// 16-byte async copy global -> shared; copies src_bytes (0..16) and zero-fills the rest
__device__ __forceinline__ void cp_async16(uint32_t sdst, const void* gsrc, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global.L2::128B [%0], [%1], 16, %2;" ::"r"(sdst), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- shared-memory layout, computed identically by the launcher and the kernel ---------------------------------------------
// bytes between consecutive table entries; class-table entries are 4 bytes (128 when replicated)
// in-row XOR swizzle of class row k of a single-copy table (row_bytes = padded_states * stride, a power of two): words
__host__ __device__ inline uint32_t walk_swizzle(uint32_t k, uint32_t row_bytes) { return (k << 2) & (row_bytes - 1u) & 0x7Cu; }
__host__ __device__ inline uint32_t walk_stride(uint32_t table_mode) { return table_mode == TABLE_REPL ? 128u : table_mode == TABLE_REPL16 ? 64u : table_mode == TABLE_PLAIN16 ? 2u : 4u; }
__host__ __device__ inline uint32_t walk_cls_stride(uint32_t table_mode, uint32_t cls_repl) { return table_mode == TABLE_REPL || table_mode == TABLE_REPL16 || cls_repl ? 128u : 4u; }
__host__ __device__ inline uint32_t walk_align_up(uint32_t x, uint32_t a) { return (x + a - 1) & ~(a - 1); }

// columns of a def's shared-memory bins: the compact layout (kernels.cuh, bin_cols) for two or three defs on 16-bit tables, else one per byte
__host__ __device__ inline uint32_t walk_bin_cols(const WalkParams& p) {
    const bool e16 = p.table_mode == TABLE_PLAIN16 || p.table_mode == TABLE_REPL16;
    return (e16 && p.hist_mode == HIST_SMEM && p.n_defs >= 2 && p.n_defs <= 3 && p.bin_cols && p.bin_cols < 256) ? p.bin_cols : 256u;
}

struct WalkLayout {
    uint32_t tab[B2R_MAX_DEFS];    // byte offsets from the aligned base; table rows are P*stride bytes and aligned to that
    uint32_t cls;                  // 256 entries of `stride` bytes
    uint32_t hist[B2R_MAX_DEFS];   // (S+1) x 256 u32 bins per def (HIST_SMEM) / the bin cache (HIST_GLOBAL)
    uint32_t emit;                 // emit tables + endpoint counters (emit.cuh), fused mode
    uint32_t zero;                 // WALK_ZERO_BYTES of zeros, fused mode
    uint32_t tiles;                // first per-warp tile
    uint32_t per_warp, st_off, stash_off;   // bytes per warp; offsets of the state tile / granule stash inside
    uint32_t align;                // alignment the base needs (the largest table row)
};
__host__ __device__ inline WalkLayout walk_layout(const WalkParams& p, uint32_t state_bytes) {
    WalkLayout L{};
    uint32_t cur = 0, al = 128;
    if (p.table_mode != TABLE_GLOBAL) {
        const uint32_t stride = walk_stride(p.table_mode);
        for (uint32_t d = 0; d < p.n_defs; d++) {
            const uint32_t rb = p.def[d].padded_states * stride;
            cur = walk_align_up(cur, rb);
            L.tab[d] = cur;
            cur += p.def[d].num_classes * rb;
            if (rb > al) al = rb;
        }
        cur = walk_align_up(cur, 128);
        L.cls = cur;
        cur += 256 * walk_cls_stride(p.table_mode, p.cls_repl);
    }
    if (p.hist_mode == HIST_SMEM)
        for (uint32_t d = 0; d < p.n_defs; d++) { L.hist[d] = cur; cur += (p.def[d].num_states + 1) * walk_bin_cols(p) * 4u; }
    if (p.hist_mode == HIST_GLOBAL)   // bin cache: 2^log2 slots of {key, count}
        for (uint32_t d = 0; d < p.n_defs; d++) { L.hist[d] = cur; cur += 8u << p.hist_cache_log2; }
    cur = walk_align_up(cur, 16);
    L.emit = cur;
    if (p.fuse) cur += emit_smem_bytes(p);
    cur = walk_align_up(cur, 128);
    L.zero = cur;
    if (p.fuse || p.fill_in_walk) cur += WALK_ZERO_BYTES;
    L.tiles = cur;
    // per warp: two input tiles (double buffer); a state tile per def — except for one def with 1-byte states, whose states
    // overwrite the consumed bytes of the current input tile; the stash of one flagged granule per lane (fused emit stage)
    const bool inplace = p.n_defs == 1 && state_bytes == 1;
    L.st_off = 2 * 32 * WALK_PITCH;
    L.stash_off = L.st_off + (inplace ? 0u : p.n_defs * 32 * (WALK_DCH * state_bytes + 16));
    L.per_warp = L.stash_off + ((p.fuse && p.n_defs == 1) ? 32u * 16u * (1u + p.n_defs * state_bytes) : 0u);   // stash: one def only (else the warps matter more)
    L.align = al;
    return L;
}
__host__ __device__ inline size_t walk_smem_bytes(const WalkParams& p, uint32_t state_bytes, int warps) {
    const WalkLayout L = walk_layout(p, state_bytes);
    return (size_t)L.align + L.tiles + (size_t)warps * L.per_warp;   // + align: the dynamic base is only 16-byte aligned
}

// TM: TABLE_REPL, TABLE_REPL16, TABLE_PLAIN, TABLE_PLAIN16 or TABLE_GLOBAL.  HM: HIST_SMEM or HIST_GLOBAL.
// CH: chunked batch mode (kernels.cuh, chunk_k): the "strings" are LONG_CHUNK-row slots of the batch strings.
template <int D, typename ST, int TM, int HM, bool CH = false>
__global__ void __launch_bounds__(WALK_MAX_THREADS, 1) walk_kernel(const __grid_constant__ WalkParams p) {
    constexpr int DCH = WALK_DCH, PITCH = WALK_PITCH;
    constexpr int SB = sizeof(ST);
    constexpr int SPITCH = DCH * SB + 16;        // state tile row pitch
    constexpr int VPR = DCH / 16;                // input vectors per row and chunk
    constexpr int VPS = DCH * SB / 16;           // state vectors per row and chunk
    constexpr bool SMEM_TAB = TM != (int)TABLE_GLOBAL;
    extern __shared__ __align__(16) unsigned char dsmem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
#ifdef B2R_PROBE
    unsigned long long pr_entry;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(pr_entry));
#endif

    const WalkLayout lay = walk_layout(p, SB);
    const uint32_t base_s = (smem_u32(dsmem) + lay.align - 1) & ~(lay.align - 1);
    // bytes per zero-fill op: smaller ops spread more evenly over the chunk loop (one def: 58 ops of 2 KB, two per lane;
    // 1.45 -> 1.43 ms on config 1; 8 KB ops: 1.50 ms), but a lane defers at most two, so more defs keep 4 KB ops
    constexpr uint32_t ZOP = D == 1 ? 2048u : WALK_ZERO_BYTES;
    constexpr bool REPL = TM == (int)TABLE_REPL || TM == (int)TABLE_REPL16;   // one copy of every entry per lane
    constexpr bool E16 = TM == (int)TABLE_PLAIN16 || TM == (int)TABLE_REPL16;   // 16-bit entries: next << NSH | rare, next << NSH = next * stride
                                                                        // (else next << 16 | next * stride | rare)
    // TABLE_REPL16 is PAIR-PACKED: the entries of the adjacent states 2m and 2m+1 (same class) share one 32-bit word per lane, i.e. one
    // 128-byte block per state pair with lane l's word at + l*4 and state 2m+1 in its upper half.  Lane l then reads bank l whatever its
    // state (a 64-byte stride per state puts two lanes in one bank word and costs a replay whenever the two need different entries).
    // Entry = (next >> 1) << 7 | (next & 1) << 1 | rare: masked with EMASK it IS the byte offset of state `next` inside a class row.
    constexpr bool PAIR = TM == (int)TABLE_REPL16;
    constexpr uint32_t NSH = E16 ? 1u : 16u;                             // entry >> NSH = the state (not for PAIR: stof below)
    constexpr uint32_t EMASK = PAIR ? 0xFF82u : 0xFFFEu;                 // 16-bit entries: the bits of the state's byte offset
    auto stof = [](uint32_t e) -> uint32_t { return PAIR ? ((e >> 6) | ((e >> 1) & 1u)) : (e >> NSH); };   // entry -> state
    auto enc16 = [](uint32_t st) -> uint32_t { return PAIR ? (((st >> 1) << 7) | ((st & 1u) << 1)) : (st << 1); };   // state -> 16-bit entry (rare = 0)
    constexpr uint32_t stride = TM == (int)TABLE_REPL ? 128u : TM == (int)TABLE_REPL16 ? 64u : TM == (int)TABLE_PLAIN ? 4u : E16 ? 2u : 0u;
    const uint32_t cstride = REPL ? 128u : (p.cls_repl ? 128u : 4u);      // class-table entry stride (a constant for replicated tables)
    const uint32_t laneoff = REPL ? (uint32_t)lane * 4u : 0u;
    const uint32_t claneoff = (REPL || p.cls_repl) ? (uint32_t)lane * 4u : 0u;   // the class table holds 32-bit entries in either case
    constexpr bool CBINS = E16 && HM == (int)HIST_SMEM && D >= 2 && D <= 3;   // compact bins possible (walk_bin_cols decides)
    const uint32_t bcols = walk_bin_cols(p);

    // ---- stage the tables ----------------------------------------------------------------------------------------------
    if (SMEM_TAB) {
        constexpr uint32_t csh = REPL ? 5u : 0u;   // log2(copies)
        // (four global loads per thread in flight, then their stores: the shared-memory stores are compiler barriers, and a loop of
        //  load -> store round trips made the prologue of a one-string launch 100 us long)
        constexpr int SU = 4;
#pragma unroll
        for (int d = 0; d < D; d++) {
            const uint32_t n = p.def[d].num_classes * p.def[d].padded_states;
            const uint32_t t0 = base_s + lay.tab[d];
            for (uint32_t i0 = threadIdx.x; i0 < (n << csh); i0 += SU * blockDim.x) {
                uint32_t ev[SU];
#pragma unroll
                for (int u = 0; u < SU; u++) { const uint32_t i = i0 + u * blockDim.x; ev[u] = i < (n << csh) ? __ldg(p.def[d].hot + (i >> csh)) : 0u; }
#pragma unroll
                for (int u = 0; u < SU; u++) {
                    const uint32_t i = i0 + u * blockDim.x;
                    if (i >= (n << csh)) break;
                    const uint32_t idx = i >> csh, l = i & ((1u << csh) - 1u), e = ev[u];
                    // single-copy tables: row k is XOR-swizzled by its class (walk_swizzle) — lanes in the same state with
                    // different classes would otherwise all hit one bank (the row size is a power of two)
                    const uint32_t swz = REPL ? 0u : walk_swizzle(idx / p.def[d].padded_states, p.def[d].padded_states * stride);
                    if (PAIR) asm volatile("st.shared.u16 [%0], %1;" ::"r"(t0 + (idx >> 1) * 128 + l * 4 + (idx & 1u) * 2), "h"((unsigned short)(enc16(e >> 16) | (e & 1u))) : "memory");
                    else if (E16) asm volatile("st.shared.u16 [%0], %1;" ::"r"(t0 + ((idx * 2) ^ swz)), "h"((unsigned short)(((e >> 16) << 1) | (e & 1u))) : "memory");
                    else sts32(t0 + ((idx * stride) ^ swz) + l * 4, e | ((e >> 16) * stride));
                }
            }
        }
        const uint32_t ccsh = (REPL || p.cls_repl) ? 5u : 0u;             // log2(copies) of the class table
        for (uint32_t i0 = threadIdx.x; i0 < (256u << ccsh); i0 += SU * blockDim.x) {
            uint32_t kv4[SU][D];
#pragma unroll
            for (int u = 0; u < SU; u++) {
                const uint32_t i = i0 + u * blockDim.x;
#pragma unroll
                for (int d = 0; d < D; d++) kv4[u][d] = i < (256u << ccsh) ? (uint32_t)__ldg(p.def[d].byte_class + (i >> ccsh)) : 0u;
            }
#pragma unroll
            for (int u = 0; u < SU; u++) {
                const uint32_t i = i0 + u * blockDim.x;
                if (i >= (256u << ccsh)) break;
                const uint32_t c = i >> ccsh, l = i & ((1u << ccsh) - 1u);
                uint32_t v;
                if (D == 1) {
                    const uint32_t k = kv4[u][0], rb = p.def[0].padded_states * stride;
                    v = base_s + lay.tab[0] + k * rb + (REPL ? l * 4 : 0u) + (REPL ? 0u : walk_swizzle(k, rb));
                } else {
                    v = 0;
#pragma unroll
                    for (int d = 0; d < D; d++) v |= kv4[u][d] << (8 * d);
                    if (CBINS) v |= (bcols < 256u ? (uint32_t)__ldg(p.bin_of_byte + c) : c) << 24;   // the bin column of the byte
                }
                sts32(base_s + lay.cls + c * cstride + l * 4, v);
            }
        }
    }
    if (HM == (int)HIST_SMEM) {
#pragma unroll
        for (int d = 0; d < D; d++)
            for (uint32_t i = threadIdx.x; i < (p.def[d].num_states + 1) * bcols; i += blockDim.x) sts32(base_s + lay.hist[d] + i * 4, 0u);
    } else {
#pragma unroll
        for (int d = 0; d < D; d++)
            for (uint32_t i = threadIdx.x; i < (2u << p.hist_cache_log2); i += blockDim.x) sts32(base_s + lay.hist[d] + i * 4, 0u);
    }
    EmitTables<D> etb;
    const uint32_t zero_s = base_s + lay.zero;
    const bool fillw = p.fuse || p.fill_in_walk;                        // this kernel zero-fills the sparse columns of its tiles
    if (p.fuse) emit_tables_init<D>(p, dsmem + (base_s - smem_u32(dsmem)) + lay.emit, etb);
    if (fillw) {
        for (uint32_t i = threadIdx.x * 16; i < WALK_ZERO_BYTES; i += blockDim.x * 16) sts128(zero_s + i, 0u, 0u, 0u, 0u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // zero buffer -> visible to the TMA (async proxy)
    }
    __syncthreads();
    if (p.stagger_ns && warp) {
        // every warp has the same period (tile setup, walk, emit stage), so warps that start together stay in phase: all of them
        // walk (the shared-memory pipe saturates) and then all of them run the emit stage (it idles).  Offset starts keep them apart.
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        const unsigned long long until = t0 + (unsigned long long)warp * p.stagger_ns;
        do { __nanosleep(500); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1)); } while (t1 < until);
    }
    TileEmitter<D, ST> emitter(p, etb, lane);
    EmitTotals tot;

    const uint32_t M = p.max_chars;
    const uint32_t Mpad = (M + 15u) & ~15u;                             // rows written (row_pitch >= Mpad by contract)
    const uint32_t n_chunks = CH ? LONG_CHUNK / DCH : (Mpad + DCH - 1) / DCH;   // a slot never stores a row past LONG_CHUNK
    const uint64_t rp = p.row_pitch;
    const uint32_t cls_lane_s = base_s + lay.cls + claneoff;
    uint32_t tabl[D], rowb[D], hist_s[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        tabl[d] = base_s + lay.tab[d] + laneoff;
        rowb[d] = p.def[d].padded_states * stride;
        hist_s[d] = base_s + lay.hist[d];
    }
    const uint32_t in_s = base_s + lay.tiles + (uint32_t)warp * lay.per_warp;
    constexpr bool INPLACE = D == 1 && SB == 1;                         // states overwrite the consumed input bytes
    const uint32_t st_s = in_s + lay.st_off;
    const uint32_t stash_s = in_s + lay.stash_off + lane * 16;         // vector v of my stash at stash_s + v*512
    const int kv = lane % VPR, r0 = lane / VPR;                         // input staging: vector kv of rows r0 + (32/VPR)*i
    const int skv = lane % VPS, sr0 = lane / VPS;                       // state store:   vector skv of rows sr0 + (32/VPS)*i

    // one position of def d: `cur` is the entry that led to the current state, c the byte.  Returns the next entry.
    auto lookup = [&](int d, uint32_t cur, uint32_t c, uint32_t cent) -> uint32_t {
        if (SMEM_TAB) {
            uint32_t row;
            if (D == 1) row = cent;
            else {
                const uint32_t k = (cent >> (8 * d)) & 0xFFu;
                row = tabl[d] + k * rowb[d] + (REPL ? 0u : walk_swizzle(k, rowb[d]));
            }
            // XOR, not OR: the low bits of `row` of a single-copy table carry the class swizzle (they are zero otherwise)
            if (E16) { uint32_t e; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(e) : "r"((cur & EMASK) ^ row)); return e; }
            return lds32((cur & 0xFFFCu) ^ row);
        } else {
            const uint32_t k = __ldg(p.def[d].byte_class + c);
            return __ldg(p.def[d].hot + k * p.def[d].padded_states + stof(cur));
        }
    };
    const uint32_t cache_log2 = p.hist_cache_log2;
    auto count = [&](int d, uint32_t cur, uint32_t c, uint32_t cent) {
        if (CBINS) red_shared_inc(hist_s[d] + (stof(cur) * bcols + (cent >> 24)) * 4);
        else if (HM == (int)HIST_SMEM) red_shared_inc(hist_s[d] + ((stof(cur) << 8) | c) * 4);
        else {
            // bin cache: slot = {key, count}; a slot is claimed by the first key that hashes to it and never changes owner,
            // every other key of that slot goes to the global bins (exact either way)
            const uint32_t s = stof(cur);
            if (s < p.def[d].num_states) {
                const uint32_t key = ((s << 8) | c) + 1u;
                // keys and counts in two arrays (not {key, count} pairs: those would put every key in an even bank)
                const uint32_t slot = hist_s[d] + (((key * 0x9E3779B1u) >> (32 - cache_log2)) << 2);
                uint32_t owner = lds32(slot);
                if (owner == 0) {
                    asm volatile("atom.shared.cas.b32 %0, [%1], 0, %2;" : "=r"(owner) : "r"(slot), "r"(key) : "memory");
                    if (owner == 0) owner = key;
                }
                if (owner == key) red_shared_inc(slot + (4u << cache_log2));
                else atomicAdd(p.def[d].hist + (size_t)c * p.def[d].num_states + s, 1ull);
            }
        }
    };

#ifdef B2R_PROBE   // development aid (tools/README): where a warp's time goes, tile by tile; -DB2R_PROBE builds print it per warp
    auto gtime = [] { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };
    const unsigned long long pr_start = gtime();
    unsigned long long pr_sum[4] = {0, 0, 0, 0};
    uint32_t pr_tiles = 0;
#endif
    for (;;) {
#ifdef B2R_PROBE
        const unsigned long long pr_t0 = gtime();
#endif
        unsigned long long t64 = 0;
        if (lane == 0) t64 = atomicAdd(&p.counters->tile_counter, 1ull);
        t64 = __shfl_sync(0xffffffffu, t64, 0);
        if (t64 >= p.n_tiles) break;
        const uint64_t tile_base = t64 * 32;
        const uint64_t idx = tile_base + lane;
        const bool valid = idx < p.n_strings;
        uint64_t off = 0, end = 0;
        uint64_t ch_j = 0;                                              // chunked mode: the slot's string and chunk
        uint32_t ch_c = 0;
        bool ch_beyond = false;                                         // the slot starts past the string's final-state row
        if (valid && CH) {
            ch_j = idx / p.chunk_k; ch_c = (uint32_t)(idx - ch_j * p.chunk_k);
            const uint64_t so = p.offsets[ch_j], se = p.offsets[ch_j + 1];
            // a too-long string is walked as empty, as the batch walk does
            const uint64_t len = (se < so || se - so > (uint64_t)(p.chunk_max_chars - 1) || se > p.total_bytes) ? 0 : se - so;
            const uint64_t a = (uint64_t)ch_c * LONG_CHUNK;
            ch_beyond = a > len;
            off = so + (a < len ? a : len);
            end = so + (a + LONG_CHUNK < len ? a + LONG_CHUNK : len);
        } else if (valid) { off = p.offsets[idx]; end = p.offsets[idx + 1]; }
        // SURVEY 8(a) row 6: emit reports it; walk nothing.  Offsets that leave the byte buffer are treated the same way
        // (nothing outside [0, total_bytes) is ever read)
        const bool too_long = valid && (end < off || end - off > (uint64_t)(M - 1) || end > p.total_bytes);
        if (too_long) end = off;
        const uint32_t L = (uint32_t)(end - off);
        const uint32_t rows_here = (p.n_strings - tile_base < 32) ? (uint32_t)(p.n_strings - tile_base) : 32u;

        uint32_t cur[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            uint32_t f = (p.def[d].init_states && valid) ? (uint32_t)p.def[d].init_states[idx] : p.def[d].first_state;
            if (CH && ch_beyond) f = p.def[d].num_states;                 // dummy rows only
            cur[d] = E16 ? enc16(f) : (f << 16) | (f * stride);
        }

        // staging geometry
        const uint32_t shift = (uint32_t)(off & 15);
        const bool any_shift = __any_sync(0xffffffffu, shift != 0);
        const uint8_t* in_ptr[VPR];                                     // vector kv of chunk 0 of row r0 + (32/VPR)*i
        uint32_t in_left[VPR];                                          // bytes from there to the end of that string
#pragma unroll
        for (int i = 0; i < VPR; i++) {
            const int row = r0 + (32 / VPR) * i;
            const uint64_t roff = __shfl_sync(0xffffffffu, off, row);
            const uint64_t rend = __shfl_sync(0xffffffffu, end, row);
            const uint64_t a = (roff & ~uint64_t(15)) + (uint32_t)kv * 16;
            in_ptr[i] = p.bytes + a;
            in_left[i] = rend > a ? (uint32_t)(rend - a) : 0u;
        }
        // chunked mode: where the rows of the slots this lane stores go in the batch columns, and how many of them there are
        uint64_t ch_base[VPS];
        uint32_t ch_rows[VPS];
        if (CH) {
            const uint32_t Mpad_b = (p.chunk_max_chars + 15u) & ~15u;
#pragma unroll
            for (int i = 0; i < VPS; i++) {
                const int row = sr0 + (32 / VPS) * i;
                const uint64_t j = __shfl_sync(0xffffffffu, ch_j, row);
                const uint32_t c = __shfl_sync(0xffffffffu, ch_c, row);
                ch_base[i] = j * rp + (uint64_t)c * LONG_CHUNK;
                ch_rows[i] = Mpad_b - c * LONG_CHUNK < LONG_CHUNK ? Mpad_b - c * LONG_CHUNK : LONG_CHUNK;
            }
        }
        const uint64_t tail_a = (off & ~uint64_t(15)) + DCH;            // extra vector of this lane's own row (unaligned strings)
        const uint8_t* const my_tail = p.bytes + tail_a;
        const uint32_t my_tail_left = end > tail_a ? (uint32_t)(end - tail_a) : 0u;

        auto stage = [&](uint32_t chunk) {   // async copy of chunk `chunk` into input tile (chunk & 1)
            const uint32_t cbase = chunk * DCH;
            const uint32_t dst = in_s + (chunk & 1) * (32 * PITCH) + kv * 16;
#pragma unroll
            // src-size = the bytes of the string that are left (at most 16): nothing past the end of the string is read
            for (int i = 0; i < VPR; i++) cp_async16(dst + (r0 + (32 / VPR) * i) * PITCH, in_ptr[i] + cbase, cbase < in_left[i] ? min(16u, in_left[i] - cbase) : 0u);
            if (any_shift) cp_async16(in_s + (chunk & 1) * (32 * PITCH) + lane * PITCH + DCH, my_tail + cbase, cbase < my_tail_left ? min(16u, my_tail_left - cbase) : 0u);
            cp_async_commit();
        };
        stage(0);
        // fused emit stage, fill: the tile's rows of every sparse column are contiguous.  Zero them with TMA bulk stores from
        // the shared zero buffer, one per lane, now; they complete in the background while the tile is walked (ordinary
        // stores would queue in the LSU in front of the other warps' table lookups).
        // Each lane owns ops lane, lane+32, ... (numbered region by region).  Its first two are not issued here but spread
        // over the chunk loop (op j at chunk j * n_chunks / n_ops): a burst of ~30 ops per warp backs up the bulk-copy queue
        // (the issuing warps stall) and bunches the HBM writes in front of the other warps' input loads.
        uint8_t *dz_ptr0 = nullptr, *dz_ptr1 = nullptr;
        uint32_t dz_bytes0 = 0u, dz_bytes1 = 0u, dz_chunk0 = NO_POS, dz_chunk1 = NO_POS;
        if (fillw && !(p.debug & 1)) {
            const uint64_t cbytes = (uint64_t)rows_here * rp, bbytes = (uint64_t)rows_here * p.bitmap_pitch;
            uint8_t* reg_ptr[3 * D + 2];
            uint64_t reg_bytes[3 * D + 2];
#pragma unroll
            for (int d = 0; d < D; d++) {
                reg_ptr[3 * d] = p.def[d].substr_ids ? p.def[d].substr_ids + tile_base * rp : nullptr; reg_bytes[3 * d] = cbytes;
                reg_ptr[3 * d + 1] = p.def[d].start_enable ? p.def[d].start_enable + tile_base * p.bitmap_pitch : nullptr; reg_bytes[3 * d + 1] = bbytes;
                reg_ptr[3 * d + 2] = p.def[d].end_enable ? p.def[d].end_enable + tile_base * p.bitmap_pitch : nullptr; reg_bytes[3 * d + 2] = bbytes;
            }
            reg_ptr[3 * D] = p.masked_chars ? p.masked_chars + tile_base * rp : nullptr; reg_bytes[3 * D] = cbytes;
            reg_ptr[3 * D + 1] = p.masked_substr_ids ? p.masked_substr_ids + tile_base * rp : nullptr; reg_bytes[3 * D + 1] = cbytes;
            uint32_t total_ops = 0;
#pragma unroll
            for (int r = 0; r < 3 * D + 2; r++)
                if (reg_ptr[r]) total_ops += ((uint32_t)(reg_bytes[r] & ~15ull) + ZOP - 1) / ZOP;
            const bool spread = p.spread_fill && n_chunks > 1;
            const uint32_t sched_den = total_ops > n_chunks ? total_ops : n_chunks;
            uint32_t first = 0;
#pragma unroll
            for (int r = 0; r < 3 * D + 2; r++) {
                if (!reg_ptr[r]) continue;
                const uint32_t bulk_bytes = (uint32_t)(reg_bytes[r] & ~15ull);   // bitmap regions of a partial tile can end on a 4-byte boundary
                const uint32_t n_ops = (bulk_bytes + ZOP - 1) / ZOP;
                for (uint32_t op = (lane + 32u - (first & 31u)) & 31u; op < n_ops; op += 32) {
                    const uint32_t o = op * ZOP;
                    const uint32_t nb = bulk_bytes - o < ZOP ? bulk_bytes - o : ZOP;
                    const uint32_t j = first + op;                      // j % 32 == lane
                    if (spread && j < 64) {
                        const uint32_t at = j * n_chunks / sched_den;
                        if (j < 32) { dz_ptr0 = reg_ptr[r] + o; dz_bytes0 = nb; dz_chunk0 = at; }
                        else { dz_ptr1 = reg_ptr[r] + o; dz_bytes1 = nb; dz_chunk1 = at; }
                    } else {
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reg_ptr[r] + o), "r"(zero_s), "r"(nb) : "memory");
                    }
                }
                for (uint64_t o = bulk_bytes + (uint64_t)lane * 4; o < reg_bytes[r]; o += 128) *reinterpret_cast<uint32_t*>(reg_ptr[r] + o) = 0u;
                first += n_ops;
            }
        }

#ifdef B2R_PROBE
        cp_async_wait<0>();
        const unsigned long long pr_t1 = gtime();
#endif
        uint32_t fm = 0, fw0 = 0, fw1 = 0;                              // granule flags: current group of 32 granules, words 0 and 1
        uint32_t stash_g = NO_POS;                                      // granule kept in my stash
#pragma unroll 1
        for (uint32_t chunk = 0; chunk < n_chunks; chunk++) {
            const uint32_t cbase = chunk * DCH;
            if (chunk + 1 < n_chunks) { stage(chunk + 1); cp_async_wait<1>(); } else cp_async_wait<0>();
            __syncwarp();
            if (dz_chunk0 == chunk)
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dz_ptr0), "r"(zero_s), "r"(dz_bytes0) : "memory");
            if (dz_chunk1 == chunk)
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dz_ptr1), "r"(zero_s), "r"(dz_bytes1) : "memory");

            const uint32_t my_in = in_s + (chunk & 1) * (32 * PITCH) + lane * PITCH;
#pragma unroll 1
            for (int g = 0; g < DCH / 16; g++) {
                const uint32_t gbase = cbase + g * 16;
                if (gbase >= Mpad) break;
                if (!valid) continue;                                   // a lane without a string (partial tile): its rows are never stored; without this it would drag
                                                                        // the warp through the byte-by-byte ragged path in every granule (a one-string call: 196 us -> see DESIGN)
                uint32_t w[4];
                if (!any_shift) {
                    const uint4 v = lds128(my_in + g * 16);
                    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
                } else {
                    const uint32_t q = my_in + g * 16 + (shift & ~3u);
                    const uint32_t sh = (shift & 3u) * 8;
                    const uint32_t x0 = lds32(q), x1 = lds32(q + 4), x2 = lds32(q + 8), x3 = lds32(q + 12), x4 = lds32(q + 16);
                    w[0] = __funnelshift_r(x0, x1, sh); w[1] = __funnelshift_r(x1, x2, sh);
                    w[2] = __funnelshift_r(x2, x3, sh); w[3] = __funnelshift_r(x3, x4, sh);
                }
                uint32_t pk[D][4 * SB];
                uint32_t acc = 0;
                if (gbase + 16 <= L) {
                    // ---- hot path: 16 real characters, no data-dependent branch ---------------------------------------
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        uint32_t before[D][4];                          // the entry that led to the state of row 4q + j
                        // the class lookups of the word first: they do not depend on the state, and issue is in order — inside the
                        // chain each of them would add its latency to the dependent state lookup behind it
                        uint32_t cw[4], centw[4];
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            cw[j] = prmt(w[q], 0u, 0x4440u + j);
                            centw[j] = 0;
                            if (SMEM_TAB) centw[j] = lds32(cls_lane_s + cw[j] * cstride);
                        }
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const uint32_t c = cw[j], cent = centw[j];
#pragma unroll
                            for (int d = 0; d < D; d++) {
                                const uint32_t e = lookup(d, cur[d], c, cent);
                                if (HM == (int)HIST_SMEM && SB == 1 && !E16)   // bin index (state << 8 | byte) in one byte permute
                                    red_shared_inc(hist_s[d] + prmt(cur[d], w[q], 0x3324u + j) * 4);
                                else count(d, cur[d], c, cent);
                                before[d][j] = cur[d];
                                cur[d] = e;
                            }
                        }
#pragma unroll
                        for (int d = 0; d < D; d++) {
                            acc |= before[d][1] | before[d][2];           // entries of rows 4q, 4q+1 (3-input LOP3s)
                            acc |= before[d][3] | cur[d];                 // rows 4q+2, 4q+3
                            if (E16) {                                    // 16-bit entries: the state is stof(entry)
                                if (SB == 1) pk[d][q] = stof(before[d][0]) | (stof(before[d][1]) << 8) | (stof(before[d][2]) << 16) | (stof(before[d][3]) << 24);
                                else {
                                    pk[d][q * 2] = stof(before[d][0]) | (stof(before[d][1]) << 16);
                                    pk[d][q * 2 + 1] = stof(before[d][2]) | (stof(before[d][3]) << 16);
                                }
                            } else if (SB == 1) {                         // state bytes (entry byte 2) of four rows into one word
                                const uint32_t lo = prmt(before[d][0], before[d][1], 0x4462u), hi = prmt(before[d][2], before[d][3], 0x4462u);
                                pk[d][q] = prmt(lo, hi, 0x5410u);
                            } else {
                                pk[d][q * 2] = prmt(before[d][0], before[d][1], 0x7632u);
                                pk[d][q * 2 + 1] = prmt(before[d][2], before[d][3], 0x7632u);
                            }
                        }
                    }
                } else {
                    // ---- ragged end: characters, then the final-state row, then dummy rows -------------------------
#pragma unroll
                    for (int d = 0; d < D; d++)
#pragma unroll
                        for (int i = 0; i < 4 * SB; i++) pk[d][i] = 0;
                    uint32_t v0 = w[0], v1 = w[1], v2 = w[2], v3 = w[3];   // shifted along: no dynamic register indexing
#pragma unroll 1
                    for (int b = 0; b < 16; b++) {
                        const uint32_t pos = gbase + b;
                        const uint32_t c = v0 & 0xFFu;
                        v0 = __funnelshift_r(v0, v1, 8); v1 = __funnelshift_r(v1, v2, 8); v2 = __funnelshift_r(v2, v3, 8); v3 >>= 8;
                        uint32_t cent = 0;
                        if (SMEM_TAB && pos < L) cent = lds32(cls_lane_s + c * cstride);
#pragma unroll
                        for (int d = 0; d < D; d++) {
                            const uint32_t stv = (pos <= L) ? stof(cur[d]) : p.def[d].num_states;   // state, final state, then dummy
                            if (pos < L) {
                                const uint32_t e = lookup(d, cur[d], c, cent);
                                count(d, cur[d], c, cent);
                                acc |= e;
                                cur[d] = e;
                            }
                            // insert stv at element b of the pack: rotate the pack down by one element, put stv on top
                            if (SB == 1) {
                                pk[d][0] = __funnelshift_r(pk[d][0], pk[d][1], 8); pk[d][1] = __funnelshift_r(pk[d][1], pk[d][2], 8);
                                pk[d][2] = __funnelshift_r(pk[d][2], pk[d][3], 8); pk[d][3] = (pk[d][3] >> 8) | (stv << 24);
                            } else {
#pragma unroll
                                for (int i = 0; i < 7; i++) pk[d][i] = __funnelshift_r(pk[d][i], pk[d][i + 1], 16);
                                pk[d][7] = (pk[d][7] >> 16) | (stv << 16);
                            }
                        }
                    }
                }
#pragma unroll
                for (int d = 0; d < D; d++) {
                    const uint32_t a = INPLACE ? my_in + g * 16 : st_s + (d * 32 + lane) * SPITCH + g * 16 * SB;
                    sts128(a, pk[d][0], pk[d][1], pk[d][2], pk[d][3]);
                    if (SB == 2) sts128(a + 16, pk[d][4 * (SB - 1)], pk[d][4 * (SB - 1) + 1], pk[d][4 * (SB - 1) + 2], pk[d][4 * (SB - 1) + 3]);
                }
                const uint32_t gi = (cbase >> 4) + g;                   // granule index
                if (acc & 1u) {
                    fm |= 1u << (gi & 31);
                    if (D == 1 && p.fuse && stash_g == NO_POS) {        // keep the first flagged granule of my string for the emit stage
                        stash_g = gi;
                        sts128(stash_s, w[0], w[1], w[2], w[3]);
#pragma unroll
                        for (int d = 0; d < D; d++) {
                            sts128(stash_s + (1 + d * SB) * 512, pk[d][0], pk[d][1], pk[d][2], pk[d][3]);
                            if (SB == 2) sts128(stash_s + (2 + d * SB) * 512, pk[d][4 * (SB - 1)], pk[d][4 * (SB - 1) + 1], pk[d][4 * (SB - 1) + 2], pk[d][4 * (SB - 1) + 3]);
                        }
                    }
                }
            }
            __syncwarp();

            // store the state tile: coalesced 16-byte vectors, one 32-byte sector (u8) per row
#pragma unroll
            for (int d = 0; d < D; d++) {
                uint8_t* const col = reinterpret_cast<uint8_t*>(p.def[d].states);
#pragma unroll
                for (int i = 0; i < VPS; i++) {
                    const int row = sr0 + (32 / VPS) * i;
                    const uint32_t elem = cbase + (uint32_t)skv * (16 / SB);   // first row-element of this vector
                    bool mine = row < (int)rows_here && elem < (CH ? ch_rows[i] : Mpad);
                    if (!CH && p.segment_mode) {   // a chunk of a long string owns rows [0, len) only; the last chunk also the final-state row
                        const uint32_t rl = __shfl_sync(0xffffffffu, L, row);
                        mine = mine && (elem < rl || (tile_base + row + 1 == p.n_strings && elem < ((rl + 16u) & ~15u)));
                    }
                    if (mine) {
                        const uint4 v = lds128(INPLACE ? in_s + (chunk & 1) * (32 * PITCH) + row * PITCH + skv * 16 : st_s + (d * 32 + row) * SPITCH + skv * 16);
                        *reinterpret_cast<uint4*>(col + ((CH ? ch_base[i] : (tile_base + row) * rp) + elem) * SB) = v;
                    }
                }
            }
            // publish a word of granule flags every 32 granules and at the end of the rows
            const uint32_t gcount = (chunk + 1) * (DCH / 16);
            if ((gcount & 31u) == 0 || chunk + 1 == n_chunks) {
                const uint32_t wi = (gcount - 1) >> 5;
                if (wi == 0) fw0 = fm; else if (wi == 1) fw1 = fm;
                if (CH) {
                    if (valid && 2 * ch_c + wi < p.chunk_fm_words) p.fmask[(size_t)(2 * ch_c + wi) * p.chunk_stride + ch_j] = fm;
                } else if (valid && wi < p.fm_words && (!p.fuse || wi >= 2)) p.fmask[(size_t)wi * p.n_strings + idx] = fm;
                fm = 0;
            }
            __syncwarp();
        }
#ifdef B2R_PROBE
        const unsigned long long pr_t2 = gtime();
#endif
        // long-string path: the flag summary of the ordered emit stage (a tile of 32 chunks is exactly one summary word)
        if (p.segment_mode && p.summary && p.fm_words <= 2) {
            const uint32_t word = __ballot_sync(0xffffffffu, valid && (fw0 | fw1) != 0u);
            if (lane == 0) {
                p.summary[t64] = word;
                if (word) atomicOr(p.summary2 + (t64 >> 5), 1u << (t64 & 31u));
            }
        }
        // ---- fused emit stage: the tile's states are in L1/L2, its flags and final states in registers --------------------
        if (fillw) {
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // my zero-fill stores have completed ...
            __syncwarp();                                                 // ... and so have those of the other lanes
        }
        if (p.fuse) {
#ifdef B2R_PROBE
            const unsigned long long pr_t3 = gtime();
#endif
            uint32_t fin[D];
#pragma unroll
            for (int d = 0; d < D; d++) fin[d] = stof(cur[d]);
            emitter.run_tile(tile_base, valid, valid && !too_long, off, L, fw0, fw1, fin, tot, /*filled=*/true, stash_g, stash_s);
#ifdef B2R_PROBE
            const unsigned long long pr_t4 = gtime();
            pr_sum[0] += pr_t1 - pr_t0; pr_sum[1] += pr_t2 - pr_t1; pr_sum[2] += pr_t3 - pr_t2; pr_sum[3] += pr_t4 - pr_t3; pr_tiles++;
#endif
        }
    }
#ifdef B2R_PROBE
    if (lane == 0 && (blockIdx.x % 37) == 0 && p.n_tiles > 1000) {   // four CTAs: printing from every warp would stretch the kernel
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        printf("probe cta %3d sm %3u warp %2d tiles %2u | us: prologue %5.1f setup %6.1f walk %7.1f fillwait %6.1f emit %6.1f loop %7.1f\n", blockIdx.x, smid, warp, pr_tiles,
               (pr_start - pr_entry) * 1e-3, pr_sum[0] * 1e-3, pr_sum[1] * 1e-3, pr_sum[2] * 1e-3, pr_sum[3] * 1e-3, (gtime() - pr_start) * 1e-3);
    }
    const unsigned long long pr_loop_end = gtime();
#endif
    if (p.fuse) emit_publish<D>(p, etb, tot);

    // ---- flush the multiplicity bins: bin (s,c) of def d -> dense global histogram [c*S + s] -------------------------------
    if (HM != (int)HIST_SMEM) {
        __syncthreads();
#pragma unroll
        for (int d = 0; d < D; d++) {
            const uint32_t S = p.def[d].num_states;
            for (uint32_t i = threadIdx.x; i < (1u << cache_log2); i += blockDim.x) {
                const uint32_t key = lds32(hist_s[d] + i * 4), v = lds32(hist_s[d] + (4u << cache_log2) + i * 4);
                if (key && v) atomicAdd(p.def[d].hist + (size_t)((key - 1) & 255u) * S + ((key - 1) >> 8), (unsigned long long)v);
            }
        }
    }
    if (HM == (int)HIST_SMEM) {
        __syncthreads();
#pragma unroll
        for (int d = 0; d < D; d++) {
            const uint32_t S = p.def[d].num_states;
            if (CBINS && bcols < 256u) {   // compact bins: column k stands for byte bin_byte[k]; the last column is nobody's
                for (uint32_t i = threadIdx.x; i < S * bcols; i += blockDim.x) {
                    const uint32_t s = i / bcols, k = i - s * bcols;
                    const uint32_t v = lds32(hist_s[d] + i * 4);
                    if (v && k + 1 < bcols) atomicAdd(p.def[d].hist + (size_t)__ldg(p.bin_byte + k) * S + s, (unsigned long long)v);
                }
                continue;
            }
            for (uint32_t i = threadIdx.x; i < S * 256u; i += blockDim.x) {
                const uint32_t s = i >> 8, c = i & 255u;
                const uint32_t v = lds32(hist_s[d] + i * 4);
                if (v) atomicAdd(p.def[d].hist + (size_t)c * S + s, (unsigned long long)v);
            }
        }
    }
#ifdef B2R_PROBE
    __syncthreads();
    if (threadIdx.x == 0 && (blockIdx.x % 37) == 0 && p.n_tiles > 1000)
        printf("probe cta %3d: kernel entry -> tile loop %.1f us, epilogue (publish + bin flush, after the slowest warp of the CTA) %.1f us, entry -> exit %.1f us\n", blockIdx.x,
               (pr_start - pr_entry) * 1e-3, (gtime() - pr_loop_end) * 1e-3, (gtime() - pr_entry) * 1e-3);
#endif
}

}  // namespace b2r
