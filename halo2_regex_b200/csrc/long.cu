// Launchers of the long-string path (long.cuh).
#include "long.cuh"

#include <algorithm>
#include <type_traits>
#include <vector>

#include "defs.hpp"
#include "emit.cuh"

namespace b2r {

// chunk offsets for the walk kernel
__global__ void long_offsets_kernel(uint64_t* offsets, uint32_t n_chunks, uint64_t len) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n_chunks) { const uint64_t o = (uint64_t)i * LONG_CHUNK; offsets[i] = o < len ? o : len; }
    if (i == 0) { offsets[n_chunks + 1] = 0; offsets[n_chunks + 2] = len; }   // the {0, len} pair of the whole string (emit stage)
}

// f_k[s] for every chunk k and state s in [0, S]; S is the trap state (an invalid transition, sticky).
// The S+1 walks of a chunk merge quickly (the shipped DFAs are down to <= 2 distinct images after a few bytes), so the
// transition vector is computed in three steps:
//   head   thread per (chunk, state): walk the first LONG_HEAD bytes                       -> maps[k][s] = image after the head
//   dedupe thread per chunk: the distinct images (at most LONG_MAXU, else the chunk is marked wide) and, per state, which one
//   tail   thread per (chunk, distinct image): walk the rest of the chunk; wide chunks: thread per (chunk, state)
//   gather thread per (chunk, state): maps[k][s] = tail result of its image
constexpr uint32_t LONG_HEAD = 64;
constexpr uint32_t LONG_MAXU = 4;

__device__ __forceinline__ uint32_t long_walk(const LongParams& p, uint32_t d, uint32_t s, uint64_t a, uint64_t b) {
    const uint32_t S = p.def[d].num_states;
    const uint8_t* cls = p.def[d].byte_class;
    const uint32_t* tr = p.def[d].trans;
    for (uint64_t i = a; i < b && s < S; i++) {
        const uint32_t e = __ldg(tr + (uint32_t)__ldg(cls + __ldg(p.bytes + i)) * S + s);
        s = (e & ENT_INVALID) ? S : (e & ENT_NEXT_MASK);
    }
    return s;
}
__device__ __forceinline__ void long_chunk_range(const LongParams& p, uint32_t k, uint64_t& a, uint64_t& mid, uint64_t& b) {
    if (p.chunk_k) {   // chunked batch: slot c of string j (a too-long string has no bytes, as in the batch walk)
        const uint32_t j = k / p.chunk_k, c = k - j * p.chunk_k;
        const uint64_t so = p.str_offsets[j], se = p.str_offsets[j + 1];
        const uint64_t len = (se < so || se - so > (uint64_t)(p.max_chars - 1) || se > p.total_bytes) ? 0 : se - so;
        const uint64_t s0 = (uint64_t)c * LONG_CHUNK;
        a = so + (s0 < len ? s0 : len);
        b = so + (s0 + LONG_CHUNK < len ? s0 + LONG_CHUNK : len);
    } else {
        a = (uint64_t)k * LONG_CHUNK;
        b = a + LONG_CHUNK < p.len ? a + LONG_CHUNK : p.len;
    }
    mid = a + LONG_HEAD < b ? a + LONG_HEAD : b;
}

// ---- the same walks against tables staged in shared memory -----------------------------------------------------------------
// cls_s[byte] = class * (S+1) (u16), tr_s[class * (S+1) + s] = next state (u16; S = the sticky trap state, also the image of
// every invalid transition): one dependent shared-memory lookup per byte, no branch, the bytes read as 16-byte vectors one
// vector ahead.  Used when class * (S+1) fits 16 bits and the tables fit in shared memory (long_tables_bytes).
__host__ __device__ inline size_t long_tables_bytes(uint32_t S, uint32_t C) { return 512 + (size_t)C * (S + 1) * 2; }

__device__ __forceinline__ void long_tables_init(const LongParams& p, uint32_t d, uint16_t* cls_s, uint16_t* tr_s) {
    const uint32_t S = p.def[d].num_states, S1 = S + 1, C = p.def[d].num_classes;
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) cls_s[i] = (uint16_t)(p.def[d].byte_class[i] * S1);
    for (uint32_t i = threadIdx.x; i < C * S1; i += blockDim.x) {
        const uint32_t c = i / S1, st = i % S1;
        uint32_t nx = S;
        if (st < S) { const uint32_t e = p.def[d].trans[c * S + st]; nx = (e & ENT_INVALID) ? S : (e & ENT_NEXT_MASK); }
        tr_s[i] = (uint16_t)nx;
    }
    __syncthreads();
}

// N independent walks over the same bytes (the distinct images of one chunk): one class lookup per byte serves all of them
template <int N>
__device__ __forceinline__ void long_walk_n(const uint8_t* __restrict__ bytes, uint64_t a, uint64_t b, uint32_t (&s)[N], const uint16_t* cls_s,
                                            const uint16_t* tr_s) {
    auto step = [&](uint32_t c) {
#pragma unroll
        for (int n = 0; n < N; n++) s[n] = tr_s[c + s[n]];
    };
    uint64_t i = a;
    for (; i < b && ((uintptr_t)(bytes + i) & 15u); i++) step(cls_s[__ldg(bytes + i)]);
    auto step16 = [&](const uint4& v) {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint32_t c0 = cls_s[w[q] & 255u], c1 = cls_s[(w[q] >> 8) & 255u], c2 = cls_s[(w[q] >> 16) & 255u], c3 = cls_s[w[q] >> 24];
            step(c0); step(c1); step(c2); step(c3);
        }
    };
    // 64 bytes per round, the next round's four vectors in flight while this one is walked
    if (i + 64 <= b) {
        const uint4* q = reinterpret_cast<const uint4*>(bytes + i);
        uint4 n0 = __ldg(q), n1 = __ldg(q + 1), n2 = __ldg(q + 2), n3 = __ldg(q + 3);
        for (; i + 64 <= b; i += 64) {
            const uint4 v0 = n0, v1 = n1, v2 = n2, v3 = n3;
            if (i + 128 <= b) { q = reinterpret_cast<const uint4*>(bytes + i + 64); n0 = __ldg(q); n1 = __ldg(q + 1); n2 = __ldg(q + 2); n3 = __ldg(q + 3); }
            step16(v0); step16(v1); step16(v2); step16(v3);
        }
    }
    for (; i + 16 <= b; i += 16) step16(__ldg(reinterpret_cast<const uint4*>(bytes + i)));
    for (; i < b; i++) step(cls_s[__ldg(bytes + i)]);
}

__device__ __forceinline__ uint32_t long_walk_s(const uint8_t* __restrict__ bytes, uint64_t a, uint64_t b, uint32_t s0, const uint16_t* cls_s,
                                                const uint16_t* tr_s) {
    uint32_t s[1] = {s0};
    long_walk_n<1>(bytes, a, b, s, cls_s, tr_s);
    return s[0];
}

template <bool SMEM>
__global__ void __launch_bounds__(256) long_maps_head_kernel(const __grid_constant__ LongParams p, uint32_t d) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    uint16_t* cls_s = reinterpret_cast<uint16_t*>(long_smem);
    uint16_t* tr_s = cls_s + 256;
    if (SMEM) long_tables_init(p, d, cls_s, tr_s);
    const uint32_t S1 = p.def[d].num_states + 1;
    const uint64_t total = (uint64_t)p.n_chunks * S1;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t a, mid, b;
        long_chunk_range(p, (uint32_t)(t / S1), a, mid, b);
        p.def[d].maps[t] = (uint16_t)(SMEM ? long_walk_s(p.bytes, a, mid, (uint32_t)(t % S1), cls_s, tr_s) : long_walk(p, d, (uint32_t)(t % S1), a, mid));
    }
}

// uniq[k][0..LONG_MAXU): the distinct images of chunk k (count in n_uniq[k]; LONG_MAXU+1 = more than that: wide chunk);
// which[k*S1 + s]: index of the image of state s
__global__ void __launch_bounds__(256) long_dedupe_kernel(const __grid_constant__ LongParams p, uint32_t d, uint16_t* uniq, uint8_t* n_uniq, uint8_t* which) {
    const uint32_t S1 = p.def[d].num_states + 1;
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= p.n_chunks) return;
    const uint16_t* img = p.def[d].maps + (size_t)k * S1;
    uint16_t u[LONG_MAXU];
    uint32_t n = 0;
    for (uint32_t s = 0; s < S1 && n <= LONG_MAXU; s++) {
        const uint16_t v = img[s];
        uint32_t j = 0;
        while (j < n && u[j] != v) j++;
        if (j == n) { if (n < LONG_MAXU) u[n] = v; n++; }
        if (n <= LONG_MAXU) which[(size_t)k * S1 + s] = (uint8_t)j;
    }
    n_uniq[k] = (uint8_t)n;
    for (uint32_t j = 0; j < LONG_MAXU; j++) uniq[(size_t)k * LONG_MAXU + j] = j < n ? u[j] : 0;
}

// narrow chunks: thread per (chunk, distinct image) walks the rest of the chunk; result overwrites uniq
template <bool SMEM>
__global__ void __launch_bounds__(256) long_maps_tail_kernel(const __grid_constant__ LongParams p, uint32_t d, uint16_t* uniq, const uint8_t* n_uniq) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    uint16_t* cls_s = reinterpret_cast<uint16_t*>(long_smem);
    uint16_t* tr_s = cls_s + 256;
    if (SMEM) long_tables_init(p, d, cls_s, tr_s);
    if (SMEM) {
        // thread per chunk: its (<= 4) distinct images walk together
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < p.n_chunks; k += gridDim.x * blockDim.x) {
            const uint32_t n = n_uniq[k];
            if (n > LONG_MAXU) continue;
            uint64_t a, mid, b;
            long_chunk_range(p, k, a, mid, b);
            uint16_t* u = uniq + (size_t)k * LONG_MAXU;
            if (n == 1) { uint32_t s[1] = {u[0]}; long_walk_n<1>(p.bytes, mid, b, s, cls_s, tr_s); u[0] = (uint16_t)s[0]; }
            else if (n == 2) { uint32_t s[2] = {u[0], u[1]}; long_walk_n<2>(p.bytes, mid, b, s, cls_s, tr_s); u[0] = (uint16_t)s[0]; u[1] = (uint16_t)s[1]; }
            else {
                uint32_t s[4] = {u[0], u[1], u[2], n == 4 ? (uint32_t)u[3] : p.def[d].num_states};
                long_walk_n<4>(p.bytes, mid, b, s, cls_s, tr_s);
                for (uint32_t j = 0; j < n; j++) u[j] = (uint16_t)s[j];
            }
        }
        return;
    }
    const uint64_t total = (uint64_t)p.n_chunks * LONG_MAXU;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = (uint32_t)(t / LONG_MAXU), j = (uint32_t)(t % LONG_MAXU);
        if (j >= n_uniq[k] || n_uniq[k] > LONG_MAXU) continue;
        uint64_t a, mid, b;
        long_chunk_range(p, k, a, mid, b);
        uniq[t] = (uint16_t)long_walk(p, d, uniq[t], mid, b);
    }
}

// thread per (chunk, state): narrow chunks gather the result of their image, wide chunks walk the rest themselves
template <bool SMEM>
__global__ void __launch_bounds__(256) long_maps_gather_kernel(const __grid_constant__ LongParams p, uint32_t d, const uint16_t* uniq, const uint8_t* n_uniq, const uint8_t* which) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    uint16_t* cls_s = reinterpret_cast<uint16_t*>(long_smem);
    uint16_t* tr_s = cls_s + 256;
    if (SMEM) long_tables_init(p, d, cls_s, tr_s);
    const uint32_t S1 = p.def[d].num_states + 1;
    const uint64_t total = (uint64_t)p.n_chunks * S1;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = (uint32_t)(t / S1);
        if (n_uniq[k] <= LONG_MAXU) { p.def[d].maps[t] = uniq[(size_t)k * LONG_MAXU + which[t]]; continue; }
        uint64_t a, mid, b;
        long_chunk_range(p, k, a, mid, b);
        p.def[d].maps[t] = (uint16_t)(SMEM ? long_walk_s(p.bytes, mid, b, p.def[d].maps[t], cls_s, tr_s) : long_walk(p, d, p.def[d].maps[t], mid, b));
    }
}

// chunked batch: the map of every string's LAST slot becomes the constant map s -> first_state.  The composition over all slots
// then starts every string in first_state, and every other slot gets the composition of its own string's earlier slots only
// (no segmented scan); thread per (string, state)
__global__ void __launch_bounds__(256) long_reset_kernel(uint16_t* maps, uint32_t n_strings, uint32_t chunk_k, uint32_t S1, uint32_t first) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)n_strings * S1) return;
    const uint64_t j = t / S1, s = t - j * S1;
    maps[((j + 1) * chunk_k - 1) * S1 + s] = (uint16_t)first;
}

// level l+1 map i = composition of its (up to 64) children at level l; thread per (node, state)
__global__ void __launch_bounds__(256) long_compose_kernel(const uint16_t* child_maps, uint16_t* parent_maps, uint32_t n_child, uint32_t n_parent, uint32_t S1) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_parent * S1) return;
    const uint32_t i = t / S1;
    uint32_t s = t % S1;
    const uint32_t c0 = i * LONG_FANOUT, c1 = c0 + LONG_FANOUT < n_child ? c0 + LONG_FANOUT : n_child;
    for (uint32_t c = c0; c < c1; c++) s = child_maps[(size_t)c * S1 + s];
    parent_maps[t] = (uint16_t)s;
}

// entry states of the children of every node at level l+1, given the node's own entry state; thread per parent node
__global__ void __launch_bounds__(256) long_propagate_kernel(const uint16_t* child_maps, const uint16_t* parent_entry, uint16_t* child_entry, uint32_t n_child,
                                                              uint32_t n_parent, uint32_t S1) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_parent) return;
    uint32_t s = parent_entry[i];
    const uint32_t c0 = i * LONG_FANOUT, c1 = c0 + LONG_FANOUT < n_child ? c0 + LONG_FANOUT : n_child;
    for (uint32_t c = c0; c < c1; c++) { child_entry[c] = (uint16_t)s; s = child_maps[(size_t)c * S1 + s]; }
}

// the root of the composition tree starts in first_state.  Written by a kernel rather than copied from the host, so that the
// long-string path stays capturable in a CUDA graph (a captured host copy would read this call's stack variable at every replay)
__global__ void long_root_kernel(uint16_t* root_entry, uint32_t first) { *root_entry = (uint16_t)first; }

// The same tree with one CTA per parent node: a Hillis-Steele scan (composition is associative, not commutative: earlier
// children are applied first) over its <= 64 children in shared memory.  The child maps are replaced IN PLACE by their
// exclusive prefixes E_c = f_{c-1} o ... o f_0 (E_0 = identity); the parent gets the composition of all of them.
__global__ void __launch_bounds__(256) long_scan_kernel(uint16_t* child_maps, uint16_t* parent_maps, uint32_t n_child, uint32_t S1) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    uint16_t* A = reinterpret_cast<uint16_t*>(long_smem);
    uint16_t* B = A + (size_t)LONG_FANOUT * S1;
    const uint32_t c0 = blockIdx.x * LONG_FANOUT;
    const uint32_t nc = n_child - c0 < LONG_FANOUT ? n_child - c0 : LONG_FANOUT;
    const uint32_t tot = nc * S1;
    uint16_t* mine = child_maps + (size_t)c0 * S1;
    for (uint32_t i = threadIdx.x; i < tot; i += blockDim.x) A[i] = mine[i];
    __syncthreads();
    for (uint32_t o = 1; o < nc; o <<= 1) {
        for (uint32_t i = threadIdx.x; i < tot; i += blockDim.x) {
            const uint32_t c = i / S1, s = i - c * S1;
            B[i] = c >= o ? A[c * S1 + A[(c - o) * S1 + s]] : A[i];
        }
        __syncthreads();
        uint16_t* t = A; A = B; B = t;
    }
    for (uint32_t i = threadIdx.x; i < tot; i += blockDim.x) {
        const uint32_t c = i / S1, s = i - c * S1;
        mine[i] = c == 0 ? (uint16_t)s : A[(c - 1) * S1 + s];
    }
    for (uint32_t s = threadIdx.x; s < S1; s += blockDim.x) parent_maps[(size_t)blockIdx.x * S1 + s] = A[(nc - 1) * S1 + s];
}

// entry state of every chunk: first_state pushed down through the exclusive prefixes of its ancestors; thread per chunk
struct LongLevels { uint32_t n; uint32_t off[12]; };   // off[l]: first node of level l in `maps` (level 0 = chunks)
__global__ void __launch_bounds__(256) long_resolve_kernel(const uint16_t* maps, uint16_t* entry0, LongLevels lv, uint32_t n_chunks, uint32_t S1, uint32_t first) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    uint32_t s = first;
    for (int l = (int)lv.n - 2; l >= 0; l--) {
        uint32_t node = c;
        for (int k = 0; k < l; k++) node /= LONG_FANOUT;
        s = maps[((size_t)lv.off[l] + node) * S1 + s];
    }
    entry0[c] = (uint16_t)s;
}

// ---- fused prefix pass (small DFAs) ------------------------------------------------------------------------------------------
// ONE kernel computes every chunk's transition vector and the exclusive prefixes inside groups of LONG_GROUP chunks, a second
// (tiny) one pushes first_state through the group aggregates: 2 launches instead of 9.
//   thread = half a chunk.  All S states walk rounds of 32 bytes until at most 4 distinct images are left (the shipped DFAs collapse
//   in the first round), which then walk the rest of the chunk together; every lookup goes to BANK-REPLICATED tables (entry of
//   lane l in bank l, as in walk.cuh): 32 chunks with arbitrary bytes and states, one wavefront per lookup.
//   cls_r[byte][lane] = absolute shared address of (class row, state 0, this lane); tr_r[(class * P + state)][lane] = next state * 128.
template <int SP>
__global__ void __launch_bounds__(LONG_FUSED_THREADS, SP == 16 ? 2 : 1) long_maps_fused_kernel(const __grid_constant__ LongParams p, uint32_t d, uint32_t P, uint32_t n_groups) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    __shared__ uint32_t is_last, absorbing_s;
    __shared__ uint8_t wagg[(LONG_FUSED_THREADS / 32) * 32];              // aggregate of every warp's 32 maps
    const uint32_t S = p.def[d].num_states, C = p.def[d].num_classes;
    uint32_t* tr_r = reinterpret_cast<uint32_t*>(long_smem);
    uint32_t* cls_r = tr_r + (size_t)C * P * 32;                             // [256][32]: absolute shared address of (class row of the byte, state 0, lane)
    uint8_t* maps = reinterpret_cast<uint8_t*>(cls_r + 256 * 32);            // [LONG_FUSED_THREADS][SP], then the staging buffers
    const uint32_t lane = threadIdx.x & 31;
    {
        // the compact tables first (coalesced), then their per-lane copies out of shared memory
        const bool staged = (size_t)C * S * 4 + 256 <= (size_t)LONG_FUSED_THREADS * SP;
        uint32_t* tmp_tr = reinterpret_cast<uint32_t*>(maps + 256);
        if (threadIdx.x == 0) absorbing_s = 0;
        if (staged) {
            for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) maps[i] = p.def[d].byte_class[i];
            for (uint32_t i = threadIdx.x; i < C * S; i += blockDim.x) tmp_tr[i] = p.def[d].trans[i];
        }
        __syncthreads();
        // absorbing states (every class leads back to the state itself, e.g. an accepting sink): their image never has to be walked
        if (threadIdx.x < S) {
            bool fixed = true;
            for (uint32_t c = 0; c < C; c++) {
                const uint32_t t = staged ? tmp_tr[c * S + threadIdx.x] : p.def[d].trans[c * S + threadIdx.x];
                fixed = fixed && !(t & ENT_INVALID) && (t & ENT_NEXT_MASK) == threadIdx.x;
            }
            if (fixed) atomicOr(&absorbing_s, 1u << threadIdx.x);
        }
        {
            const uint32_t tr_s0 = (uint32_t)__cvta_generic_to_shared(tr_r);
            for (uint32_t i = threadIdx.x; i < 256 * 32; i += blockDim.x)
                cls_r[i] = tr_s0 + (uint32_t)(staged ? maps[i >> 5] : p.def[d].byte_class[i >> 5]) * P * 128u + (i & 31u) * 4u;
        }
        for (uint32_t i = threadIdx.x; i < C * P * 32; i += blockDim.x) {
            const uint32_t e = i >> 5, c = e / P, st = e % P;
            uint32_t nx = S;                                              // trap state: sticky, also the image of every invalid transition
            if (st < S) { const uint32_t t = staged ? tmp_tr[c * S + st] : p.def[d].trans[c * S + st]; nx = (t & ENT_INVALID) ? S : (t & ENT_NEXT_MASK); }
            tr_r[i] = nx * 128u;
        }
        __syncthreads();
    }
    const uint32_t absorbing = absorbing_s | (1u << S);                   // the trap state is sticky too
    const uint32_t cls_lane = (uint32_t)__cvta_generic_to_shared(cls_r) + lane * 4;
    // the tables are read-only from here on: plain (movable) loads, so that the class rows of a whole vector of bytes are
    // looked up ahead of the dependent chain of state lookups (issue is in order: a class lookup inside the chain would stall it)
    auto lds = [](uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; };
    // absolute shared address of (class row of `byte`, state 0, this lane)
    auto row_of = [&](uint32_t byte) { return lds(cls_lane + byte * 128u); };

    // input staging: the 32 half chunks of a warp are ONE contiguous 16 KB block.  It comes in through shared memory, 64 bytes of
    // every half chunk at a time, with coalesced 16-byte cp.async (four lanes per row: whole 64-byte pieces of four lines per
    // instruction instead of 32 different lines); lane l then reads ITS row with conflict-free LDS.128 (row pitch 80 bytes).
    constexpr uint32_t STAGE = 64, ROWP = STAGE + 16;
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(maps + LONG_FUSED_THREADS * SP) + (threadIdx.x >> 5) * (32u * ROWP);
    auto lds128 = [](uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v; };
    enum : uint32_t { MODE_ALL = 0, MODE_W0 = 1, MODE_W1 = 2, MODE_W2 = 3, MODE_W4 = 4 };

    for (uint32_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        // thread = sub-chunk of LONG_SUB bytes (half a chunk: twice the warps for the same chains)
        const uint32_t k = grp * LONG_FUSED_THREADS + threadIdx.x;
        if ((k & 1u) == 0 && (k >> 1) < p.n_chunks) p.offsets[k >> 1] = (uint64_t)(k >> 1) * LONG_CHUNK;   // chunk offsets for the walk kernel
        if (k == 0) { p.offsets[p.n_chunks] = p.len; p.offsets[p.n_chunks + 1] = 0; p.offsets[p.n_chunks + 2] = p.len; }   // + the {0, len} pair of the whole string
        uint32_t st[SP];
#pragma unroll
        for (int s = 0; s < SP; s++) st[s] = ((uint32_t)s < S ? (uint32_t)s : S) * 128u;
        uint32_t u0 = 0, u1 = 0, u2 = 0, u3 = 0, n = SP + 1;
        uint64_t which = 0;
        const uint64_t a = (uint64_t)k * LONG_SUB;
        const uint32_t mylen = a < p.len ? (uint32_t)(p.len - a < LONG_SUB ? p.len - a : LONG_SUB) : 0u;
        const uint64_t warp_a = (uint64_t)(k & ~31u) * LONG_SUB;           // first byte of the warp's block
        uint32_t mode = MODE_ALL, wa = 0, wb = 0;
        int ia = 0, ib = 1;

        // one 16-byte vector (or the last `avail` < 16 bytes of the string) in the lane's current mode
        auto all_states = [&](const uint4& v, uint32_t avail) {
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            if (avail == 16) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint32_t rows[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) rows[j] = row_of((w[q] >> (8 * j)) & 255u);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
#pragma unroll
                        for (int s = 0; s < SP; s++) st[s] = lds(rows[j] + st[s]);
                    }
                }
            } else {
                uint32_t x0 = w[0], x1 = w[1], x2 = w[2], x3 = w[3];
                for (uint32_t t = 0; t < avail; t++) {
                    const uint32_t cabs = row_of(x0 & 255u);
                    x0 = __funnelshift_r(x0, x1, 8); x1 = __funnelshift_r(x1, x2, 8); x2 = __funnelshift_r(x2, x3, 8); x3 >>= 8;
#pragma unroll
                    for (int s = 0; s < SP; s++) st[s] = lds(cabs + st[s]);
                }
            }
            n = 0; which = 0;
#pragma unroll
            for (int s = 0; s < SP; s++) {
                if ((uint32_t)s >= S) continue;                         // real states only: the trap state maps to itself
                const uint32_t x = st[s];
                uint32_t j = (n > 0 && x == u0) ? 0u : (n > 1 && x == u1) ? 1u : (n > 2 && x == u2) ? 2u : (n > 3 && x == u3) ? 3u : 4u;
                if (j == 4u) {
                    if (n == 0) u0 = x; else if (n == 1) u1 = x; else if (n == 2) u2 = x; else if (n == 3) u3 = x;
                    j = n; n++;
                }
                which |= (uint64_t)(j & 3u) << (2 * s);
            }
            if (n > 4) return;
            // at most four distinct images: from here on only those that are not absorbing states walk on
            if (n < 4) u3 = S * 128u;
            if (n < 3) u2 = S * 128u;
            if (n < 2) u1 = S * 128u;
            const bool f0 = (absorbing >> (u0 >> 7)) & 1u, f1 = (absorbing >> (u1 >> 7)) & 1u, f2 = (absorbing >> (u2 >> 7)) & 1u, f3 = (absorbing >> (u3 >> 7)) & 1u;
            const uint32_t moving = (f0 ? 0u : 1u) + (f1 ? 0u : 1u) + (f2 ? 0u : 1u) + (f3 ? 0u : 1u);
            mode = moving == 0 ? MODE_W0 : moving == 1 ? MODE_W1 : moving == 2 ? MODE_W2 : MODE_W4;
            if (moving == 1 || moving == 2) {
                ia = !f0 ? 0 : !f1 ? 1 : !f2 ? 2 : 3;
                ib = ia;
                if (moving == 2) ib = (!f1 && ia < 1) ? 1 : (!f2 && ia < 2) ? 2 : 3;
                wa = ia == 0 ? u0 : ia == 1 ? u1 : ia == 2 ? u2 : u3;
                wb = ib == 0 ? u0 : ib == 1 ? u1 : ib == 2 ? u2 : u3;
            }
        };
        auto walk_vec = [&](auto width_tag, const uint4& v, uint32_t avail) {
            constexpr int W = decltype(width_tag)::value;                 // 1, 2: wa (, wb); 4: u0..u3
            auto step_row = [&](uint32_t cabs) {
                if (W == 4) { u0 = lds(cabs + u0); u1 = lds(cabs + u1); u2 = lds(cabs + u2); u3 = lds(cabs + u3); }
                else { wa = lds(cabs + wa); if (W == 2) wb = lds(cabs + wb); }
            };
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            if (avail == 16) {
                uint32_t rows[16];
#pragma unroll
                for (int q = 0; q < 16; q++) rows[q] = row_of((w[q >> 2] >> (8 * (q & 3))) & 255u);
#pragma unroll
                for (int q = 0; q < 16; q++) step_row(rows[q]);
            } else {
                uint32_t x0 = w[0], x1 = w[1], x2 = w[2], x3 = w[3];
                for (uint32_t t = 0; t < avail; t++) {
                    step_row(row_of(x0 & 255u));
                    x0 = __funnelshift_r(x0, x1, 8); x1 = __funnelshift_r(x1, x2, 8); x2 = __funnelshift_r(x2, x3, 8); x3 >>= 8;
                }
            }
        };

        if (__any_sync(0xffffffffu, mylen != 0)) {
#pragma unroll 1
            for (uint32_t stg = 0; stg < LONG_SUB / STAGE; stg++) {       // warp-uniform: the staging is cooperative
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const uint32_t row = i * 8 + (lane >> 2), vv = lane & 3u;
                    const uint64_t g = warp_a + (uint64_t)row * LONG_SUB + stg * STAGE + vv * 16;
                    const uint32_t left = g < p.len ? (uint32_t)(p.len - g < 16 ? p.len - g : 16) : 0u;   // nothing past the end of the string is read
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(stage_s + row * ROWP + vv * 16), "l"(p.bytes + (left ? g : 0)), "r"(left) : "memory");
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
                if (__all_sync(0xffffffffu, mode == MODE_W1 && mylen >= (stg + 1) * STAGE)) {   // the common case, no per-vector checks
#pragma unroll
                    for (uint32_t r = 0; r < STAGE / 16; r++) walk_vec(std::integral_constant<int, 1>{}, lds128(stage_s + lane * ROWP + r * 16), 16u);
                    __syncwarp();
                    continue;
                }
#pragma unroll 1
                for (uint32_t r = 0; r < STAGE / 16; r++) {
                    const uint32_t pos = stg * STAGE + r * 16;
                    const uint32_t avail = mylen > pos ? (mylen - pos < 16 ? mylen - pos : 16u) : 0u;
                    if (!avail || mode == MODE_W0) continue;
                    const uint4 v = lds128(stage_s + lane * ROWP + r * 16);
                    if (mode == MODE_W1) walk_vec(std::integral_constant<int, 1>{}, v, avail);
                    else if (mode == MODE_ALL) all_states(v, avail);
                    else if (mode == MODE_W2) walk_vec(std::integral_constant<int, 2>{}, v, avail);
                    else walk_vec(std::integral_constant<int, 4>{}, v, avail);
                }
                __syncwarp();                                             // everybody is done with the buffer before it is refilled
            }
        }
        if (mode == MODE_W1 || mode == MODE_W2) { if (ia == 0) u0 = wa; else if (ia == 1) u1 = wa; else if (ia == 2) u2 = wa; else u3 = wa; }
        if (mode == MODE_W2) { if (ib == 1) u1 = wb; else if (ib == 2) u2 = wb; else u3 = wb; }
        if (mode == MODE_ALL) n = SP + 1;                                 // never collapsed (or no bytes at all): the vector of all states is the map
        // the chunk's transition vector as state indices (chunks past the end of the string, and an empty string: the identity)
        uint8_t* mine = maps + threadIdx.x * SP;
#pragma unroll
        for (int s = 0; s < SP; s++) {
            uint32_t v = st[s];
            if (n <= 4) { const uint32_t j = (uint32_t)(which >> (2 * s)) & 3u; v = j == 0 ? u0 : j == 1 ? u1 : j == 2 ? u2 : u3; }
            if ((uint32_t)s >= S) v = S * 128u;
            mine[s] = (uint8_t)(v >> 7);
        }
        __syncthreads();
        // ---- exclusive prefixes inside the group, in place, and the group aggregate: every warp scans its own 32 maps (lane =
        //      state), the warp aggregates are combined, and every warp applies the prefix of the warps before it ------------------
        {
            const uint32_t warp = threadIdx.x >> 5, c0 = warp * 32;
            uint32_t cur = lane < SP ? lane : 0u;
            for (uint32_t c = c0; c < c0 + 32; c++) {
                const uint32_t nxt = lane < SP ? maps[c * SP + cur] : 0u;
                __syncwarp();
                if (lane < SP) maps[c * SP + lane] = (uint8_t)cur;
                __syncwarp();
                cur = nxt;
            }
            if (lane < SP) wagg[warp * SP + lane] = (uint8_t)cur;
            __syncthreads();
            uint32_t pw = lane < SP ? lane : 0u;                           // composition of the warps in front of mine
            for (uint32_t v = 0; v < warp; v++) pw = wagg[v * SP + pw];
            if (warp > 0) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    uint32_t val[16];
#pragma unroll
                    for (int c = 0; c < 16; c++) val[c] = lane < SP ? maps[(c0 + 16 * h + c) * SP + pw] : 0u;
                    __syncwarp();
#pragma unroll
                    for (int c = 0; c < 16; c++) if (lane < SP) maps[(c0 + 16 * h + c) * SP + lane] = (uint8_t)val[c];
                    __syncwarp();
                }
            }
            if (warp == LONG_FUSED_THREADS / 32 - 1 && lane < SP) { p.agg[(size_t)grp * SP + lane] = wagg[warp * SP + pw]; __threadfence(); }
        }
        __syncthreads();
        {
            uint4* dst = reinterpret_cast<uint4*>(p.excl + (size_t)grp * LONG_FUSED_THREADS * SP);
            const uint4* src = reinterpret_cast<const uint4*>(maps);
            for (uint32_t i = threadIdx.x; i < LONG_FUSED_THREADS * SP / 16; i += blockDim.x) dst[i] = src[i];
        }
        // ---- the last group of a super group to arrive composes the super group's aggregate --------------------------------------------
        const uint32_t sg = grp / LONG_SUPER;
        const uint32_t g0 = sg * LONG_SUPER, g1 = g0 + LONG_SUPER < n_groups ? g0 + LONG_SUPER : n_groups;
        __syncthreads();
        if (threadIdx.x == 0) { __threadfence(); is_last = atomicAdd(p.super_cnt + sg, 1u) == g1 - g0 - 1u; }
        __syncthreads();
        if (is_last) {
            __threadfence();
            // the group aggregates in one round trip (the maps buffer is free again), then the chain in shared memory
            for (uint32_t i = threadIdx.x; i < (g1 - g0) * SP; i += blockDim.x) maps[i] = __ldcg(p.agg + (size_t)g0 * SP + i);
            __syncthreads();
            if (threadIdx.x < 32) {
                uint32_t cur = lane < SP ? lane : 0u;
                for (uint32_t g = 0; g < g1 - g0; g++) cur = maps[g * SP + cur];
                if (lane < SP) p.super[(size_t)sg * SP + lane] = (uint8_t)cur;
            }
        }
        __syncthreads();
    }
}

// entry state of every chunk: first_state through the super-group aggregates, then the group aggregates, then the chunk's exclusive
// prefix inside its group; CTA per group
__global__ void __launch_bounds__(LONG_GROUP) long_entry_kernel(const __grid_constant__ LongParams p, uint32_t d, uint32_t SP) {
    extern __shared__ __align__(16) unsigned char long_smem[];
    __shared__ uint32_t entry_s;
    const uint32_t b = blockIdx.x, sg = b / LONG_SUPER, g0 = sg * LONG_SUPER;
    const uint32_t n_stage = (sg + (b - g0)) * SP;                         // supers [0, sg), then groups [g0, b)
    for (uint32_t i = threadIdx.x; i < n_stage; i += blockDim.x)
        long_smem[i] = i < sg * SP ? __ldcg(p.super + i) : __ldcg(p.agg + (size_t)g0 * SP + (i - sg * SP));
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = p.def[d].first_state;
        for (uint32_t t = 0; t < sg + (b - g0); t++) s = long_smem[t * SP + s];
        entry_s = s;
    }
    __syncthreads();
    const uint32_t k = b * LONG_GROUP + threadIdx.x;
    if (k < p.n_chunks) p.def[d].entry[k] = (uint16_t)__ldcg(p.excl + (size_t)k * (LONG_CHUNK / LONG_SUB) * SP + entry_s);   // the prefix in front of its first sub-chunk
}

static size_t long_fused_smem(uint32_t C, uint32_t P, uint32_t SP) {   // tables, class table, maps, one staging buffer per warp
    return (size_t)256 * 128 + (size_t)C * P * 128 + (size_t)LONG_FUSED_THREADS * SP + (size_t)(LONG_FUSED_THREADS / 32) * 32 * 80;
}
static uint32_t long_padded(uint32_t S1) { uint32_t P = 1; while (P < S1) P <<= 1; return P; }

bool long_fused_ok(const LongParams& lp) {
    int n_sm = 0, max_smem = 0;
    if (device_limits(&n_sm, &max_smem)) return false;
    for (uint32_t d = 0; d < lp.n_defs; d++) {
        const uint32_t S1 = lp.def[d].num_states + 1;
        if (S1 > 32) return false;
        if (long_fused_smem(lp.def[d].num_classes, long_padded(S1), S1 <= 16 ? 16 : 32) > (size_t)max_smem) return false;
        if ((uint64_t)((lp.n_chunks + LONG_GROUP - 1) / LONG_GROUP / LONG_SUPER + LONG_SUPER) * 32 > 160 * 1024) return false;   // staging area of long_entry_kernel
    }
    return true;
}

// bit c of word w: chunk 32w + c has a flagged granule
// bit w of summary2 word v: summary word 32v + w is non-zero (summary2 is zeroed before the launch)
__global__ void __launch_bounds__(256) long_summary_kernel(const uint32_t* fmask, uint32_t fm_words, uint32_t n_chunks, uint32_t* summary, uint32_t* summary2) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t any = 0;
    if (c < n_chunks)
        for (uint32_t w = 0; w < fm_words; w++) any |= fmask[(size_t)w * n_chunks + c];
    const uint32_t word = __ballot_sync(0xffffffffu, any != 0);
    if ((threadIdx.x & 31) == 0 && c < n_chunks) {
        summary[c >> 5] = word;
        if (word) atomicOr(summary2 + (c >> 10), 1u << ((c >> 5) & 31u));
    }
}

// One warp: the emit stage of the single long string.  `p` describes the string as ONE string (n_strings = 1, offsets = {0, len},
// max_chars = len + 1); fmask holds the granule flags per chunk: word w of chunk c at fmask[w * n_chunks + c].
template <int D, typename ST>
__global__ void __launch_bounds__(128) long_emit_kernel(const __grid_constant__ WalkParams p, const uint32_t* summary, const uint32_t* summary2, uint32_t n_chunks, uint32_t chunk_fm_words) {
    extern __shared__ __align__(16) unsigned char esmem[];
    const int lane = threadIdx.x & 31;
    EmitTables<D> tb;
    emit_tables_init<D>(p, esmem, tb);                                  // all four warps stage the tables; warp 0 does the (ordered) work
    __syncthreads();
    if (threadIdx.x < 32) {
    const uint32_t L = p.max_chars - 1;
    constexpr uint32_t GPC = LONG_CHUNK / 16;                            // granules per chunk
    LaneString<D, ST> ls(p, tb, 0, p.bytes, L);
    uint32_t r_nrec = 0, r_ncmp = 0, r_flags = 0;
    bool patch = false;
    auto pass = [&](auto patch_tag) {
        constexpr bool PATCH = decltype(patch_tag)::value;
        ls.scan_begin();
        bool stop = false;                                               // warp-uniform: lane 0 hit an invalid transition
        const uint32_t n_words = (n_chunks + 31) / 32, n_words2 = (n_words + 31) / 32;
        // second level first, 32 words per load: stretches of 1024 chunks without a flagged granule cost nothing
        for (uint32_t v0 = 0; v0 < n_words2 && !stop; v0 += 32) {
            const uint32_t mine2 = v0 + lane < n_words2 ? __ldcg(summary2 + v0 + lane) : 0u;
            uint32_t lanes2 = __ballot_sync(0xffffffffu, mine2 != 0);
            while (lanes2 && !stop) {
                const int l2 = __ffs((int)lanes2) - 1;
                lanes2 &= lanes2 - 1;
                const uint32_t lvl2 = __shfl_sync(0xffffffffu, mine2, l2);
                const uint32_t w0 = (v0 + (uint32_t)l2) * 32;                // 32 summary words, one per lane
                const uint32_t mine = (w0 + lane < n_words && ((lvl2 >> lane) & 1u)) ? __ldcg(summary + w0 + lane) : 0u;
                uint32_t lanes = __ballot_sync(0xffffffffu, mine != 0);
                while (lanes && !stop) {
                    const int l = __ffs((int)lanes) - 1;
                    lanes &= lanes - 1;
                    uint32_t chunks = __shfl_sync(0xffffffffu, mine, l);
                    while (chunks && !stop) {
                        const uint32_t c = (w0 + l) * 32 + ((uint32_t)__ffs((int)chunks) - 1u);
                        chunks &= chunks - 1;
                        if (lane == 0) {
                            for (uint32_t w = 0; w < chunk_fm_words && !ls.invalid; w++) {
                                const uint32_t fw = p.fmask[(size_t)w * n_chunks + c];
                                uint32_t bits = fw;
                                while (bits && !ls.invalid) {
                                    const uint32_t g = (uint32_t)__ffs((int)bits) - 1u;
                                    bits &= bits - 1;
                                    ls.template scan_granule<PATCH>(c * GPC + w * 32 + g, (fw >> (g ^ 1u)) & 1u);
                                }
                            }
                        }
                        stop = __shfl_sync(0xffffffffu, (int)ls.invalid, 0) != 0;
                    }
                }
            }
        }
        if (lane == 0) ls.template scan_end<PATCH>();
    };
    pass(std::false_type{});
    if (lane == 0) {
        if (ls.invalid) r_flags = B2R_ST_INVALID_TRANSITION;
        else {
            if (ls.overlap) r_flags = B2R_ST_OVERLAP;
            patch = ls.n_seg > EMIT_NSEG;
            if (!patch) {
                ls.write_masks(); r_nrec = ls.n_rec; r_ncmp = ls.n_cmp;
                if (LaneString<D, ST>::SECTORS && p.compact_bytes && p.compact_pitch <= 8) ls.store_compact();
            }
        }
    }
    if (__any_sync(0xffffffffu, patch)) {
        pass(std::true_type{});
        if (lane == 0) { r_nrec = ls.n_rec; r_ncmp = ls.n_cmp; }
    }
    if (lane == 0 && (r_flags & B2R_ST_OVERLAP)) { r_nrec = 0; r_ncmp = 0; }   // no records for a string two defs flag on one row
    if (lane == 0) {
        uint32_t fin[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            fin[d] = (uint32_t)__ldcg(reinterpret_cast<const ST*>(p.def[d].states) + L);
            if (fin[d] >= p.def[d].num_states) r_flags = B2R_ST_INVALID_TRANSITION;
        }
        if (r_flags & B2R_ST_INVALID_TRANSITION) kill_string(p, 0);
        else {
            uint32_t flags = r_flags;
#pragma unroll
            for (int d = 0; d < D; d++)
                if (fin[d] == p.def[d].accepted_state) flags |= B2R_ST_ACCEPTED(d);
            if (p.records && r_nrec > p.max_records) flags |= B2R_ST_RECORDS_TRUNCATED;
            if (p.compact_bytes && r_ncmp > p.compact_pitch) flags |= B2R_ST_COMPACT_TRUNCATED;
            if (p.status) {
                b2r_string_status st = {};
                st.flags = flags; st.err_pos = NO_POS; st.n_records = r_nrec; st.n_compact = r_ncmp;
                p.status[0] = st;
            }
            atomicAdd(&p.counters->pad_rows, 1ull);                      // row len is the only row with enable = 0
            atomicAdd(&p.counters->n_ok_strings, 1ull);
            if (r_flags & B2R_ST_OVERLAP) atomicAdd(&p.counters->n_overlap, 1ull);
        }
    }
    }
    EmitTotals none;
    emit_publish<D>(p, tb, none);
}


size_t long_level_nodes(uint32_t n_chunks) {
    size_t total = 0;
    for (uint32_t n = n_chunks;; n = (n + LONG_FANOUT - 1) / LONG_FANOUT) { total += n; if (n <= 1) break; }
    return total;
}

#define LAUNCH_CHECK(what)                                                                                     \
    do {                                                                                                       \
        cudaError_t e_ = cudaGetLastError();                                                                   \
        if (e_ != cudaSuccess) { set_error(what " launch: %s", cudaGetErrorString(e_)); return B2R_ERR_CUDA; } \
    } while (0)

// chunk offsets, chunk maps, the composition tree and the entry states of every chunk (level 0 of `entry`)
int launch_long_prepare(const LongParams& lp, void* stream, uint32_t* launches) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!lp.fused && !lp.chunk_k) {   // the fused pass writes the chunk offsets itself; the chunked batch walk reads the string offsets
        long_offsets_kernel<<<(lp.n_chunks + 1 + 255) / 256, 256, 0, st>>>(lp.offsets, lp.n_chunks, lp.len);
        LAUNCH_CHECK("long_offsets_kernel"); (*launches)++;
    }
    for (uint32_t d = 0; d < lp.n_defs; d++) {
        const uint32_t S1 = lp.def[d].num_states + 1;
        const uint64_t threads = (uint64_t)lp.n_chunks * S1;
        if (lp.fused) {
            int n_sm = 0, max_smem = 0;
            { const int rc = device_limits(&n_sm, &max_smem); if (rc) return rc; }
            const uint32_t SP = S1 <= 16 ? 16u : 32u, P = long_padded(S1);
            const uint32_t n_groups = (lp.n_chunks + LONG_GROUP - 1) / LONG_GROUP, n_supers = (n_groups + LONG_SUPER - 1) / LONG_SUPER;
            const size_t smem = long_fused_smem(lp.def[d].num_classes, P, SP);
            auto kern = SP == 16 ? long_maps_fused_kernel<16> : long_maps_fused_kernel<32>;
            if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { set_error("cudaFuncSetAttribute(long_maps_fused_kernel)"); return B2R_ERR_CUDA; }
            // resident CTAs only (equal work per group: a static stride balances): the tables are staged once per CTA
            int per_sm = 1;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, (int)LONG_FUSED_THREADS, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
            const uint32_t grid = std::min<uint32_t>(n_groups, (uint32_t)(n_sm * per_sm));
            LongParams q = lp;
            q.super_cnt = lp.super_cnt + (size_t)d * n_supers;            // zeroed by the caller, one set of counters per def
            kern<<<grid, LONG_FUSED_THREADS, smem, st>>>(q, d, P, n_groups);
            LAUNCH_CHECK("long_maps_fused_kernel"); (*launches)++;
            const size_t esmem = (size_t)(n_supers + LONG_SUPER) * SP;
            if (esmem > 48 * 1024 && cudaFuncSetAttribute(long_entry_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)esmem) != cudaSuccess) { set_error("cudaFuncSetAttribute(long_entry_kernel)"); return B2R_ERR_CUDA; }
            long_entry_kernel<<<n_groups, LONG_GROUP, esmem, st>>>(lp, d, SP);
            LAUNCH_CHECK("long_entry_kernel"); (*launches)++;
            continue;
        }
        // tables in shared memory when they fit (and class * (S+1) fits the u16 of the class table)
        int n_sm = 0, max_smem = 0;
        { const int rc = device_limits(&n_sm, &max_smem); if (rc) return rc; }
        const size_t tb = long_tables_bytes(lp.def[d].num_states, lp.def[d].num_classes);
        const bool smem_ok = (uint64_t)lp.def[d].num_classes * S1 <= 65535u && tb <= (size_t)max_smem;
        const size_t smem = smem_ok ? tb : 0;
        const unsigned per_sm = smem_ok ? (unsigned)std::max<size_t>(1, std::min<size_t>(8, (size_t)max_smem / (tb + 1024))) : 8u;
        auto grid_for = [&](uint64_t work) { const uint64_t need = (work + 255) / 256, cap = (uint64_t)n_sm * per_sm; return (unsigned)std::max<uint64_t>(1, std::min(need, cap)); };
        // thread per chunk: small CTAs so that the chunks spread over all SMs
        auto grid_for_small = [&](uint64_t work) { const uint64_t need = (work + 63) / 64, cap = (uint64_t)n_sm * per_sm * 4; return (unsigned)std::max<uint64_t>(1, std::min(need, cap)); };
        if (smem > 48 * 1024) {
            if (cudaFuncSetAttribute(long_maps_head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(long_maps_tail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(long_maps_gather_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
                set_error("cudaFuncSetAttribute(long_maps_*_kernel)"); return B2R_ERR_CUDA;
            }
        }
        if (smem_ok) long_maps_head_kernel<true><<<grid_for(threads), 256, smem, st>>>(lp, d);
        else long_maps_head_kernel<false><<<grid_for(threads), 256, 0, st>>>(lp, d);
        LAUNCH_CHECK("long_maps_head_kernel"); (*launches)++;
        long_dedupe_kernel<<<(lp.n_chunks + 255) / 256, 256, 0, st>>>(lp, d, lp.uniq, lp.n_uniq, lp.which);
        LAUNCH_CHECK("long_dedupe_kernel"); (*launches)++;
        if (smem_ok) long_maps_tail_kernel<true><<<grid_for_small(lp.n_chunks), 64, smem, st>>>(lp, d, lp.uniq, lp.n_uniq);
        else long_maps_tail_kernel<false><<<grid_for((uint64_t)lp.n_chunks * LONG_MAXU), 256, 0, st>>>(lp, d, lp.uniq, lp.n_uniq);
        LAUNCH_CHECK("long_maps_tail_kernel"); (*launches)++;
        if (smem_ok) long_maps_gather_kernel<true><<<grid_for(threads), 256, smem, st>>>(lp, d, lp.uniq, lp.n_uniq, lp.which);
        else long_maps_gather_kernel<false><<<grid_for(threads), 256, 0, st>>>(lp, d, lp.uniq, lp.n_uniq, lp.which);
        LAUNCH_CHECK("long_maps_gather_kernel"); (*launches)++;
        if (lp.chunk_k) {
            const uint32_t n_str = lp.n_chunks / lp.chunk_k;
            long_reset_kernel<<<(unsigned)(((uint64_t)n_str * S1 + 255) / 256), 256, 0, st>>>(lp.def[d].maps, n_str, lp.chunk_k, S1, lp.def[d].first_state);
            LAUNCH_CHECK("long_reset_kernel"); (*launches)++;
        }
        // up the tree
        std::vector<uint32_t> n_level{lp.n_chunks};
        std::vector<size_t> off_level{0};
        while (n_level.back() > 1) {
            off_level.push_back(off_level.back() + n_level.back());
            n_level.push_back((n_level.back() + LONG_FANOUT - 1) / LONG_FANOUT);
        }
        const size_t scan_smem = 2 * (size_t)LONG_FANOUT * S1 * sizeof(uint16_t);
        if (scan_smem <= (size_t)max_smem && n_level.size() <= 12) {
            // one CTA per parent node: scan in shared memory, exclusive prefixes left in place of the child maps
            if (scan_smem > 48 * 1024 && cudaFuncSetAttribute(long_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem) != cudaSuccess) {
                set_error("cudaFuncSetAttribute(long_scan_kernel)"); return B2R_ERR_CUDA;
            }
            for (size_t l = 0; l + 1 < n_level.size(); l++) {
                long_scan_kernel<<<n_level[l + 1], 256, scan_smem, st>>>(lp.def[d].maps + off_level[l] * S1, lp.def[d].maps + off_level[l + 1] * S1, n_level[l], S1);
                LAUNCH_CHECK("long_scan_kernel"); (*launches)++;
            }
            LongLevels lv;
            lv.n = (uint32_t)n_level.size();
            for (size_t l = 0; l < n_level.size(); l++) lv.off[l] = (uint32_t)off_level[l];
            long_resolve_kernel<<<(lp.n_chunks + 255) / 256, 256, 0, st>>>(lp.def[d].maps, lp.def[d].entry, lv, lp.n_chunks, S1, lp.def[d].first_state);
            LAUNCH_CHECK("long_resolve_kernel"); (*launches)++;
            continue;
        }
        for (size_t l = 0; l + 1 < n_level.size(); l++) {
            const uint32_t nc = n_level[l], np = n_level[l + 1];
            long_compose_kernel<<<(np * S1 + 255) / 256, 256, 0, st>>>(lp.def[d].maps + off_level[l] * S1, lp.def[d].maps + off_level[l + 1] * S1, nc, np, S1);
            LAUNCH_CHECK("long_compose_kernel"); (*launches)++;
        }
        // the root starts in first_state; down the tree
        long_root_kernel<<<1, 1, 0, st>>>(lp.def[d].entry + off_level.back(), lp.def[d].first_state);
        LAUNCH_CHECK("long_root_kernel"); (*launches)++;
        for (size_t l = n_level.size() - 1; l-- > 0;) {
            const uint32_t nc = n_level[l], np = n_level[l + 1];
            long_propagate_kernel<<<(np + 255) / 256, 256, 0, st>>>(lp.def[d].maps + off_level[l] * S1, lp.def[d].entry + off_level[l + 1], lp.def[d].entry + off_level[l], nc, np, S1);
            LAUNCH_CHECK("long_propagate_kernel"); (*launches)++;
        }
    }
    return B2R_OK;
}

template <int D, typename ST>
static int launch_long_emit_one(const WalkParams& p, const uint32_t* summary, const uint32_t* summary2, uint32_t n_chunks, uint32_t chunk_fm_words, cudaStream_t st) {
    const size_t smem = emit_smem_bytes(p);
    auto kern = long_emit_kernel<D, ST>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(long_emit_kernel): %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    }
    kern<<<1, 128, smem, st>>>(p, summary, summary2, n_chunks, chunk_fm_words);
    LAUNCH_CHECK("long_emit_kernel");
    return B2R_OK;
}

int launch_long_emit(const WalkParams& p, bool wide, const uint32_t* fmask_chunks, uint32_t* summary, uint32_t* summary2, uint32_t n_chunks, uint32_t chunk_fm_words, void* stream, uint32_t* launches) {
    cudaStream_t st = (cudaStream_t)stream;
    if (fmask_chunks) {   // null: the segment walk has written the summary itself
        long_summary_kernel<<<(n_chunks + 255) / 256, 256, 0, st>>>(fmask_chunks, chunk_fm_words, n_chunks, summary, summary2);
        LAUNCH_CHECK("long_summary_kernel"); (*launches)++;
    }
    (*launches)++;
#define GO(D_) return wide ? launch_long_emit_one<D_, uint16_t>(p, summary, summary2, n_chunks, chunk_fm_words, st) : launch_long_emit_one<D_, uint8_t>(p, summary, summary2, n_chunks, chunk_fm_words, st)
    switch (p.n_defs) {
        case 1: GO(1);
        case 2: GO(2);
        case 3: GO(3);
        case 4: GO(4);
    }
#undef GO
    set_error("unsupported number of defs %u", p.n_defs);
    return B2R_ERR_UNSUPPORTED;
}

}  // namespace b2r
