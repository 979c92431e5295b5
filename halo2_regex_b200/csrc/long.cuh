// Long-string path (b2r_match_long; BASELINE config "single 64 MiB string"): ONE string of `len` bytes, M = len + 1 rows.
//
// The walk is a dependent chain over the whole string, so it is cut into chunks of LONG_CHUNK bytes:
//   1. long_maps_*_kernel    every chunk's transition vector f_k : S -> S (state after the chunk for EVERY state before
//                            it): all states over a 64-byte head, then only the distinct images over the rest;
//   2. long_compose_kernel   parallel-prefix composition, 64-ary tree: level l+1 map i = f of its 64 children composed;
//      long_propagate_kernel back down the tree: the state in which every node starts, from first_state at the root;
//   3. walk_kernel           in segment mode: chunk k is "string" k, starts in its now-known entry state, writes its slice
//                            of the single state row, its granule flags and the multiplicity bins (walk.cuh);
//   4. long_summary_kernel + long_emit_kernel   the emit stage for one string whose flags are spread over the chunks:
//                            one warp, flagged granules visited in order (emit.cuh's LaneString), after the sparse
//                            columns were zeroed with a memset.  The boundary stream of the mask algebra is sequential;
//                            the flagged granules are few.
#pragma once   // declarations only: the kernels live in long.cu
#include <cuda_runtime.h>

#include <cstdint>

#include "kernels.cuh"

namespace b2r {

constexpr uint32_t LONG_CHUNK = 1024;      // bytes per chunk: a multiple of 32 (whole 32-row windows), <= 1024 (two flag words)
constexpr uint32_t LONG_FANOUT = 64;

struct LongParams {
    const uint8_t* bytes;
    uint64_t len;
    uint32_t n_chunks;
    uint32_t n_defs;
    struct {
        const uint8_t* byte_class;
        const uint32_t* trans;           // [C][S] packed entries (defs.hpp)
        uint32_t num_states, first_state, num_classes;
        uint16_t* maps;                  // all levels back to back: level 0 [n_chunks][S+1], level 1 [ceil(n/64)][S+1], ...
        uint16_t* entry;                 // all levels back to back: entry state of every node
    } def[B2R_MAX_DEFS];
    uint64_t* offsets;                   // [n_chunks + 1]
    // scratch of the transition-vector pass (reused by every def): distinct images per chunk, their count, image index per state
    uint16_t* uniq;                      // [n_chunks][4]
    uint8_t* n_uniq;                     // [n_chunks]
    uint8_t* which;                      // [n_chunks][max S + 1]
    // fused prefix pass (small DFAs, long_fused_ok): per group of LONG_GROUP chunks the exclusive prefixes of the chunk maps
    // [n_chunks][SP] (SP = 16 or 32 bytes per map), the group aggregates [n_groups][SP], the aggregates of LONG_SUPER groups
    // [n_supers][SP], and one arrival counter per super group (zeroed before the pass)
    uint8_t* excl;
    uint8_t* agg;
    uint8_t* super;
    uint32_t* super_cnt;
    uint32_t fused;                      // 1: the fused pass is used (decided by long_plan)
    // chunked batch (b2r_match_batch_chunked): chunk k is slot k % chunk_k of string k / chunk_k, whose bytes are
    // [str_offsets[j], str_offsets[j+1]) (a string longer than max_chars - 1, or outside [0, total_bytes), has none); 0: one string
    uint32_t chunk_k;
    uint32_t max_chars;
    const uint64_t* str_offsets;
    uint64_t total_bytes;
};

constexpr uint32_t LONG_GROUP = 256;       // chunks per CTA of the fused prefix pass (16 warps share one copy of the replicated tables)
constexpr uint32_t LONG_SUB = 512;         // bytes per thread of the fused prefix pass (a sub-chunk)
constexpr uint32_t LONG_FUSED_THREADS = LONG_GROUP * (LONG_CHUNK / LONG_SUB);
constexpr uint32_t LONG_SUPER = 32;        // groups per super group

// fused prefix pass: usable when every def has at most 31 states and its bank-replicated tables fit next to four CTAs' maps
bool long_fused_ok(const LongParams& lp);

// host-callable (long.cu)
int launch_long_prepare(const LongParams& lp, void* stream, uint32_t* launches);
// summary: one bit per chunk ("has a flagged granule"), summary2: one bit per summary word (zeroed by the caller, as are the super-group counters)
int launch_long_emit(const WalkParams& p, bool wide, const uint32_t* fmask_chunks, uint32_t* summary, uint32_t* summary2, uint32_t n_chunks, uint32_t chunk_fm_words, void* stream, uint32_t* launches);
size_t long_level_nodes(uint32_t n_chunks);   // total nodes over all tree levels

}  // namespace b2r
