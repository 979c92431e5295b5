// Device-side parameter blocks shared by the kernels (walk.cuh, emit.cuh, kernels.cu) and api.cu.
//
// The batch path is three launches:
//   walk_kernel     (walk.cuh)   bytes -> state columns + one "granule flag" bit per 16 rows + multiplicity bins
//   emit_kernel     (emit.cuh)   state columns + flags -> every other witness column, status, records, endpoint counters
//   finalize_kernel (kernels.cu) dense bins -> multiplicities in the reference's table-row order
#pragma once
#include <cstdint>

#include "../../include/b2r.h"

namespace b2r {

struct DefDev {
    // class-compressed tables of defs.hpp (emit + diagnose): entry = next | substr id | is_start | is_end | invalid
    const uint8_t* byte_class;       // [256]
    const uint32_t* trans;           // [num_classes][num_states]
    // walk table: [num_classes][padded_states], entry = next << 16 | rare (bit 0); next == num_states is the trap state
    const uint32_t* hot;
    uint32_t num_states;             // S (= dummy state value = trap state index)
    uint32_t num_classes;
    uint32_t padded_states;          // P: power of two >= S + 1
    uint32_t first_state;
    uint32_t accepted_state;
    uint32_t sid_offset;
    uint32_t num_substrs;
    const uint16_t* init_states;     // segment mode: state in which string j starts (null: first_state)
    uint32_t hot_states[2];          // bit s: some transition out of state s (< 64) carries a substr id (emit.cuh prefilter)
    unsigned long long* hist;        // dense [256][S] multiplicity bins (global, u64)
    unsigned long long* ep_start;    // [num_substrs][S] start-endpoint counters
    unsigned long long* ep_end;      // [num_substrs][S]
    // outputs
    void* states;                    // never null inside the library (scratch column when the caller passes NULL)
    uint8_t* substr_ids;
    uint8_t* start_enable;
    uint8_t* end_enable;
};

struct BatchCounters {               // zeroed before every batch (one memset node)
    unsigned long long first_bad_inv; // ~(lowest string index with an invalid transition / too long), kept with atomicMax; 0 = none
    unsigned long long n_overlap;
    unsigned long long pad_rows;     // sum over strings of (M - len): multiplicity of table row 0
    unsigned long long n_ok_strings; // strings that were processed to the end
    unsigned long long tile_counter; // next tile of 32 strings to hand out (dynamic scheduling of the persistent walk CTAs)
    unsigned long long emit_tile_counter;   // the same for emit_kernel
    unsigned long long reserved[2];
    __host__ __device__ bool any_bad() const { return first_bad_inv != 0; }
    __host__ __device__ unsigned long long first_bad() const { return ~first_bad_inv; }
};

struct WalkParams {
    const uint8_t* bytes;
    const uint64_t* offsets;
    uint64_t n_strings;
    uint64_t total_bytes;
    uint64_t row_pitch, bitmap_pitch;
    uint32_t max_chars;              // M
    uint32_t n_defs;
    DefDev def[B2R_MAX_DEFS];
    uint8_t* masked_chars;
    uint8_t* masked_substr_ids;
    b2r_string_status* status;
    b2r_substr_record* records;
    uint8_t* compact_bytes;
    uint32_t max_records, compact_pitch;
    BatchCounters* counters;
    uint32_t n_tiles;                // ceil(n_strings / 32)
    // granule flags: bit g of string j says rows [16g, 16g+16) contain a row with a non-zero substr id or an invalid
    // transition in some def.  Word w of string j lives at fmask[w * n_strings + j]; fm_words = ceil(ceil((M-1)/16) / 32).
    uint32_t* fmask;
    uint32_t fm_words;
    uint32_t table_mode;             // TABLE_REPL / TABLE_REPL16 / TABLE_PLAIN / TABLE_PLAIN16 / TABLE_GLOBAL (walk.cuh)
    // two or three defs on 16-bit tables with shared-memory bins: the bins have one column per byte that SOME def can read (bin_cols - 1
    // of them, plus one column for every other byte) instead of 256; the column of a byte rides in the spare byte of the class-table entry
    uint32_t bin_cols;               // columns of the compact bins (<= 256)
    const uint8_t* bin_of_byte;      // [256] byte -> column (device)
    const uint8_t* bin_byte;         // [bin_cols - 1] column -> byte (device)
    uint32_t cls_repl;               // single-copy tables: the byte -> class table is still replicated once per lane (32 KB) when that costs no warp
    uint32_t hist_mode;              // HIST_NONE / HIST_SMEM / HIST_GLOBAL
    uint32_t hist_cache_log2;        // HIST_GLOBAL: log2 of the slots of the per-def shared-memory bin cache in front of L2
    uint32_t ep_smem_bytes;          // bytes of shared memory for the endpoint counters (0: count with global atomics)
    uint32_t emit_smem_tables;       // 1: emit_kernel stages byte_class / trans in shared memory
    uint32_t segment_mode;           // 1: the "strings" are consecutive chunks of ONE long string (long.cuh): string j starts in
                                     //    init_states[j], stores only its own rows (the last one also the final state), no emit stage
    uint32_t* summary;               // segment mode: one bit per chunk "has a flagged granule" (one word per tile), and
    uint32_t* summary2;              //   one bit per summary word (zeroed by the caller); null: not wanted
    uint32_t fuse;                   // 1: walk_kernel runs the emit stage itself, tile by tile (no emit_kernel launch)
    uint32_t fill_in_walk;           // fuse == 0: walk_kernel still zero-fills the sparse columns of its tiles (TMA stores spread over the chunk loop,
                                     //   as in fused mode); emit_kernel then runs with prefilled = 1 and only scans
    uint32_t prefilled;              // 1: the sparse columns were zeroed before the emit stage runs (long-string path: memset)
    uint32_t spread_fill;            // 1: the fused zero-fill ops are issued across the chunk loop instead of in one burst per tile
    uint32_t stagger_ns;             // warp w of a CTA starts w * stagger_ns late: the warps' walk and emit phases interleave instead of coinciding
    uint32_t debug;                  // timing experiments only (B2R_DEBUG env): emit skips 1 zero-fill, 2 scan, 4 final-state loads, 8 status
    // chunked batch mode (b2r_match_batch_chunked, walk_kernel<..., CH = true>): the "strings" are slots of LONG_CHUNK rows, slot k =
    // chunk k % chunk_k of batch string k / chunk_k (offsets = the batch's string offsets).  A slot starts in init_states[k], stores its
    // rows of the batch row (final state at the string's length, dummy after) and its two flag words in the batch layout
    // (word w of slot c of string j at fmask[(2c + w) * chunk_stride + j])
    uint32_t chunk_k;                // slots per string: ceil(M / LONG_CHUNK)
    uint32_t chunk_fm_words;         // fm_words of the batch (M rows)
    uint32_t chunk_max_chars;        // M of the batch (too-long rule, rows stored)
    uint64_t chunk_stride;           // N of the whole batch (the flag-word stride)
};

constexpr uint32_t TABLE_REPL = 0;   // shared memory, one copy of every entry per bank (stride 128 B): conflict-free lookups
constexpr uint32_t TABLE_PLAIN = 1;  // shared memory, one copy (stride 4 B)
constexpr uint32_t TABLE_GLOBAL = 2; // global memory (L1/L2)
constexpr uint32_t TABLE_PLAIN16 = 3; // shared memory, one copy of 16-bit entries (next << 1 | rare): half the size, for large DFAs
constexpr uint32_t TABLE_REPL16 = 4;  // shared memory, 16-bit entries replicated once per lane, the entries of two adjacent states in one 32-bit word per lane
                                      // (lane l always reads bank l): conflict-free lookups at half the footprint of TABLE_REPL — several small DFAs side by side
// HIST_SMEM: dense bins [state][byte] in shared memory.  HIST_GLOBAL (bins too large for that): 64-bit atomics on the global
// bins, behind a shared-memory cache of (key, count) slots that absorbs the hot (byte, state) pairs.
constexpr uint32_t HIST_NONE = 0, HIST_SMEM = 1, HIST_GLOBAL = 2;

struct FinalizeParams {
    uint32_t n_defs;
    uint32_t accumulate;
    uint64_t n_rows_total;           // N*M, for the endpoint row-0 counts
    const BatchCounters* counters;
    BatchCounters* counters_copy;    // optional: a copy of the batch counters next to the outputs (small-batch host path: one D2H copy)
    struct {
        const unsigned long long* hist;
        const uint32_t* row_bin;     // [T]
        uint32_t n_rows;             // T
        const unsigned long long *ep_start, *ep_end;
        const uint32_t *erow_start_bin, *erow_end_bin;
        uint32_t n_erows;            // E
        unsigned long long* mult;    // out [T] or null
        unsigned long long* endpoint_mult;  // out [2E] or null
    } def[B2R_MAX_DEFS];
};

struct LaunchInfo {
    int grid, block;
    size_t smem_bytes;
};

// host-callable launchers (kernels.cu / walk_inst.cu)
// chooses table_mode / hist_mode for this device (force_* >= 0: preferred placement, testing hook); 0 or an error
int device_limits(int* n_sm, int* max_smem);   // SM count and opt-in shared memory per block of the current device
int plan_walk(WalkParams& p, bool wide_states, int force_table_mode, int force_hist_mode, int hist_cache_log2);
int launch_walk(const WalkParams& p, bool wide_states, void* stream, LaunchInfo* chosen);
int launch_emit(const WalkParams& p, bool wide_states, void* stream, LaunchInfo* chosen);
int launch_finalize(const FinalizeParams& p, void* stream);
int launch_diagnose(const WalkParams& p, uint64_t string_idx, b2r_batch_status* d_out, void* stream);

}  // namespace b2r
