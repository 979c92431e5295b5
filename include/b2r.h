/*
 * b2r.h — C ABI of the B200-native DFA witness-generation path for zkemail/halo2-regex.
 *
 * This is the drop-in boundary: a Rust (or any FFI-capable) host keeps the reference's
 * `RegexVerifyConfig / AllstrRegexDef / SubstrRegexDef` API and replaces only
 *   - the definition loaders          (reference src/defs.rs:54-110, 184-265),
 *   - the table row materialisation   (reference src/table.rs:61-198),
 *   - the assignment-value derivation (reference src/lib.rs:316-318 `derive_states`,
 *     `derive_substr_ids`, `derive_is_start_end`, the padding rules :339-348/:388-418, the
 *     accept rule :427-457, the cross-def sums :459-519 and the mask scans :593-764)
 * with calls into this library.  Cell assignment (halo2) stays in the host.
 *
 * Conventions
 *   - every function returns an int: 0 (B2R_OK) or a negative B2R_ERR_* code; the library never aborts
 *     and never throws across the boundary; b2r_last_error() returns a thread-local message.
 *   - the caller allocates every input/output buffer; the library owns only its opaque handles.
 *   - there is NO CPU fallback: b2r_config_new fails with B2R_ERR_CUDA when no sm_100 device is usable.
 *   - all witness values are bit-exact to the reference after zero-extension to u64 / usize / bool.
 */
#ifndef B2R_H_
#define B2R_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2R_MAX_DEFS 4 /* regex definitions (RegexDefs) per RegexVerifyConfig handled in one pass */

/* ---- error codes -------------------------------------------------------------------------------------- */
#define B2R_OK 0
#define B2R_ERR_PARSE (-1)              /* defs text is malformed (the reference panics: src/defs.rs:85-100, 219-238) */
#define B2R_ERR_IO (-2)                 /* file could not be opened (reference: File::open().unwrap(), src/defs.rs:55) */
#define B2R_ERR_INVALID_ARG (-3)
#define B2R_ERR_CUDA (-4)               /* CUDA runtime failure / no usable device */
#define B2R_ERR_INVALID_TRANSITION (-5) /* reference: panic!("The transition from {} by {} is invalid!") src/lib.rs:817 */
#define B2R_ERR_TOO_LONG (-6)           /* a string has len > max_chars_size-1 (final-state row would be lost, src/lib.rs:404-418),
                                           or its offsets leave [0, total_bytes] */
#define B2R_ERR_UNSUPPORTED (-7)        /* definition outside what the packed tables can hold (see b2r_config_new) */
#define B2R_ERR_ALIGNMENT (-8)          /* an output pointer / pitch violates the documented alignment */

const char* b2r_last_error(void);
const char* b2r_version(void);

/* ---- AllstrRegexDef (reference src/defs.rs:26-36) -------------------------------------------------------- */
typedef struct b2r_allstr b2r_allstr;

/* read_from_reader (src/defs.rs:75-110): line0 first state, line1 accepted state, line2 largest state,
 * lines>=3 "cur next char"; `char as u8` truncates; a duplicate (char,cur) key overwrites (later line wins);
 * extra tokens are ignored; an empty/short line or a non-u64 token is an error (the reference panics).
 * On B2R_ERR_PARSE *err_line (optional) receives the 0-based line index. */
int b2r_allstr_parse(const char* text, size_t len, b2r_allstr** out, uint64_t* err_line);
/* read_from_text (src/defs.rs:54-58) */
int b2r_allstr_read_from_text(const char* path, b2r_allstr** out, uint64_t* err_line);
void b2r_allstr_free(b2r_allstr*);
uint64_t b2r_allstr_first_state_val(const b2r_allstr*);
uint64_t b2r_allstr_accepted_state_val(const b2r_allstr*);
uint64_t b2r_allstr_largest_state_val(const b2r_allstr*);
uint64_t b2r_allstr_num_transitions(const b2r_allstr*); /* state_lookup.len() */
/* state_lookup.get(&(ch,state)): returns 1 and fills (*line_idx,*next) when present, else 0 */
int b2r_allstr_lookup(const b2r_allstr*, uint8_t ch, uint64_t state, uint64_t* line_idx, uint64_t* next);
/* state_lookup entries in table order (sorted by line index, src/table.rs:103-108): out[i] = {char,cur,next,line_idx} */
int b2r_allstr_entries(const b2r_allstr*, uint64_t* out4, uint64_t capacity_rows);

/* ---- SubstrRegexDef (reference src/defs.rs:115-132) ------------------------------------------------------ */
typedef struct b2r_substr b2r_substr;

/* read_from_reader (src/defs.rs:209-265): line0 max_length, line1 min_position, line2 max_position,
 * line3 start states (may be empty), line4 end states (may be empty), lines>=5 "cur next". */
int b2r_substr_parse(const char* text, size_t len, b2r_substr** out, uint64_t* err_line);
int b2r_substr_read_from_text(const char* path, b2r_substr** out, uint64_t* err_line);
/* SubstrRegexDef::new (src/defs.rs:147-163); pairs = n_pairs x {cur,next} */
int b2r_substr_new(uint64_t max_length, uint64_t min_position, uint64_t max_position, const uint64_t* pairs,
                   uint64_t n_pairs, const uint64_t* start_states, uint64_t n_start, const uint64_t* end_states,
                   uint64_t n_end, b2r_substr** out);
void b2r_substr_free(b2r_substr*);
uint64_t b2r_substr_max_length(const b2r_substr*);
uint64_t b2r_substr_min_position(const b2r_substr*);
uint64_t b2r_substr_max_position(const b2r_substr*);
uint64_t b2r_substr_num_transitions(const b2r_substr*); /* valid_state_transitions.len() (set: duplicates collapse) */
uint64_t b2r_substr_num_start_states(const b2r_substr*);
uint64_t b2r_substr_num_end_states(const b2r_substr*);
int b2r_substr_transitions(const b2r_substr*, uint64_t* out2, uint64_t capacity); /* sorted (cur,next) */
int b2r_substr_start_states(const b2r_substr*, uint64_t* out, uint64_t capacity); /* file order */
int b2r_substr_end_states(const b2r_substr*, uint64_t* out, uint64_t capacity);
int b2r_substr_contains(const b2r_substr*, uint64_t cur, uint64_t next); /* valid_state_transitions.get(..).is_some() */

/* ---- RegexVerifyConfig (reference src/lib.rs:97-131) ------------------------------------------------------
 * Packs D = n_defs RegexDefs{allstr, substrs[]} into the device tables and binds the handle to CUDA `device`.
 * `max_chars_size` is the reference's M: every per-row column has M rows per string.
 * The substr_id offset runs across defs exactly as in RegexVerifyConfig::load / derive_substr_ids
 * (src/lib.rs:780-783, 827-842): offset_0 = 1, offset_{d+1} = offset_d + n_substrs[d].
 * Fails with B2R_ERR_UNSUPPORTED when: D > B2R_MAX_DEFS; the sum over defs of the largest substr id > 255
 * (masked_substr_ids would not fit a byte); largest_state_val+1 > 65535; a state id in the body exceeds
 * largest_state_val (the dummy state would collide with a real one, SURVEY 8(a) out-of-domain iii). */
typedef struct b2r_config b2r_config;
int b2r_config_new(const b2r_allstr* const* allstr, const b2r_substr* const* const* substrs,
                   const uint32_t* n_substrs, uint32_t n_defs, uint64_t max_chars_size, int device,
                   b2r_config** out);
void b2r_config_free(b2r_config*);
uint32_t b2r_config_num_defs(const b2r_config*);
uint64_t b2r_config_max_chars_size(const b2r_config*);
int b2r_config_device(const b2r_config*);
uint32_t b2r_config_state_width(const b2r_config*, uint32_t d);   /* bytes per state, the same for every def: 1 if all dummy<=255 else 2 */
uint64_t b2r_config_dummy_state(const b2r_config*, uint32_t d);   /* largest_state_val+1 */
uint32_t b2r_config_substr_id_offset(const b2r_config*, uint32_t d);
uint32_t b2r_config_num_byte_classes(const b2r_config*, uint32_t d); /* incl. the "no transition" class */
/* smallest pitch >= max_chars_size that keeps every row 32-byte (one DRAM sector) aligned */
uint64_t b2r_config_recommended_row_pitch(const b2r_config*);
uint64_t b2r_config_recommended_bitmap_pitch(const b2r_config*);

/* One process, several GPUs (reference call site src/lib.rs:311-318 is one process; SURVEY 8(b), 8(e)): the same definitions
 * bound to `n_devices` CUDA devices.  b2r_match_batch_host on such a handle shards the strings into contiguous ranges balanced
 * by bytes, runs one host thread + stream set per device, and sums the multiplicity counters with ONE ncclAllReduce (u64 sum)
 * over NVLink before they are copied back; every other column needs no exchange.  NCCL is resolved at run time
 * (dlopen "libnccl.so.2"); B2R_ERR_UNSUPPORTED when it cannot be loaded.  Table queries work as on a single-device handle;
 * the device-pointer entry points need a single-device handle. */
int b2r_config_new_multi(const b2r_allstr* const* allstr, const b2r_substr* const* const* substrs,
                         const uint32_t* n_substrs, uint32_t n_defs, uint64_t max_chars_size, const int* device_ids,
                         uint32_t n_devices, b2r_config** out);
uint32_t b2r_config_num_devices(const b2r_config*);
/* testing / tuning knobs of a handle, the same ones the B2R_* environment variables set when it is created (none is needed in
 * production; results are bit-identical under every setting, except non-zero `debug` and `host_debug`, which skip work to time
 * the rest and so produce wrong results):
 *   table_mode   repl | repl16 | plain | plain16 | global   placement of the walk tables (default: chosen by shared-memory budget)
 *   hist_mode    smem | global                              placement of the multiplicity bins
 *   fuse         1 | 2 | 0 | -1    emit stage inside walk_kernel / own kernel after a walk that zero-fills / own kernel that zero-fills too /
 *                                  default (1 for one def with replicated tables, else 2)
 *   stagger_ns   start offset between the warps of a walk CTA (-1: default)
 *   slices, host_threads, small_path, sparse_cap, sparse_direct, trace_host   host entry points (b2r_match_batch_host)
 *   hist_cache_log2, spread_fill, long_fused, debug, host_debug               kernel tuning / timing experiments
 *   chunked_max_maps   b2r_match_batch_chunked: bytes of chunk transition vectors per pass (0: the default 1 GiB); b2r_string_mult:
 *                      bytes of per-string counters per pass (0: the default 256 MiB); small values force many passes */
int b2r_config_set_option(b2r_config*, const char* name, const char* value);

/* Page-locked host memory for the buffers handed to the host-pointer entry points (a copy into pageable memory cannot overlap
 * with anything): b2r_host_alloc / b2r_host_free own the memory, b2r_host_register / b2r_host_unregister pin memory the caller
 * already owns (e.g. a Rust Vec). */
int b2r_host_alloc(size_t bytes, void** out);
int b2r_host_free(void* p);
int b2r_host_register(void* p, size_t bytes);
int b2r_host_unregister(void* p);

/* RegexTableConfig::load row order (src/table.rs:101-122): row 0 = (0,dummy,dummy,0), then state_lookup sorted by
 * line index, each with the first-match substr id.  out4[r] = {char, cur_state, next_state, substr_id}. */
uint64_t b2r_table_num_rows(const b2r_config*, uint32_t d);
int b2r_table_rows(const b2r_config*, uint32_t d, uint64_t* out4, uint64_t capacity_rows);
/* endpoint table (src/table.rs:126-196): row 0 = (0,dummy,dummy); per substr one (id,start,dummy) per start state
 * then one (id,dummy,end) per end state, file order.  out3[r] = {substr_id, start_state, end_state}. */
uint64_t b2r_endpoint_num_rows(const b2r_config*, uint32_t d);
int b2r_endpoint_rows(const b2r_config*, uint32_t d, uint64_t* out3, uint64_t capacity_rows);

/* ---- per-string status -------------------------------------------------------------------------------- */
#define B2R_ST_ACCEPTED(d) (1u << (d))     /* state[len] == accepted_state_val of def d (src/lib.rs:427-457) */
#define B2R_ST_OVERLAP (1u << 8)           /* two defs flagged the same row (is_start or is_end sum > 1): the reference's
                                              and/not/select arithmetic is non-boolean there (src/lib.rs:613-642);
                                              masked outputs of this string are unspecified, and it has no records:
                                              n_records = n_compact = 0, no truncation flag */
#define B2R_ST_INVALID_TRANSITION (1u << 9) /* reference panics (src/lib.rs:817); err_* describe the first one */
#define B2R_ST_TOO_LONG (1u << 10)         /* len > max_chars_size-1 (or offsets outside the byte buffer): string skipped, its rows are unspecified */
#define B2R_ST_RECORDS_TRUNCATED (1u << 11)
#define B2R_ST_COMPACT_TRUNCATED (1u << 12)

typedef struct b2r_string_status {
    uint32_t flags;
    uint32_t err_pos;   /* position of the first invalid transition of the lowest def index, else 0xFFFFFFFF */
    uint32_t err_state; /* the `state` of the reference's panic text */
    uint8_t err_byte;   /* the `char` of the reference's panic text */
    uint8_t err_def;
    uint16_t reserved0;
    uint32_t n_records; /* number of substring records found (may exceed max_records; only the first are stored) */
    uint32_t n_compact; /* number of masked bytes (may exceed compact_pitch; only the first are stored) */
    uint32_t reserved1[2];
} b2r_string_status; /* 32 bytes */

/* one maximal run of rows with mask = start_mask & end_mask = 1 and a constant substr-id sum */
typedef struct b2r_substr_record {
    uint32_t start;      /* first row of the run */
    uint32_t len;        /* rows in the run */
    uint32_t substr_id;  /* masked_substr_ids value over the run */
    uint32_t compact_off;/* offset of the run's bytes in this string's compact byte area */
} b2r_substr_record;

typedef struct b2r_batch_status {
    int32_t code;          /* B2R_OK, B2R_ERR_INVALID_TRANSITION or B2R_ERR_TOO_LONG (lowest string index wins) */
    uint32_t reserved;
    uint64_t string_idx;   /* the offending string */
    uint32_t pos, state;
    uint8_t byte, def;
    uint16_t reserved2;
    uint32_t n_overlap_lo; /* number of strings flagged B2R_ST_OVERLAP (low 32 bits) */
} b2r_batch_status;

/* ---- outputs of the hot call ------------------------------------------------------------------------------
 * All pointers are DEVICE pointers for b2r_match_batch and HOST pointers for b2r_match_batch_host.  A NULL
 * column is not produced.  Row-major per string: element (j, i) of a byte column lives at j*row_pitch + i.
 * Rows i in [0, M) are defined exactly as the reference assigns them (SURVEY 8(a) row 6):
 *   states[d]       u8 (state_width 1) or u16 (2): s_i for i < len, the final state at i == len, dummy for i > len
 *   substr_ids[d]   u8: per-def substr id, 0 for i >= len                                   (src/lib.rs:825-845)
 *   start_enable[d] bitmap, bit i (LSB first) = enable[i] * is_start_d[i]                   (src/lib.rs:482-493)
 *   end_enable[d]   bitmap, bit i = enable[i] * is_end_d[i+1]                               (src/lib.rs:501-513)
 *   masked_chars    u8: (start_mask & end_mask)[i] * char[i]                                (src/lib.rs:740-764)
 *   masked_substr_ids u8: mask[i] * sum_d substr_ids[d][i]
 * Bytes in [M, row_pitch) / bits >= M of a row are unspecified (the library may write padding there).
 * Alignment: every column pointer 16-byte aligned, row_pitch % 16 == 0, bitmap_pitch % 4 == 0.
 *   mult[d]          T_d u64 counters: lookup-input multiplicity of table row r of b2r_table_rows (src/lib.rs:207-233)
 *   endpoint_mult[d] 2*E_d u64: [0,E_d) multiplicities of the start-endpoint lookup (src/lib.rs:235-258),
 *                    [E_d,2E_d) those of the end-endpoint lookup (src/lib.rs:260-284), rows of b2r_endpoint_rows
 * Invariants: sum_r mult[d][r] = N*M; each half of endpoint_mult[d] sums to N*M. */
#define B2R_OUT_ACCUMULATE_MULT 1u /* add into mult/endpoint_mult instead of overwriting them */
#define B2R_OUT_SPARSE_D2H 2u      /* host-pointer entry points only: substr_ids, start_enable, end_enable, masked_chars and
                                      masked_substr_ids are zero almost everywhere; with this flag they cross PCIe as their non-zero
                                      32-byte sectors (compacted on the device after the kernels wrote the dense columns) and are
                                      expanded into the caller's dense buffers by host threads inside the call (memset + scatter).
                                      Same results, about a third of the device-to-host bytes.  A column slice that is not sparse
                                      after all is copied densely. */

#define B2R_OUT_SPARSE_REUSE 4u    /* with B2R_OUT_SPARSE_D2H: the caller promises that the zero-dominated columns still hold exactly what
                                      the PREVIOUS call on this handle wrote into these same buffers (same n_strings, pitches and
                                      pointers; nothing non-zero was written into them since).  The library then clears only the
                                      sectors it scattered last time instead of zeroing the whole columns (3.5 GB of host memory
                                      writes per 2^20 x 1 KiB strings otherwise).  Ignored (full zeroing) when the buffers or the batch
                                      geometry differ from the previous call. */

typedef struct b2r_outputs {
    uint64_t row_pitch;    /* >= M */
    uint64_t bitmap_pitch; /* bytes, >= ceil(M/8) */
    void* states[B2R_MAX_DEFS];
    uint8_t* substr_ids[B2R_MAX_DEFS];
    uint8_t* start_enable[B2R_MAX_DEFS];
    uint8_t* end_enable[B2R_MAX_DEFS];
    uint8_t* masked_chars;
    uint8_t* masked_substr_ids;
    b2r_string_status* status;       /* N entries */
    b2r_substr_record* records;      /* N * max_records entries, or NULL */
    uint32_t max_records;
    uint32_t compact_pitch;          /* bytes reserved per string in compact_bytes */
    uint8_t* compact_bytes;          /* N * compact_pitch bytes, or NULL */
    uint64_t* mult[B2R_MAX_DEFS];
    uint64_t* endpoint_mult[B2R_MAX_DEFS];
    uint32_t flags;                  /* B2R_OUT_* */
    uint32_t reserved;
} b2r_outputs;

/* ---- the hot call ------------------------------------------------------------------------------------------
 * Replaces, for a whole batch, reference src/lib.rs:316-318 + the value computation of :339-348, :388-418,
 * :427-519, :593-764.  `bytes` holds the N strings back to back, string j = bytes[offsets[j] .. offsets[j+1]).
 * Device-pointer variant: asynchronous on `cuda_stream` (a cudaStream_t, may be NULL for the default stream).
 * It always returns after enqueueing; per-string problems are reported in out->status and summarised by
 * b2r_batch_result(), which synchronises the stream. */
int b2r_match_batch(b2r_config* cfg, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n_strings,
                    uint64_t total_bytes, const b2r_outputs* d_out, void* cuda_stream);
int b2r_batch_result(b2r_config* cfg, void* cuda_stream, b2r_batch_status* out);

/* Same contract as b2r_match_batch (device pointers, M = the handle's max_chars_size, asynchronous on cuda_stream, per-string
 * problems in out->status, summarised by b2r_batch_result) — every defined output byte, status, record and counter is identical
 * to what b2r_match_batch writes for the same call.  Strings are cut into 1 KiB chunks that are walked in parallel: for batches
 * of few, long strings (b2r_match_batch gives each string one GPU lane; a few thousand strings do not fill the GPU).
 * Workspace: the chunks' S-state transition vectors take ceil(M/1024) * (S+1) * 2 bytes per string and def; the strings are
 * processed in passes of at most 1 GiB of them (at least one string per pass), so the handle keeps about that much device
 * memory after a call with long strings and large DFAs.  No host copy or synchronisation inside the call: once a first call
 * of the same shape has sized the workspace, the call can be captured in a CUDA graph.  b2r_last_launch_count, b2r_last_plan
 * and the timing queries report on it (ms3[0] covers the transition vectors and the walk). */
int b2r_match_batch_chunked(b2r_config* cfg, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n_strings,
                            uint64_t total_bytes, const b2r_outputs* d_out, void* cuda_stream);

/* Host-buffer variant (what a drop-in shim calls): copies bytes/offsets to the device, runs the kernels, copies
 * every requested column back, synchronises, and returns B2R_ERR_INVALID_TRANSITION / B2R_ERR_TOO_LONG when a
 * string failed (details in *result, optional).  Device staging memory is owned by the handle and reused. */
int b2r_match_batch_host(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                         const b2r_outputs* h_out, b2r_batch_status* result);

/* Host-buffer variant of b2r_match_batch_chunked, for batches of few, long strings from host memory.  The contract is that of
 * b2r_match_batch_host — arguments, return codes, *result, flags (B2R_OUT_SPARSE_D2H, B2R_OUT_SPARSE_REUSE, B2R_OUT_ACCUMULATE_MULT),
 * pinned or pageable buffers, NULL columns, multi-device handles — and every defined output byte, status, record and counter is
 * identical to what b2r_match_batch_host writes for the same call; the kernels are those of b2r_match_batch_chunked.  The batch
 * is cut into slices balanced by bytes at multiples of 4 strings (b2r_match_batch_host: by count, at multiples of 32), so that
 * a few hundred long strings also overlap the H2D copies, the kernels and the D2H copies; a multi-device handle splits the
 * strings at multiples of 4 as well.  b2r_last_launch_count counts the kernels of every slice, b2r_last_host_bytes and
 * b2r_last_plan report on the call as after b2r_match_batch_host. */
int b2r_match_batch_chunked_host(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                                 const b2r_outputs* h_out, b2r_batch_status* result);

/* Single-string convenience with the exact shape of match_substrs (src/lib.rs:311-315): one &[u8] in,
 * M-row columns out (host pointers, row_pitch ignored -> M). */
int b2r_match_substrs(b2r_config* cfg, const uint8_t* characters, uint64_t len, const b2r_outputs* h_out,
                      b2r_batch_status* result);

/* Long-string path (BASELINE config "single 64 MiB string"): one string of `len` bytes resident on the device,
 * M = len+1 rows, processed by the chunked parallel-prefix composition of S-state transition vectors.
 * Same outputs and semantics as a 1-string b2r_match_batch with max_chars_size = len+1 (the handle's own
 * max_chars_size is ignored). */
int b2r_match_long(b2r_config* cfg, const uint8_t* d_bytes, uint64_t len, const b2r_outputs* d_out,
                   void* cuda_stream);

/* The same with host pointers (the shape a shim around match_substrs, src/lib.rs:311-315, has for one very long input):
 * the string is copied up, the M = len+1 rows of every requested column are copied back; row_pitch >= M. */
int b2r_match_long_host(b2r_config* cfg, const uint8_t* h_bytes, uint64_t len, const b2r_outputs* h_out,
                        b2r_batch_status* result);

/* ---- per-string lookup multiplicities ---------------------------------------------------------------------------------------------
 * mult / endpoint_mult of b2r_outputs are sums over every string of a call: the multiplicity column of ONE lookup argument over
 * the whole batch.  A prover that makes one proof per string (the reference: one match_substrs per synthesize pass,
 * src/lib.rs:311-318) needs them per string.  b2r_string_mult computes them on the device from the state columns an earlier call
 * wrote; the _mult host entry points run the same post-pass inside the host pipeline.
 *
 * Contract:
 *   - Definition.  For every string without B2R_ST_INVALID_TRANSITION or B2R_ST_TOO_LONG, the counts of string j and def d are
 *     exactly the mult[d] and endpoint_mult[d] that a one-string b2r_match_batch of string j writes, on the same handle with the
 *     same M.  A stored entry is a (row, count) with count > 0, rows ascending (rows of b2r_table_rows).  Row 0 carries M - len,
 *     so sum(count) = M, and each half of endpoint_counts sums to M.
 *   - Flagged strings.  A string flagged invalid or too long gets n_entries = 0 and all-zero endpoint counts; its entry slots are
 *     left untouched (the reference panics on such a string and counts nothing).  So over all strings of a call, sum_j of the
 *     per-string counts equals the batch mult[d] / endpoint_mult[d] of the same call.  The post-pass applies the too-long rule to
 *     its own max_chars_size as well: a string with len > M - 1 for the M passed here (e.g. the handle's M after a b2r_match_long
 *     of a longer string) is treated like a flagged one, whatever its status says.
 *   - The state columns and status must be those the match call wrote for the same bytes and offsets; other contents give
 *     unspecified counts (the call still completes).
 *   - Truncation.  n_entries[j] is the true number of distinct rows; only the first max_entries (the lowest rows) are stored, and
 *     the slots after n_entries are left untouched.  max_entries >= min(M, T_d) never truncates.
 *   - Errors (nothing is enqueued): B2R_ERR_INVALID_ARG for a non-NULL entries[d] with a NULL n_entries[d], max_entries == 0 with
 *     entries set, and (device entry only) a NULL status or a NULL states[d] of a def whose counts are asked for;
 *     B2R_ERR_ALIGNMENT for entries not 8-byte aligned or n_entries / endpoint_counts not 4-byte aligned; B2R_ERR_CUDA on a handle
 *     created with device = -1; B2R_ERR_INVALID_ARG for b2r_string_mult on a multi-device handle (b2r_config_new_multi: the device
 *     entry takes pointers of one device; the host entries split the strings over the devices).
 *   - b2r_last_launch_count counts the post-pass kernels (one per pass of strings, plus one compaction per pass when M - 1 > 4096).
 * Cost: the post-pass reads the bytes and the state columns once and writes 8 bytes per stored entry.  A string longer than 4096
 * bytes is counted in pieces into a device workspace of (T_d + 2 E_d) u32 per string and def, in passes of at most 256 MiB of it
 * (chunked_max_maps, when set, bounds it instead), which the handle keeps. */
typedef struct b2r_row_count {
    uint32_t row;
    uint32_t count;
} b2r_row_count; /* 8 bytes */

typedef struct b2r_string_mult_outputs {
    uint32_t max_entries;                     /* entries reserved per string and def */
    uint32_t reserved;
    b2r_row_count* entries[B2R_MAX_DEFS];     /* N * max_entries, string j at j * max_entries, rows ascending; or NULL */
    uint32_t* n_entries[B2R_MAX_DEFS];        /* N: number of distinct rows of string j (may exceed max_entries); or NULL */
    uint32_t* endpoint_counts[B2R_MAX_DEFS];  /* N * 2*E_d (E_d = b2r_endpoint_num_rows), dense, halves as in endpoint_mult; or NULL */
} b2r_string_mult_outputs;

/* Device post-pass over the columns that an earlier b2r_match_batch / b2r_match_batch_chunked / b2r_match_long call on the same
 * bytes and offsets wrote: reads d_out->states[d], row_pitch and status.  Asynchronous on cuda_stream.
 * max_chars_size 0 = the handle's M (after b2r_match_long: pass len + 1, and offsets {0, len}). */
int b2r_string_mult(b2r_config* cfg, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n_strings, uint64_t total_bytes,
                    uint64_t max_chars_size, const b2r_outputs* d_out, const b2r_string_mult_outputs* d_sm, void* cuda_stream);

/* b2r_match_batch_host / b2r_match_batch_chunked_host plus the per-string counts (host pointers), copied back with each slice.
 * h_out->states and h_out->status may be NULL: the library then uses its own scratch columns.  Every column, status, record and
 * counter is what the call without _mult writes; the entry slots the post-pass does not write keep what the caller had in them. */
int b2r_match_batch_host_mult(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                              const b2r_outputs* h_out, const b2r_string_mult_outputs* h_sm, b2r_batch_status* result);
int b2r_match_batch_chunked_host_mult(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                                      const b2r_outputs* h_out, const b2r_string_mult_outputs* h_sm, b2r_batch_status* result);

/* ---- per-string lookup multiplicities, packed ---------------------------------------------------------------------------------------
 * The same counts in a compressed-row layout: the lists of every string back to back, string j of def d at
 * entries[d][row_start[d][j] .. row_start[d][j+1]).  No per-string cap to choose, and only the entries a string has are written
 * (and, from the host entry points, copied back).
 *
 * Contract:
 *   - Definition.  The list of string j and def d is exactly the list b2r_string_mult writes with max_entries >= min(M, T_d): rows
 *     ascending, row 0 first with M - len.  A string flagged invalid or too long (or too long for the M passed) has an empty list,
 *     row_start[j+1] == row_start[j], and all-zero endpoint counts.  endpoint_counts is that of b2r_string_mult_outputs.
 *   - Offsets.  row_start[d] holds N + 1 u64, always complete: row_start[0] = 0, row_start[N] = the total, even when the total
 *     exceeds capacity.
 *   - Capacity.  The list of string j is stored only when row_start[j+1] <= capacity, so the stored lists are those of a prefix of
 *     the strings, and no list is stored in part.  Every entry slot outside a stored list is left untouched.  entries[d] == NULL or
 *     capacity == 0 writes the offsets only (a caller can size its buffer that way).
 *   - Errors (nothing is enqueued): B2R_ERR_INVALID_ARG for entries[d] without row_start[d], and (device entry only) a NULL status
 *     or NULL states[d] of a def whose counts are asked for, and a multi-device handle; B2R_ERR_ALIGNMENT for entries or row_start
 *     not 8-byte aligned or endpoint_counts not 4-byte aligned; B2R_ERR_CUDA on a handle created with device = -1.
 *   - Device entry.  Asynchronous on cuda_stream, no host synchronisation inside: once a first call of the same shape has sized the
 *     workspace, the call can be captured in a CUDA graph.  The counting kernels of b2r_string_mult write each list whole into a
 *     device workspace of max_d min(M, T_d) slots per string and def, in passes of at most 256 MiB of it (chunked_max_maps, when
 *     set, bounds it instead; at least one string per pass), which the handle keeps; a scan and a pack kernel follow each pass.
 *     b2r_last_launch_count counts the kernels of every pass: those of b2r_string_mult, one scan, and one pack when entries are
 *     stored.
 *   - Host entry points.  Every column, status, record and counter is what the call without _mult_packed writes (flags, pinned or
 *     pageable buffers, NULL states / status, the small path, multi-device handles: as b2r_match_batch_host_mult).  No entry is
 *     copied to the device; only the stored entries, row_start and the endpoint counts come back, and b2r_last_host_bytes reports
 *     exactly those bytes on top of the call's own. */
typedef struct b2r_string_mult_packed_outputs {
    uint64_t capacity;                        /* entries reserved in entries[d] (per def) */
    b2r_row_count* entries[B2R_MAX_DEFS];     /* string j: entries[d][row_start[d][j] .. row_start[d][j+1]), rows ascending; or NULL */
    uint64_t* row_start[B2R_MAX_DEFS];        /* N + 1: exclusive prefix of the per-string list lengths, [N] = total; or NULL */
    uint32_t* endpoint_counts[B2R_MAX_DEFS];  /* N * 2*E_d, dense, as in b2r_string_mult_outputs; or NULL */
} b2r_string_mult_packed_outputs;

int b2r_string_mult_packed(b2r_config* cfg, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n_strings, uint64_t total_bytes,
                           uint64_t max_chars_size, const b2r_outputs* d_out, const b2r_string_mult_packed_outputs* d_pk, void* cuda_stream);
int b2r_match_batch_host_mult_packed(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                                     const b2r_outputs* h_out, const b2r_string_mult_packed_outputs* h_pk, b2r_batch_status* result);
int b2r_match_batch_chunked_host_mult_packed(b2r_config* cfg, const uint8_t* h_bytes, const uint64_t* h_offsets, uint64_t n_strings,
                                             const b2r_outputs* h_out, const b2r_string_mult_packed_outputs* h_pk, b2r_batch_status* result);

/* ---- the step after the path: witness columns as field elements (SURVEY 8(f) rank 1) ------------------------------------------
 * The reference places every value of the path in a cell as Value::known(F::from(x as u64)) (src/lib.rs:342-347, 388-418), with
 * F = halo2curves::bn256::Fr in its own circuits (src/lib.rs:896).  b2r_column_to_fr converts a whole DEVICE column into an array
 * of Fr in that type's in-memory layout: per cell four little-endian u64 limbs in Montgomery form (x * 2^256 mod r, what
 * `Fr::from(u64)` = `Fr([x,0,0,0]) * R2` yields), cell (j, i) at d_fr[(j * rows + i) * 4], i < rows, so that a shim can hand
 * `assign_advice` ready-made field elements (a &[Fr] view of the buffer) instead of converting cell by cell.
 *   kind B2R_COL_U8 / _U16 / _U64: d_col[j * pitch + i] (pitch in elements); B2R_COL_BITMAP: bit i (LSB first) of row j of a bitmap
 *   column (pitch in bytes) -> 0 / 1; B2R_COL_CHARS / B2R_COL_ENABLE: d_col = the batch's input bytes, d_offsets its N+1 offsets:
 *   character_values / enable_values of src/lib.rs:339-348 (the byte, resp. 1, for i < len; 0 after).  d_offsets is ignored otherwise.
 * Asynchronous on cuda_stream. */
#define B2R_COL_U8 1u
#define B2R_COL_U16 2u
#define B2R_COL_U64 3u
#define B2R_COL_BITMAP 4u
#define B2R_COL_CHARS 5u
#define B2R_COL_ENABLE 6u
int b2r_column_to_fr(b2r_config* cfg, const void* d_col, uint32_t kind, const uint64_t* d_offsets, uint64_t n_strings, uint64_t rows,
                     uint64_t pitch, uint64_t* d_fr, void* cuda_stream);

/* kernel launches enqueued by the last b2r_match_* call on this handle (for benchmark accounting).  A sliced
 * b2r_match_batch_host call (and b2r_match_substrs) reports the kernels of its LAST slice only; b2r_match_batch_chunked_host
 * reports those of every slice plus the sparse-D2H kernels; a multi-device handle sums over its devices. */
uint32_t b2r_last_launch_count(const b2r_config*);
/* bytes the last host-pointer call moved over PCIe in each direction */
int b2r_last_host_bytes(const b2r_config*, uint64_t* h2d_bytes, uint64_t* d2h_bytes);
/* name + device time (ms, CUDA events on the launching stream) of the dominant kernel of the last call;
 * valid after b2r_batch_result().  Enabled by b2r_config_set_timing(cfg,1). */
int b2r_config_set_timing(b2r_config*, int enable);
int b2r_last_kernel_ms(b2r_config*, float* walk_ms, float* total_ms);
/* device time (ms) of the three stages of the last call: ms3[0] walk_kernel, ms3[1] emit_kernel, ms3[2] finalize_kernel */
int b2r_last_stage_ms(b2r_config*, float* ms3);
/* where the last call kept the walk tables (0 replicated shared memory, 1 shared memory, 2 global) and the
 * multiplicity bins (1 shared memory, 2 global).  After b2r_match_long / b2r_match_long_host and b2r_match_batch_chunked:
 * the placement of their walk over the chunks. */
int b2r_last_plan(const b2r_config*, uint32_t* table_mode, uint32_t* hist_mode);

#ifdef __cplusplus
}
#endif
#endif /* B2R_H_ */
