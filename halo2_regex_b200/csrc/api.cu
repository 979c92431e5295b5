// extern "C" boundary (include/b2r.h): handles, table queries, the device-pointer batch entry points.  The host-pointer entry
// points live in host.cu.
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "config.hpp"
#include "long.cuh"

using namespace b2r;

namespace {

int upload_tables(b2r_config* c) {
    size_t total = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const PackedDef& pd = c->packed[d];
        total += align_up(256, 256) + align_up(pd.trans.size() * 4, 256) + align_up(pd.row_bin.size() * 4, 256) +
                 2 * align_up(pd.erows.size() * 4, 256) + align_up((size_t)pd.num_classes * padded_states(pd.num_states) * 4, 256) +
                 2 * align_up(pd.rows.size() * 4, 256);
    }
    total += 512;                                                          // the two byte <-> bin column maps
    CUDA_TRY(cudaMalloc(&c->tables, total));
    unsigned char* base = (unsigned char*)c->tables;
    size_t off = 0;
    cudaError_t put_err = cudaSuccess;                                    // first failing upload
    auto put = [&](const void* src, size_t n) -> void* {
        void* dst = base + off;
        if (n) { const cudaError_t e = cudaMemcpy(dst, src, n, cudaMemcpyHostToDevice); if (e != cudaSuccess && put_err == cudaSuccess) put_err = e; }
        off += align_up(n, 256);
        return dst;
    };
    size_t scratch = align_up(sizeof(BatchCounters), 256);
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const PackedDef& pd = c->packed[d];
        c->dev[d].byte_class = (uint8_t*)put(pd.byte_class.data(), 256);
        c->dev[d].trans = (uint32_t*)put(pd.trans.data(), pd.trans.size() * 4);
        {
            std::vector<uint32_t> hot;
            build_walk_table(pd, hot);
            c->dev[d].hot = (uint32_t*)put(hot.data(), hot.size() * 4);
        }
        c->dev[d].row_bin = (uint32_t*)put(pd.row_bin.data(), pd.row_bin.size() * 4);
        c->dev[d].erow_start_bin = (uint32_t*)put(pd.erow_start_bin.data(), pd.erows.size() * 4);
        c->dev[d].erow_end_bin = (uint32_t*)put(pd.erow_end_bin.data(), pd.erows.size() * 4);
        {   // the per-string post-pass maps the few distinct bins of a string to rows by binary search (a dense 256 * S map would
            // take 67 MB at S = 65535)
            std::vector<std::pair<uint32_t, uint32_t>> br;
            for (size_t r = 1; r < pd.rows.size(); r++) br.push_back({pd.row_bin[r], (uint32_t)r});
            std::sort(br.begin(), br.end());
            std::vector<uint32_t> bins, rows;
            for (const auto& x : br) { bins.push_back(x.first); rows.push_back(x.second); }
            c->dev[d].sorted_bins = (uint32_t*)put(bins.data(), bins.size() * 4);
            c->dev[d].sorted_rows = (uint32_t*)put(rows.data(), rows.size() * 4);
        }
        scratch += align_up((size_t)256 * pd.num_states * 8, 256) + 2 * align_up((size_t)std::max<uint32_t>(pd.num_substrs, 1) * pd.num_states * 8, 256);
    }
    {   // compact bins: a column for every byte that some def has a transition for, one more for all the others
        uint8_t of_byte[256], byte_of[256];
        uint32_t nb = 0;
        for (int ch = 0; ch < 256; ch++) {
            bool any = false;
            for (uint32_t d = 0; d < c->n_defs && !any; d++) {
                const PackedDef& pd = c->packed[d];
                const uint32_t k = pd.byte_class[ch];
                for (uint32_t st2 = 0; st2 < pd.num_states && !any; st2++) any = !(pd.trans[(size_t)k * pd.num_states + st2] & ENT_INVALID);
            }
            of_byte[ch] = any ? (uint8_t)nb : 0xFF;
            if (any) byte_of[nb++] = (uint8_t)ch;
        }
        if (nb < 255) {
            for (int ch = 0; ch < 256; ch++) if (of_byte[ch] == 0xFF) of_byte[ch] = (uint8_t)nb;   // the column nobody reads back
            c->bin_cols = nb + 1;
        } else {   // (nearly) every byte is in use: dense bins, column = byte
            for (int ch = 0; ch < 256; ch++) { of_byte[ch] = (uint8_t)ch; byte_of[ch] = (uint8_t)ch; }
            c->bin_cols = 256;
        }
        c->d_bin_of_byte = (uint8_t*)put(of_byte, 256);
        c->d_bin_byte = (uint8_t*)put(byte_of, 256);
    }
    if (put_err != cudaSuccess) { set_error("uploading the packed tables failed: %s", cudaGetErrorString(put_err)); return B2R_ERR_CUDA; }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMalloc(&c->scratch, scratch));
    c->scratch_bytes = scratch;
    unsigned char* sb = (unsigned char*)c->scratch;
    size_t so = align_up(sizeof(BatchCounters), 256);
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const PackedDef& pd = c->packed[d];
        c->dev[d].hist = (unsigned long long*)(sb + so); so += align_up((size_t)256 * pd.num_states * 8, 256);
        const size_t ep = align_up((size_t)std::max<uint32_t>(pd.num_substrs, 1) * pd.num_states * 8, 256);
        c->dev[d].ep_start = (unsigned long long*)(sb + so); so += ep;
        c->dev[d].ep_end = (unsigned long long*)(sb + so); so += ep;
    }
    CUDA_TRY(cudaMalloc((void**)&c->d_batch_status, sizeof(b2r_batch_status)));
    return B2R_OK;
}

int parse_table_mode(const char* tm) {
    return !strcmp(tm, "repl") ? (int)TABLE_REPL : !strcmp(tm, "repl16") ? (int)TABLE_REPL16 : !strcmp(tm, "plain") ? (int)TABLE_PLAIN : !strcmp(tm, "plain16") ? (int)TABLE_PLAIN16 : !strcmp(tm, "global") ? (int)TABLE_GLOBAL : -1;
}
int parse_hist_mode(const char* hm) { return !strcmp(hm, "smem") ? (int)HIST_SMEM : !strcmp(hm, "global") ? (int)HIST_GLOBAL : -1; }

// the environment is consulted once per handle, never on the batch path
void read_env_options(b2r_config* c) {
    auto& o = c->opt;
    if (const char* e = getenv("B2R_TABLE_MODE")) o.force_table_mode = parse_table_mode(e);
    if (const char* e = getenv("B2R_HIST_MODE")) o.force_hist_mode = parse_hist_mode(e);
    if (const char* e = getenv("B2R_DEBUG")) o.debug = (uint32_t)atoi(e);
    if (const char* e = getenv("B2R_SPREAD_FILL")) o.spread_fill = e[0] == '0' ? 0u : 1u;
    if (const char* e = getenv("B2R_FUSE")) o.fuse = atoi(e);
    if (const char* e = getenv("B2R_STAGGER_NS")) o.stagger_ns = atoi(e);
    if (const char* e = getenv("B2R_SLICES")) o.slices = atoi(e);
    o.trace_host = getenv("B2R_TRACE_HOST") != nullptr;
    if (const char* e = getenv("B2R_HIST_CACHE_LOG2")) o.hist_cache_log2 = atoi(e);
    if (const char* e = getenv("B2R_HOST_THREADS")) o.host_threads = atoi(e);
    if (const char* e = getenv("B2R_SMALL_PATH")) o.small_path = atoi(e);
    if (const char* e = getenv("B2R_LONG_FUSED")) o.long_fused = atoi(e);
    if (const char* e = getenv("B2R_SPARSE_DIRECT")) o.sparse_direct = atoi(e);
}

}  // namespace

namespace b2r {

int check_outputs(const b2r_config* c, const b2r_outputs* o, bool check_ptrs, uint64_t M) {
    if (!M) M = c->max_chars;
    if (o->row_pitch < M || o->row_pitch % 16) { set_error("row_pitch %llu must be >= max_chars_size and a multiple of 16", (unsigned long long)o->row_pitch); return B2R_ERR_ALIGNMENT; }
    if (o->bitmap_pitch < (M + 7) / 8 || o->bitmap_pitch % 4) { set_error("bitmap_pitch %llu must be >= ceil(M/8) and a multiple of 4", (unsigned long long)o->bitmap_pitch); return B2R_ERR_ALIGNMENT; }
    if (!check_ptrs) return B2R_OK;
    bool ok = aligned16(o->masked_chars) && aligned16(o->masked_substr_ids);
    for (uint32_t d = 0; d < c->n_defs; d++)
        ok = ok && aligned16(o->states[d]) && aligned16(o->substr_ids[d]) && aligned16(o->start_enable[d]) && aligned16(o->end_enable[d]);
    if (!ok) { set_error("output columns must be 16-byte aligned"); return B2R_ERR_ALIGNMENT; }
    return B2R_OK;
}

void fill_walk_params(const b2r_config* c, WalkParams& p, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                      const b2r_outputs* o, uint64_t max_chars) {
    memset(&p, 0, sizeof p);
    p.bytes = d_bytes; p.offsets = d_offsets; p.n_strings = n; p.total_bytes = total_bytes;
    p.row_pitch = o->row_pitch; p.bitmap_pitch = o->bitmap_pitch;
    p.max_chars = (uint32_t)max_chars; p.n_defs = c->n_defs;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        const PackedDef& pd = c->packed[d];
        DefDev& dd = p.def[d];
        dd.byte_class = c->dev[d].byte_class; dd.trans = c->dev[d].trans; dd.hot = c->dev[d].hot;
        dd.padded_states = padded_states(pd.num_states);
        dd.hot_states[0] = pd.hot_states[0]; dd.hot_states[1] = pd.hot_states[1];
        dd.num_states = pd.num_states; dd.num_classes = pd.num_classes; dd.first_state = pd.first_state;
        dd.accepted_state = pd.accepted_state; dd.sid_offset = pd.substr_id_offset; dd.num_substrs = pd.num_substrs;
        dd.hist = c->dev[d].hist; dd.ep_start = c->dev[d].ep_start; dd.ep_end = c->dev[d].ep_end;
        dd.states = o->states[d]; dd.substr_ids = o->substr_ids[d]; dd.start_enable = o->start_enable[d]; dd.end_enable = o->end_enable[d];
    }
    p.bin_cols = c->bin_cols; p.bin_of_byte = c->d_bin_of_byte; p.bin_byte = c->d_bin_byte;
    p.masked_chars = o->masked_chars; p.masked_substr_ids = o->masked_substr_ids;
    p.status = o->status; p.records = o->records; p.compact_bytes = o->compact_bytes;
    p.max_records = o->records ? o->max_records : 0; p.compact_pitch = o->compact_bytes ? o->compact_pitch : 0;
    p.counters = (BatchCounters*)c->scratch;
    p.n_tiles = (uint32_t)((n + 31) / 32);
    p.debug = c->opt.debug; p.spread_fill = c->opt.spread_fill; {
        const int mode = c->opt.fuse >= 0 && c->opt.fuse <= 2 ? c->opt.fuse : (c->n_defs <= 1 ? 1 : 2);
        p.fuse = mode == 1 ? 1u : 0u; p.fill_in_walk = mode == 2 ? 1u : 0u;
    }
    // offset warp starts (walk.cuh) pay off for one def on batches of many tiles per warp: config 1 1.444 -> 1.408 ms, config 2 reading (i)
    // 54.3 -> 56.8 %, the 1023-state DFA 36.5 -> 37 %; three defs lose (35.0 -> 34.2 %), so they keep starting together
    p.stagger_ns = c->opt.stagger_ns >= 0 ? (uint32_t)c->opt.stagger_ns : (c->n_defs == 1 && p.n_tiles >= 4u * 148u * 16u ? 3u * (uint32_t)max_chars : 0u);
    p.fm_words = (uint32_t)((((max_chars - 1) + 15) / 16 + 31) / 32);
    uint64_t ep = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) ep += 2ull * c->packed[d].num_substrs * c->packed[d].num_states * 4ull;
    ep = (ep + 15) & ~15ull;
    p.ep_smem_bytes = ep <= 8192 ? (uint32_t)ep : 0u;   // many substrs x many states: count with global atomics instead
    uint64_t et = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) et += (uint64_t)c->packed[d].num_classes * c->packed[d].num_states * 4ull + 256ull;
    p.emit_smem_tables = et + p.ep_smem_bytes <= 40 * 1024 ? 1u : 0u;
}

int enqueue_finalize(b2r_config* c, const b2r_outputs* o, uint64_t n, uint64_t max_chars, cudaStream_t st) {
    FinalizeParams f;
    memset(&f, 0, sizeof f);
    f.n_defs = c->n_defs; f.accumulate = (o->flags & B2R_OUT_ACCUMULATE_MULT) ? 1 : 0;
    f.n_rows_total = n * max_chars; f.counters = (const BatchCounters*)c->scratch; f.counters_copy = c->counters_copy;
    bool any = false;
    for (uint32_t d = 0; d < c->n_defs; d++) {
        auto& fd = f.def[d];
        fd.hist = c->dev[d].hist; fd.row_bin = c->dev[d].row_bin; fd.n_rows = (uint32_t)c->packed[d].rows.size();
        fd.ep_start = c->dev[d].ep_start; fd.ep_end = c->dev[d].ep_end;
        fd.erow_start_bin = c->dev[d].erow_start_bin; fd.erow_end_bin = c->dev[d].erow_end_bin; fd.n_erows = (uint32_t)c->packed[d].erows.size();
        fd.mult = (unsigned long long*)o->mult[d]; fd.endpoint_mult = (unsigned long long*)o->endpoint_mult[d];
        any = any || fd.mult || fd.endpoint_mult;
    }
    if (!any && !f.counters_copy) return B2R_OK;
    c->last_launches++;
    return launch_finalize(f, st);
}

// ---- the hot call ------------------------------------------------------------------------------------------------------
int match_batch_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                            const b2r_outputs* o, uint64_t max_chars, cudaStream_t st) {
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    if (!o || (n && (!d_bytes && total_bytes)) || (n && !d_offsets)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    if (!aligned16(d_bytes)) { set_error("bytes must be 16-byte aligned"); return B2R_ERR_ALIGNMENT; }
    int rc = check_outputs(c, o, true);
    if (rc) return rc;
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    c->last_launches = 0;
    CUDA_TRY(cudaMemsetAsync(c->scratch, 0, c->scratch_bytes, st));
    WalkParams& p = c->last;
    fill_walk_params(c, p, d_bytes, d_offsets, n, total_bytes, o, max_chars);
    c->have_last = true;
    bool wide = false;
    for (uint32_t d = 0; d < c->n_defs; d++) wide = wide || c->packed[d].state_width == 2;
    if (n) {
        // walk -> emit hand-over: granule flags, and a scratch state column for every def the caller does not want
        if ((rc = c->ws_fmask.reserve(std::max<size_t>((size_t)p.fm_words * n * 4, 16)))) return rc;
        p.fmask = (uint32_t*)c->ws_fmask.p;
        for (uint32_t d = 0; d < c->n_defs; d++) {
            if (p.def[d].states) continue;
            if ((rc = c->ws_states[d].reserve((size_t)n * o->row_pitch * (wide ? 2 : 1)))) return rc;
            p.def[d].states = c->ws_states[d].p;
        }
        if ((rc = plan_walk(p, wide, c->opt.force_table_mode, c->opt.force_hist_mode, c->opt.hist_cache_log2))) return rc;
        // one def stays fused only with replicated tables (a small DFA): the large-DFA kernel is better off with the emit stage as
        // its own launch as well (1023 states: 5.57 -> 5.34 ms)
        if (c->opt.fuse < 0 && p.fuse && p.table_mode != TABLE_REPL && p.n_tiles > 8) {
            p.fuse = 0; p.fill_in_walk = 1;
            if ((rc = plan_walk(p, wide, c->opt.force_table_mode, c->opt.force_hist_mode, c->opt.hist_cache_log2))) return rc;
        }
    }
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[0], st));
    if (n) {
        if ((rc = launch_walk(p, wide, st, nullptr))) return rc;
        c->last_launches++;
    }
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[1], st));
    if (n && !p.fuse) {
        WalkParams pe = p;
        pe.prefilled = p.fill_in_walk;                                    // the walk has zeroed the sparse columns of every tile
        if ((rc = launch_emit(pe, wide, st, nullptr))) return rc;
        c->last_launches++;
    }
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[2], st));
    rc = enqueue_finalize(c, o, n, max_chars, st);
    if (rc) return rc;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[3], st));
    return B2R_OK;
}

void report_failure(const b2r_batch_status& r) {
    if (r.code == B2R_ERR_INVALID_TRANSITION)
        set_error("The transition from %u by %u is invalid! (string %llu, position %u, def %u)", r.state, (unsigned)r.byte,
                  (unsigned long long)r.string_idx, r.pos, (unsigned)r.def);
    else if (r.code == B2R_ERR_TOO_LONG)
        set_error("string %llu is longer than max_chars_size-1 (or its offsets leave the byte buffer)", (unsigned long long)r.string_idx);
}

}  // namespace b2r

extern "C" {

const char* b2r_last_error(void) { return get_error(); }
const char* b2r_version(void) { return "b2r 0.1 (sm_100a)"; }

// ---- AllstrRegexDef ------------------------------------------------------------------------------------------------
int b2r_allstr_parse(const char* text, size_t len, b2r_allstr** out, uint64_t* err_line) {
    if (!out || (!text && len)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    std::unique_ptr<b2r_allstr> a(new (std::nothrow) b2r_allstr);
    if (!a) { set_error("out of memory"); return B2R_ERR_INVALID_ARG; }
    int rc = parse_allstr(text, len, a->def, err_line);
    if (rc) return rc;
    *out = a.release();
    return B2R_OK;
}
int b2r_allstr_read_from_text(const char* path, b2r_allstr** out, uint64_t* err_line) {
    std::string s;
    int rc = read_file(path, s);
    if (rc) return rc;
    return b2r_allstr_parse(s.data(), s.size(), out, err_line);
}
void b2r_allstr_free(b2r_allstr* a) { delete a; }
uint64_t b2r_allstr_first_state_val(const b2r_allstr* a) { return a->def.first_state_val; }
uint64_t b2r_allstr_accepted_state_val(const b2r_allstr* a) { return a->def.accepted_state_val; }
uint64_t b2r_allstr_largest_state_val(const b2r_allstr* a) { return a->def.largest_state_val; }
uint64_t b2r_allstr_num_transitions(const b2r_allstr* a) { return a->def.state_lookup.size(); }
int b2r_allstr_lookup(const b2r_allstr* a, uint8_t ch, uint64_t state, uint64_t* line_idx, uint64_t* next) {
    auto it = a->def.state_lookup.find({state, ch});
    if (it == a->def.state_lookup.end()) return 0;
    if (line_idx) *line_idx = it->second.first;
    if (next) *next = it->second.second;
    return 1;
}
int b2r_allstr_entries(const b2r_allstr* a, uint64_t* out4, uint64_t capacity_rows) {
    const auto v = a->def.in_table_order();
    if (capacity_rows < v.size()) { set_error("capacity too small"); return B2R_ERR_INVALID_ARG; }
    for (size_t i = 0; i < v.size(); i++) { out4[4 * i] = v[i].ch; out4[4 * i + 1] = v[i].cur; out4[4 * i + 2] = v[i].next; out4[4 * i + 3] = v[i].line_idx; }
    return B2R_OK;
}

// ---- SubstrRegexDef ------------------------------------------------------------------------------------------------
int b2r_substr_parse(const char* text, size_t len, b2r_substr** out, uint64_t* err_line) {
    if (!out || (!text && len)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    std::unique_ptr<b2r_substr> s(new (std::nothrow) b2r_substr);
    if (!s) { set_error("out of memory"); return B2R_ERR_INVALID_ARG; }
    int rc = parse_substr(text, len, s->def, err_line);
    if (rc) return rc;
    *out = s.release();
    return B2R_OK;
}
int b2r_substr_read_from_text(const char* path, b2r_substr** out, uint64_t* err_line) {
    std::string s;
    int rc = read_file(path, s);
    if (rc) return rc;
    return b2r_substr_parse(s.data(), s.size(), out, err_line);
}
int b2r_substr_new(uint64_t max_length, uint64_t min_position, uint64_t max_position, const uint64_t* pairs, uint64_t n_pairs,
                   const uint64_t* start_states, uint64_t n_start, const uint64_t* end_states, uint64_t n_end, b2r_substr** out) {
    if (!out) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    std::unique_ptr<b2r_substr> s(new (std::nothrow) b2r_substr);
    if (!s) { set_error("out of memory"); return B2R_ERR_INVALID_ARG; }
    s->def.max_length = max_length; s->def.min_position = min_position; s->def.max_position = max_position;
    for (uint64_t i = 0; i < n_pairs; i++) s->def.valid_state_transitions.insert({pairs[2 * i], pairs[2 * i + 1]});
    s->def.start_states.assign(start_states, start_states + n_start);
    s->def.end_states.assign(end_states, end_states + n_end);
    *out = s.release();
    return B2R_OK;
}
void b2r_substr_free(b2r_substr* s) { delete s; }
uint64_t b2r_substr_max_length(const b2r_substr* s) { return s->def.max_length; }
uint64_t b2r_substr_min_position(const b2r_substr* s) { return s->def.min_position; }
uint64_t b2r_substr_max_position(const b2r_substr* s) { return s->def.max_position; }
uint64_t b2r_substr_num_transitions(const b2r_substr* s) { return s->def.valid_state_transitions.size(); }
uint64_t b2r_substr_num_start_states(const b2r_substr* s) { return s->def.start_states.size(); }
uint64_t b2r_substr_num_end_states(const b2r_substr* s) { return s->def.end_states.size(); }
int b2r_substr_transitions(const b2r_substr* s, uint64_t* out2, uint64_t capacity) {
    if (capacity < s->def.valid_state_transitions.size()) { set_error("capacity too small"); return B2R_ERR_INVALID_ARG; }
    size_t i = 0;
    for (const auto& pr : s->def.valid_state_transitions) { out2[2 * i] = pr.first; out2[2 * i + 1] = pr.second; i++; }
    return B2R_OK;
}
int b2r_substr_start_states(const b2r_substr* s, uint64_t* out, uint64_t capacity) {
    if (capacity < s->def.start_states.size()) { set_error("capacity too small"); return B2R_ERR_INVALID_ARG; }
    std::copy(s->def.start_states.begin(), s->def.start_states.end(), out);
    return B2R_OK;
}
int b2r_substr_end_states(const b2r_substr* s, uint64_t* out, uint64_t capacity) {
    if (capacity < s->def.end_states.size()) { set_error("capacity too small"); return B2R_ERR_INVALID_ARG; }
    std::copy(s->def.end_states.begin(), s->def.end_states.end(), out);
    return B2R_OK;
}
int b2r_substr_contains(const b2r_substr* s, uint64_t cur, uint64_t next) { return s->def.valid_state_transitions.count({cur, next}) ? 1 : 0; }

// ---- RegexVerifyConfig -----------------------------------------------------------------------------------------------
int b2r_config_new(const b2r_allstr* const* allstr, const b2r_substr* const* const* substrs, const uint32_t* n_substrs, uint32_t n_defs,
                   uint64_t max_chars_size, int device, b2r_config** out) {
    if (!allstr || !n_substrs || !out || n_defs == 0) { set_error("null / empty argument"); return B2R_ERR_INVALID_ARG; }
    if (n_defs > B2R_MAX_DEFS) { set_error("%u regex defs: at most %d are supported", n_defs, B2R_MAX_DEFS); return B2R_ERR_UNSUPPORTED; }
    if (max_chars_size == 0 || max_chars_size > 0xFFFFFFF0ull) { set_error("max_chars_size out of range"); return B2R_ERR_INVALID_ARG; }
    // every error path below releases what was created so far (device tables, streams, events, pinned memory)
    struct Free { void operator()(b2r_config* p) const { b2r_config_free(p); } };
    std::unique_ptr<b2r_config, Free> c(new (std::nothrow) b2r_config);
    if (!c) { set_error("out of memory"); return B2R_ERR_INVALID_ARG; }
    read_env_options(c.get());
    c->n_defs = n_defs; c->max_chars = max_chars_size; c->device = -1;   // bound to the device once it has been validated
    uint32_t offset = 1;  // src/lib.rs:780, 827
    uint64_t max_sum = 0;
    for (uint32_t d = 0; d < n_defs; d++) {
        std::vector<const SubstrDef*> subs;
        for (uint32_t k = 0; k < n_substrs[d]; k++) subs.push_back(&substrs[d][k]->def);
        int rc = pack_def(allstr[d]->def, subs, offset, c->packed[d]);
        if (rc) return rc;
        if (n_substrs[d]) max_sum += offset + n_substrs[d] - 1;
        offset += n_substrs[d];  // src/table.rs:197
    }
    // one storage width for every state column of the config: 2 bytes as soon as one def has a dummy state > 255
    bool any_wide = false;
    for (uint32_t d = 0; d < n_defs; d++) any_wide = any_wide || c->packed[d].state_width == 2;
    if (any_wide) for (uint32_t d = 0; d < n_defs; d++) c->packed[d].state_width = 2;
    if (max_sum > 255) { set_error("sum of the largest substr ids over defs is %llu > 255", (unsigned long long)max_sum); return B2R_ERR_UNSUPPORTED; }
    if (device >= 0) {
        int n_dev = 0;
        if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device >= n_dev) {
            set_error("CUDA device %d is not available (%d devices); this library has no CPU fallback", device, n_dev);
            return B2R_ERR_CUDA;
        }
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return B2R_ERR_CUDA; }
        DeviceGuard g(device);
        if (!g.ok) { set_error("cudaSetDevice(%d) failed", device); return B2R_ERR_CUDA; }
        c->device = device;
        int rc = upload_tables(c.get());
        if (rc) return rc;
        CUDA_TRY(cudaStreamCreateWithFlags(&c->host_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&c->in_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&c->out_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&c->pay_stream, cudaStreamNonBlocking));
        for (auto& e : c->ev_in) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : c->ev_done) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : c->ev_pay) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CUDA_TRY(cudaHostAlloc((void**)&c->h_slices, sizeof(BatchCounters) * b2r_config::MAX_SLICES, cudaHostAllocPortable | cudaHostAllocMapped));
        CUDA_TRY(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        for (auto& e : c->ev) CUDA_TRY(cudaEventCreate(&e));
    }
    *out = c.release();
    return B2R_OK;
}

void b2r_config_free(b2r_config* c) {
    if (!c) return;
    if (c->multi) { multi_free(c->multi); c->multi = nullptr; }
    c->pool.reset();                                                       // joins the host worker threads
    if (c->device >= 0) {
        DeviceGuard g(c->device);
        cudaFree(c->tables); cudaFree(c->scratch); cudaFree(c->d_batch_status);
        c->ws_fmask.release(); c->ws_long.release(); c->ws_smult.release(); c->ws_smpk.release();
        for (auto& b : c->ws_states) b.release();
        c->ws_bytes.release(); c->ws_offsets.release(); c->ws_cols.release(); c->ws_sparse.release(); c->ws_sparse_arena.release();
        c->pin_sparse[0].release(); c->pin_sparse[1].release(); c->pin_small.release(); c->pin_pk.release();
        if (c->host_stream) cudaStreamDestroy(c->host_stream);
        if (c->in_stream) cudaStreamDestroy(c->in_stream);
        if (c->out_stream) cudaStreamDestroy(c->out_stream);
        if (c->pay_stream) cudaStreamDestroy(c->pay_stream);
        for (auto& e : c->ev_in) if (e) cudaEventDestroy(e);
        for (auto& e : c->ev_done) if (e) cudaEventDestroy(e);
        for (auto& e : c->ev_pay) if (e) cudaEventDestroy(e);
        if (c->h_slices) cudaFreeHost(c->h_slices);
        if (c->ev_fork) cudaEventDestroy(c->ev_fork);
        for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    }
    delete c;
}
uint32_t b2r_config_num_defs(const b2r_config* c) { return c->n_defs; }
uint64_t b2r_config_max_chars_size(const b2r_config* c) { return c->max_chars; }
int b2r_config_device(const b2r_config* c) { return c->device; }
uint32_t b2r_config_state_width(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].state_width : 0; }
uint64_t b2r_config_dummy_state(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].num_states : 0; }
uint32_t b2r_config_substr_id_offset(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].substr_id_offset : 0; }
uint32_t b2r_config_num_byte_classes(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].num_classes : 0; }
uint64_t b2r_config_recommended_row_pitch(const b2r_config* c) { return align_up(c->max_chars, 32); }
uint64_t b2r_config_recommended_bitmap_pitch(const b2r_config* c) { return align_up((c->max_chars + 7) / 8, 32); }

uint64_t b2r_table_num_rows(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].rows.size() : 0; }
int b2r_table_rows(const b2r_config* c, uint32_t d, uint64_t* out4, uint64_t capacity_rows) {
    if (d >= c->n_defs || capacity_rows < c->packed[d].rows.size()) { set_error("bad def index / capacity"); return B2R_ERR_INVALID_ARG; }
    const auto& rows = c->packed[d].rows;
    for (size_t i = 0; i < rows.size(); i++) { out4[4 * i] = rows[i].ch; out4[4 * i + 1] = rows[i].cur; out4[4 * i + 2] = rows[i].next; out4[4 * i + 3] = rows[i].sid; }
    return B2R_OK;
}
uint64_t b2r_endpoint_num_rows(const b2r_config* c, uint32_t d) { return d < c->n_defs ? c->packed[d].erows.size() : 0; }
int b2r_endpoint_rows(const b2r_config* c, uint32_t d, uint64_t* out3, uint64_t capacity_rows) {
    if (d >= c->n_defs || capacity_rows < c->packed[d].erows.size()) { set_error("bad def index / capacity"); return B2R_ERR_INVALID_ARG; }
    const auto& rows = c->packed[d].erows;
    for (size_t i = 0; i < rows.size(); i++) { out3[3 * i] = rows[i].sid; out3[3 * i + 1] = rows[i].start; out3[3 * i + 2] = rows[i].end; }
    return B2R_OK;
}

int b2r_match_batch(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                    const b2r_outputs* d_out, void* cuda_stream) {
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    return match_batch_impl(c, d_bytes, d_offsets, n, total_bytes, d_out, c->max_chars, (cudaStream_t)cuda_stream);
}

int b2r_batch_result(b2r_config* c, void* cuda_stream, b2r_batch_status* out) {
    if (!c || c->device < 0 || !c->have_last) { set_error("no batch has been enqueued on this handle"); return B2R_ERR_INVALID_ARG; }
    DeviceGuard g(c->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    CUDA_TRY(cudaStreamSynchronize(st));
    BatchCounters h;
    CUDA_TRY(cudaMemcpy(&h, c->scratch, sizeof h, cudaMemcpyDeviceToHost));
    b2r_batch_status r;
    memset(&r, 0, sizeof r);
    r.n_overlap_lo = (uint32_t)h.n_overlap;
    if (h.any_bad()) {
        int rc = launch_diagnose(c->last, h.first_bad(), c->d_batch_status, st);
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemcpy(&r, c->d_batch_status, sizeof r, cudaMemcpyDeviceToHost));
        report_failure(r);
    }
    if (out) *out = r;
    return r.code;
}

int b2r_match_long(b2r_config* c, const uint8_t* d_bytes, uint64_t len, const b2r_outputs* o, void* cuda_stream) {
    if (!c || !o || (!d_bytes && len)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    if (len + 1 > 0xFFFFFFF0ull) { set_error("string of %llu bytes: at most 2^32 - 17 rows are supported", (unsigned long long)len); return B2R_ERR_UNSUPPORTED; }
    if (!aligned16(d_bytes)) { set_error("bytes must be 16-byte aligned"); return B2R_ERR_ALIGNMENT; }
    const uint64_t M = len + 1;
    int rc = check_outputs(c, o, true, M);
    if (rc) return rc;
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    bool wide = false;
    for (uint32_t d = 0; d < c->n_defs; d++) wide = wide || c->packed[d].state_width == 2;
    c->last_launches = 0;
    CUDA_TRY(cudaMemsetAsync(c->scratch, 0, c->scratch_bytes, st));

    // ---- workspace: chunk offsets (+ the {0, len} pair of the whole string), flag words, summary, tree of transition vectors
    const uint32_t n_chunks = (uint32_t)std::max<uint64_t>(1, (len + LONG_CHUNK - 1) / LONG_CHUNK);
    const uint32_t chunk_fm_words = (LONG_CHUNK / 16 + 31) / 32;
    const size_t nodes = long_level_nodes(n_chunks);
    size_t need = 0;
    auto slot = [&](size_t bytes) { size_t off = need; need += align_up(bytes, 256); return off; };
    const size_t off_offsets = slot((size_t)(n_chunks + 3) * 8), off_fmask = slot((size_t)chunk_fm_words * n_chunks * 4), off_summary = slot((size_t)((n_chunks + 31) / 32) * 4);
    size_t off_maps[B2R_MAX_DEFS], off_entry[B2R_MAX_DEFS], off_states[B2R_MAX_DEFS];
    for (uint32_t d = 0; d < c->n_defs; d++) {
        off_maps[d] = slot(nodes * (c->packed[d].num_states + 1) * 2);
        off_entry[d] = slot(nodes * 2);
        off_states[d] = o->states[d] ? 0 : slot(align_up(M, 16) * (wide ? 2 : 1) + 64);
    }
    uint32_t max_s1 = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) max_s1 = std::max(max_s1, c->packed[d].num_states + 1);
    const size_t off_uniq = slot((size_t)n_chunks * 4 * 2), off_nuniq = slot(n_chunks), off_which = slot((size_t)n_chunks * max_s1);
    const uint32_t n_groups = (n_chunks + LONG_GROUP - 1) / LONG_GROUP, n_supers = (n_groups + LONG_SUPER - 1) / LONG_SUPER;
    // one zeroed block: the arrival counters of the super groups (per def) and the second level of the flag summary
    const size_t n_words2 = (n_chunks + 1023) / 1024;
    const size_t off_scnt = slot(((size_t)n_supers * B2R_MAX_DEFS + n_words2) * 4), off_summary2 = off_scnt + (size_t)n_supers * B2R_MAX_DEFS * 4;
    const size_t off_excl = slot((size_t)n_groups * LONG_FUSED_THREADS * 32), off_agg = slot((size_t)n_groups * 32), off_super = slot((size_t)n_supers * 32);
    if ((rc = c->ws_long.reserve(need))) return rc;
    unsigned char* ws = (unsigned char*)c->ws_long.p;
    uint64_t* d_offsets = (uint64_t*)(ws + off_offsets);
    // (the {0, len} pair of the whole string behind the chunk offsets is written by the kernel that writes those, and the root entry
    // state of the composition tree by long_root_kernel: no host copy on this path, so a caller may capture it in a CUDA graph once a
    // first call of the same length has sized the workspace)

    // ---- 1 + 2: transition vectors of the chunks, composition tree, entry state of every chunk ------------------------------
    LongParams lp;
    memset(&lp, 0, sizeof lp);
    lp.bytes = d_bytes; lp.len = len; lp.n_chunks = n_chunks; lp.n_defs = c->n_defs; lp.offsets = d_offsets;
    lp.uniq = (uint16_t*)(ws + off_uniq); lp.n_uniq = ws + off_nuniq; lp.which = ws + off_which;
    lp.excl = ws + off_excl; lp.agg = ws + off_agg; lp.super = ws + off_super; lp.super_cnt = (uint32_t*)(ws + off_scnt);
    for (uint32_t d = 0; d < c->n_defs; d++) {
        lp.def[d].byte_class = c->dev[d].byte_class; lp.def[d].trans = c->dev[d].trans;
        lp.def[d].num_states = c->packed[d].num_states; lp.def[d].first_state = c->packed[d].first_state;
        lp.def[d].num_classes = c->packed[d].num_classes;
        lp.def[d].maps = (uint16_t*)(ws + off_maps[d]); lp.def[d].entry = (uint16_t*)(ws + off_entry[d]);
    }
    // the sparse columns are zeroed on a side stream while the (latency-bound) prefix stages and the walk run; joined before
    // the emit stage
    {
        cudaStream_t zs = c->in_stream;
        CUDA_TRY(cudaEventRecord(c->ev_fork, st));
        CUDA_TRY(cudaStreamWaitEvent(zs, c->ev_fork, 0));
        auto zero = [&](void* ptr, size_t bytes) { return ptr ? cudaMemsetAsync(ptr, 0, bytes, zs) : cudaSuccess; };
        const size_t col_bytes = align_up(M, 16), bm_bytes = align_up((M + 7) / 8, 4);
        for (uint32_t d = 0; d < c->n_defs; d++) {
            CUDA_TRY(zero(o->substr_ids[d], col_bytes));
            CUDA_TRY(zero(o->start_enable[d], bm_bytes));
            CUDA_TRY(zero(o->end_enable[d], bm_bytes));
        }
        CUDA_TRY(zero(o->masked_chars, col_bytes));
        CUDA_TRY(zero(o->masked_substr_ids, col_bytes));
        CUDA_TRY(cudaEventRecord(c->ev_done[0], zs));
    }
    lp.fused = (c->opt.long_fused && long_fused_ok(lp)) ? 1u : 0u;
    CUDA_TRY(cudaMemsetAsync(ws + off_scnt, 0, ((size_t)n_supers * B2R_MAX_DEFS + n_words2) * 4, st));
    if ((rc = launch_long_prepare(lp, st, &c->last_launches))) return rc;

    // ---- 3: the walk, chunk = string, one contiguous state row ------------------------------------------------------------
    b2r_outputs seg = *o;
    seg.row_pitch = LONG_CHUNK;
    WalkParams pw;
    fill_walk_params(c, pw, d_bytes, d_offsets, n_chunks, len, &seg, LONG_CHUNK + 1);
    pw.fuse = 0; pw.fill_in_walk = 0; pw.prefilled = 0; pw.segment_mode = 1; pw.stagger_ns = 0;
    pw.summary = (uint32_t*)(ws + off_summary); pw.summary2 = (uint32_t*)(ws + off_summary2);   // written by the walk itself (two flag words per chunk)
    pw.fmask = (uint32_t*)(ws + off_fmask);
    for (uint32_t d = 0; d < c->n_defs; d++) {
        if (!pw.def[d].states) pw.def[d].states = ws + off_states[d];
        pw.def[d].init_states = lp.def[d].entry;                          // level 0 of the tree
    }
    if ((rc = plan_walk(pw, wide, c->opt.force_table_mode, c->opt.force_hist_mode, c->opt.hist_cache_log2))) return rc;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[0], st));
    if ((rc = launch_walk(pw, wide, st, nullptr))) return rc;
    c->last_launches++;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[1], st));

    // ---- 4: the ordered emit stage of the one string (sparse columns zeroed by now) --------------------------------------------
    CUDA_TRY(cudaStreamWaitEvent(st, c->ev_done[0], 0));
    WalkParams& pe = c->last;
    fill_walk_params(c, pe, d_bytes, d_offsets + n_chunks + 1, 1, len, o, M);
    pe.fuse = 0; pe.fill_in_walk = 0; pe.prefilled = 1;
    pe.table_mode = pw.table_mode; pe.hist_mode = pw.hist_mode;           // b2r_last_plan reports the walk's placement
    pe.fmask = pw.fmask;
    for (uint32_t d = 0; d < c->n_defs; d++) pe.def[d].states = pw.def[d].states;
    c->have_last = true;
    if ((rc = launch_long_emit(pe, wide, pw.fm_words <= 2 ? nullptr : pw.fmask, (uint32_t*)(ws + off_summary), (uint32_t*)(ws + off_summary2), n_chunks, chunk_fm_words, st, &c->last_launches))) return rc;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[2], st));
    rc = enqueue_finalize(c, o, 1, M, st);
    if (rc) return rc;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[3], st));
    return B2R_OK;
}

}  // extern "C"

namespace b2r {

// Workspace of one match_batch_chunked_impl call over n strings: the pass size, and where the slot transition vectors, the entry
// states and the dedupe lists of a pass live in ws_long.  Every size grows with n.
struct ChunkedLayout {
    uint32_t K = 0, max_s1 = 0;
    uint64_t per_pass = 0;
    size_t off_maps[B2R_MAX_DEFS] = {}, off_entry[B2R_MAX_DEFS] = {}, off_uniq = 0, off_nuniq = 0, off_which = 0, need = 0;
};
static ChunkedLayout chunked_layout(const b2r_config* c, uint64_t n, uint64_t M) {
    ChunkedLayout l;
    // passes of whole strings: at most chunked_max_maps bytes (default 1 GiB) of slot transition vectors at a time, or one
    // string's worth when that is more
    l.K = (uint32_t)((M + LONG_CHUNK - 1) / LONG_CHUNK);
    uint64_t s1_sum = 0;
    for (uint32_t d = 0; d < c->n_defs; d++) { s1_sum += c->packed[d].num_states + 1; l.max_s1 = std::max(l.max_s1, c->packed[d].num_states + 1); }
    const uint64_t per_str = (uint64_t)l.K * s1_sum * 2;
    const uint64_t cap = c->opt.chunked_max_maps > 0 ? (uint64_t)c->opt.chunked_max_maps : (1ull << 30);
    l.per_pass = std::min<uint64_t>(n, std::max<uint64_t>(1, cap / per_str));
    l.per_pass = std::min<uint64_t>(l.per_pass, std::max<uint64_t>(1, (1ull << 31) / l.K));   // slot indices stay within u32
    const uint32_t max_slots = (uint32_t)(l.per_pass * l.K);
    const size_t nodes = long_level_nodes(max_slots);
    auto slot = [&](size_t bytes) { size_t off = l.need; l.need += align_up(bytes, 256); return off; };
    for (uint32_t d = 0; d < c->n_defs; d++) {
        l.off_maps[d] = slot(nodes * (c->packed[d].num_states + 1) * 2);
        l.off_entry[d] = slot(nodes * 2);
    }
    l.off_uniq = slot((size_t)max_slots * 4 * 2); l.off_nuniq = slot(max_slots); l.off_which = slot((size_t)max_slots * l.max_s1);
    return l;
}

int chunked_reserve(b2r_config* c, uint64_t n, const b2r_outputs* o, uint64_t max_chars) {
    if (!n) return B2R_OK;
    bool wide = false;
    for (uint32_t d = 0; d < c->n_defs; d++) wide = wide || c->packed[d].state_width == 2;
    const uint64_t fm_words = (((max_chars - 1) + 15) / 16 + 31) / 32;   // as fill_walk_params
    int rc;
    if ((rc = c->ws_fmask.reserve(std::max<size_t>((size_t)fm_words * n * 4, 16)))) return rc;
    for (uint32_t d = 0; d < c->n_defs; d++)
        if (!o->states[d] && (rc = c->ws_states[d].reserve((size_t)n * o->row_pitch * (wide ? 2 : 1)))) return rc;
    return c->ws_long.reserve(chunked_layout(c, n, max_chars).need);
}

// Chunked batch path: b2r_match_batch's outputs, with every string cut into K = ceil(M / LONG_CHUNK) slots that are walked in
// parallel.  Per pass of whole strings: the slots' transition vectors (general prefix pass of long.cu), the last slot of every
// string reset to the constant map -> first_state, the composition tree over all slots of the pass (entry state of every slot),
// walk_kernel<..., CH = true> over the slots (state rows and flag words straight into the batch layout).  Then emit_kernel and
// finalize_kernel over the N strings, exactly as match_batch_impl runs them when the emit stage is its own kernel.
int match_batch_chunked_impl(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                             const b2r_outputs* o, uint64_t max_chars, cudaStream_t st) {
    if (c->device < 0) { set_error("this handle was created without a device (device = -1): no CPU fallback exists"); return B2R_ERR_CUDA; }
    if (!o || (n && (!d_bytes && total_bytes)) || (n && !d_offsets)) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    if (!aligned16(d_bytes)) { set_error("bytes must be 16-byte aligned"); return B2R_ERR_ALIGNMENT; }
    int rc = check_outputs(c, o, true);
    if (rc) return rc;
    DeviceGuard g(c->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", c->device); return B2R_ERR_CUDA; }
    const uint64_t M = max_chars;
    c->last_launches = 0;
    CUDA_TRY(cudaMemsetAsync(c->scratch, 0, c->scratch_bytes, st));
    WalkParams& pe = c->last;                                             // the emit stage over the N strings (and b2r_batch_result)
    fill_walk_params(c, pe, d_bytes, d_offsets, n, total_bytes, o, M);
    pe.fuse = 0; pe.fill_in_walk = 0; pe.stagger_ns = 0;
    pe.prefilled = c->sparse_zeroed ? 1u : 0u;                            // else emit_kernel zero-fills the sparse columns itself
    c->have_last = true;
    bool wide = false;
    for (uint32_t d = 0; d < c->n_defs; d++) wide = wide || c->packed[d].state_width == 2;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[0], st));
    if (n) {
        if ((rc = chunked_reserve(c, n, o, M))) return rc;
        pe.fmask = (uint32_t*)c->ws_fmask.p;
        for (uint32_t d = 0; d < c->n_defs; d++)
            if (!pe.def[d].states) pe.def[d].states = c->ws_states[d].p;
        const ChunkedLayout l = chunked_layout(c, n, M);
        const uint32_t K = l.K;
        const uint64_t per_pass = l.per_pass;
        unsigned char* ws = (unsigned char*)c->ws_long.p;
        LongParams lp;
        memset(&lp, 0, sizeof lp);
        lp.bytes = d_bytes; lp.n_defs = c->n_defs; lp.fused = 0;
        lp.chunk_k = K; lp.max_chars = (uint32_t)M; lp.total_bytes = total_bytes;
        lp.uniq = (uint16_t*)(ws + l.off_uniq); lp.n_uniq = ws + l.off_nuniq; lp.which = ws + l.off_which;
        for (uint32_t d = 0; d < c->n_defs; d++) {
            lp.def[d].byte_class = c->dev[d].byte_class; lp.def[d].trans = c->dev[d].trans;
            lp.def[d].num_states = c->packed[d].num_states; lp.def[d].first_state = c->packed[d].first_state;
            lp.def[d].num_classes = c->packed[d].num_classes;
            lp.def[d].maps = (uint16_t*)(ws + l.off_maps[d]); lp.def[d].entry = (uint16_t*)(ws + l.off_entry[d]);
        }
        const size_t sb = wide ? 2 : 1;
        for (uint64_t j0 = 0; j0 < n; j0 += per_pass) {
            const uint64_t np = std::min<uint64_t>(per_pass, n - j0);
            const uint32_t n_slots = (uint32_t)(np * K);
            lp.n_chunks = n_slots; lp.str_offsets = d_offsets + j0;
            if ((rc = launch_long_prepare(lp, st, &c->last_launches))) return rc;
            WalkParams pw;
            fill_walk_params(c, pw, d_bytes, d_offsets + j0, n_slots, total_bytes, o, LONG_CHUNK + 1);
            pw.fuse = 0; pw.fill_in_walk = 0; pw.prefilled = 0; pw.stagger_ns = 0;
            pw.chunk_k = K; pw.chunk_fm_words = pe.fm_words; pw.chunk_max_chars = (uint32_t)M; pw.chunk_stride = n;
            pw.fmask = pe.fmask + j0;
            for (uint32_t d = 0; d < c->n_defs; d++) {
                pw.def[d].states = (unsigned char*)pe.def[d].states + j0 * o->row_pitch * sb;
                pw.def[d].init_states = lp.def[d].entry;                  // level 0 of the tree
            }
            if ((rc = plan_walk(pw, wide, c->opt.force_table_mode, c->opt.force_hist_mode, c->opt.hist_cache_log2))) return rc;
            if (j0)   // every walk hands out its tiles from a counter at 0
                CUDA_TRY(cudaMemsetAsync((unsigned char*)c->scratch + offsetof(BatchCounters, tile_counter), 0, sizeof(unsigned long long), st));
            if ((rc = launch_walk(pw, wide, st, nullptr))) return rc;
            c->last_launches++;
            pe.table_mode = pw.table_mode; pe.hist_mode = pw.hist_mode;   // b2r_last_plan reports the walk's placement
        }
    }
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[1], st));
    if (n) {
        if ((rc = launch_emit(pe, wide, st, nullptr))) return rc;
        c->last_launches++;
    }
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[2], st));
    rc = enqueue_finalize(c, o, n, M, st);
    if (rc) return rc;
    if (c->timing) CUDA_TRY(cudaEventRecord(c->ev[3], st));
    return B2R_OK;
}

}  // namespace b2r

extern "C" {

int b2r_match_batch_chunked(b2r_config* c, const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n, uint64_t total_bytes,
                            const b2r_outputs* d_out, void* cuda_stream) {
    if (!c) { set_error("null config"); return B2R_ERR_INVALID_ARG; }
    return match_batch_chunked_impl(c, d_bytes, d_offsets, n, total_bytes, d_out, c->max_chars, (cudaStream_t)cuda_stream);
}

uint32_t b2r_last_launch_count(const b2r_config* c) { return c ? c->last_launches : 0; }

// testing / tuning hooks (the same knobs the B2R_* environment variables set when a handle is created)
int b2r_config_set_option(b2r_config* c, const char* name, const char* value) {
    if (!c || !name || !value) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    auto& o = c->opt;
    const int v = atoi(value);
    if (!strcmp(name, "table_mode")) o.force_table_mode = parse_table_mode(value);
    else if (!strcmp(name, "hist_mode")) o.force_hist_mode = parse_hist_mode(value);
    else if (!strcmp(name, "debug")) o.debug = (uint32_t)v;
    else if (!strcmp(name, "spread_fill")) o.spread_fill = v ? 1u : 0u;
    else if (!strcmp(name, "fuse")) o.fuse = v < 0 || v > 2 ? -1 : v;
    else if (!strcmp(name, "stagger_ns")) o.stagger_ns = v;
    else if (!strcmp(name, "slices")) o.slices = v;
    else if (!strcmp(name, "trace_host")) o.trace_host = v != 0;
    else if (!strcmp(name, "hist_cache_log2")) o.hist_cache_log2 = v;
    else if (!strcmp(name, "host_threads")) { o.host_threads = v; c->pool.reset(); }
    else if (!strcmp(name, "small_path")) o.small_path = v;
    else if (!strcmp(name, "sparse_cap")) o.sparse_cap = v;
    else if (!strcmp(name, "sparse_direct")) o.sparse_direct = v;
    else if (!strcmp(name, "host_debug")) o.host_debug = v;
    else if (!strcmp(name, "long_fused")) o.long_fused = v;
    else if (!strcmp(name, "chunked_max_maps")) o.chunked_max_maps = atoll(value);
    else { set_error("unknown option '%s'", name); return B2R_ERR_INVALID_ARG; }
    if (c->multi) return multi_set_option(c->multi, name, value);
    return B2R_OK;
}

// ---- page-locked host memory for the callers of the host-pointer entry points ---------------------------------------------
int b2r_host_alloc(size_t bytes, void** out) {
    if (!out) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    *out = nullptr;
    CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return B2R_OK;
}
int b2r_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return B2R_OK;
}
int b2r_host_register(void* p, size_t bytes) {
    if (!p || !bytes) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return B2R_OK;
}
int b2r_host_unregister(void* p) {
    if (!p) { set_error("null argument"); return B2R_ERR_INVALID_ARG; }
    CUDA_TRY(cudaHostUnregister(p));
    return B2R_OK;
}
int b2r_config_set_timing(b2r_config* c, int enable) { if (!c) return B2R_ERR_INVALID_ARG; c->timing = enable != 0; return B2R_OK; }
int b2r_last_kernel_ms(b2r_config* c, float* walk_ms, float* total_ms) {
    if (!c || !c->timing || c->device < 0) { set_error("timing is not enabled on this handle"); return B2R_ERR_INVALID_ARG; }
    DeviceGuard g(c->device);
    CUDA_TRY(cudaEventSynchronize(c->ev[3]));
    if (walk_ms) CUDA_TRY(cudaEventElapsedTime(walk_ms, c->ev[0], c->ev[1]));
    if (total_ms) CUDA_TRY(cudaEventElapsedTime(total_ms, c->ev[0], c->ev[3]));
    return B2R_OK;
}
int b2r_last_stage_ms(b2r_config* c, float* ms3) {
    if (!c || !c->timing || c->device < 0 || !ms3) { set_error("timing is not enabled on this handle"); return B2R_ERR_INVALID_ARG; }
    DeviceGuard g(c->device);
    CUDA_TRY(cudaEventSynchronize(c->ev[3]));
    for (int i = 0; i < 3; i++) CUDA_TRY(cudaEventElapsedTime(ms3 + i, c->ev[i], c->ev[i + 1]));
    return B2R_OK;
}
int b2r_last_plan(const b2r_config* c, uint32_t* table_mode, uint32_t* hist_mode) {
    if (!c || !c->have_last) { set_error("no batch has been enqueued on this handle"); return B2R_ERR_INVALID_ARG; }
    if (table_mode) *table_mode = c->last.table_mode;
    if (hist_mode) *hist_mode = c->last.hist_mode;
    return B2R_OK;
}

}  // extern "C"
