// b2r.hpp — C++ host mirror of the reference's public API for the witness-generation path, header-only, on top of the
// C ABI of b2r.h.  (The reference is a Rust crate; no Rust toolchain exists in this image, so the compiled-language host
// side is C++.  INTEGRATION.md shows the Rust binding.)
//
// Names, argument meaning and error behaviour follow zkemail/halo2-regex:
//   halo2_regex::AllstrRegexDef / SubstrRegexDef / RegexDefs     reference src/defs.rs:26-36, 115-132, 17-22
//   halo2_regex::RegexVerifyConfig::{configure, match_substrs}   reference src/lib.rs:97-131, 311-315
//   derive_states / derive_substr_ids / derive_is_start_end      reference src/lib.rs:804-888
//   AssignedRegexResult                                          reference src/lib.rs:79-93 (integer values, not cells)
// Where the reference panics, these throw (std::runtime_error with the reference's panic text for an invalid transition).
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "b2r.h"

namespace halo2_regex {

struct RegexError : std::runtime_error {
    int code;
    RegexError(int code_, const std::string& msg) : std::runtime_error(msg), code(code_) {}
};
// reference: panic!("The transition from {} by {} is invalid!", state, char)   src/lib.rs:817
struct InvalidTransition : RegexError {
    uint32_t pos, state;
    uint8_t byte, def;
    InvalidTransition(const b2r_batch_status& s)
        : RegexError(B2R_ERR_INVALID_TRANSITION, "The transition from " + std::to_string(s.state) + " by " + std::to_string((unsigned)s.byte) + " is invalid!"),
          pos(s.pos), state(s.state), byte(s.byte), def(s.def) {}
};

namespace detail {
inline void check(int rc) {
    if (rc != B2R_OK) throw RegexError(rc, b2r_last_error());
}
}  // namespace detail

// Regex that the whole input string must satisfy (reference src/defs.rs:26-36).
class AllstrRegexDef {
public:
    uint64_t first_state_val = 0, accepted_state_val = 0, largest_state_val = 0;

    static AllstrRegexDef read_from_text(const std::string& file_path) {   // src/defs.rs:54-58
        b2r_allstr* h = nullptr;
        uint64_t line = 0;
        detail::check(b2r_allstr_read_from_text(file_path.c_str(), &h, &line));
        return AllstrRegexDef(h);
    }
    static AllstrRegexDef read_from_reader(const std::string& text) {      // src/defs.rs:75-110
        b2r_allstr* h = nullptr;
        uint64_t line = 0;
        detail::check(b2r_allstr_parse(text.data(), text.size(), &h, &line));
        return AllstrRegexDef(h);
    }
    // state_lookup.get(&(char, state)) -> Some((line_idx, next_state))
    bool state_lookup(uint8_t ch, uint64_t state, uint64_t* line_idx, uint64_t* next) const { return b2r_allstr_lookup(h_.get(), ch, state, line_idx, next) != 0; }
    uint64_t num_transitions() const { return b2r_allstr_num_transitions(h_.get()); }
    const b2r_allstr* handle() const { return h_.get(); }

private:
    explicit AllstrRegexDef(b2r_allstr* h) : h_(h, b2r_allstr_free) {
        first_state_val = b2r_allstr_first_state_val(h);
        accepted_state_val = b2r_allstr_accepted_state_val(h);
        largest_state_val = b2r_allstr_largest_state_val(h);
    }
    std::shared_ptr<b2r_allstr> h_;
};

// Regex of a substring to extract (reference src/defs.rs:115-132).
class SubstrRegexDef {
public:
    uint64_t max_length = 0, min_position = 0, max_position = 0;

    // SubstrRegexDef::new (src/defs.rs:147-163)
    SubstrRegexDef(uint64_t max_length_, uint64_t min_position_, uint64_t max_position_, const std::set<std::pair<uint64_t, uint64_t>>& valid_state_transitions,
                   const std::vector<uint64_t>& start_states, const std::vector<uint64_t>& end_states) {
        std::vector<uint64_t> pairs;
        for (const auto& pr : valid_state_transitions) { pairs.push_back(pr.first); pairs.push_back(pr.second); }
        b2r_substr* h = nullptr;
        detail::check(b2r_substr_new(max_length_, min_position_, max_position_, pairs.data(), pairs.size() / 2, start_states.data(), start_states.size(),
                                     end_states.data(), end_states.size(), &h));
        adopt(h);
    }
    static SubstrRegexDef read_from_text(const std::string& file_path) {   // src/defs.rs:184-188
        b2r_substr* h = nullptr;
        uint64_t line = 0;
        detail::check(b2r_substr_read_from_text(file_path.c_str(), &h, &line));
        return SubstrRegexDef(h);
    }
    static SubstrRegexDef read_from_reader(const std::string& text) {      // src/defs.rs:209-265
        b2r_substr* h = nullptr;
        uint64_t line = 0;
        detail::check(b2r_substr_parse(text.data(), text.size(), &h, &line));
        return SubstrRegexDef(h);
    }
    bool valid_state_transitions_contains(uint64_t cur, uint64_t next) const { return b2r_substr_contains(h_.get(), cur, next) != 0; }
    std::vector<uint64_t> start_states() const { std::vector<uint64_t> v(b2r_substr_num_start_states(h_.get())); detail::check(b2r_substr_start_states(h_.get(), v.data(), v.size())); return v; }
    std::vector<uint64_t> end_states() const { std::vector<uint64_t> v(b2r_substr_num_end_states(h_.get())); detail::check(b2r_substr_end_states(h_.get(), v.data(), v.size())); return v; }
    const b2r_substr* handle() const { return h_.get(); }

private:
    explicit SubstrRegexDef(b2r_substr* h) { adopt(h); }
    void adopt(b2r_substr* h) {
        h_ = std::shared_ptr<b2r_substr>(h, b2r_substr_free);
        max_length = b2r_substr_max_length(h); min_position = b2r_substr_min_position(h); max_position = b2r_substr_max_position(h);
    }
    std::shared_ptr<b2r_substr> h_;
};

// reference src/defs.rs:17-22
struct RegexDefs {
    AllstrRegexDef allstr;
    std::vector<SubstrRegexDef> substrs;
};

// The values behind the reference's AssignedRegexResult (src/lib.rs:79-93), M = max_chars_size entries each.
struct AssignedRegexResult {
    std::vector<uint8_t> all_enable_flags;    // 1 for i < len
    std::vector<uint8_t> all_characters;      // padded with 0
    std::vector<uint8_t> all_substr_ids;      // masked: (start_mask & end_mask) * sum of substr ids
    std::vector<uint8_t> masked_characters;   // masked characters
    // the other witness columns of the chip, per regex def
    std::vector<std::vector<uint16_t>> states;
    std::vector<std::vector<uint8_t>> substr_ids, start_enable, end_enable;   // enables: one 0/1 entry per row
    std::vector<bool> accepted;               // state[len] == accepted_state_val (the circuit asserts it, src/lib.rs:427-457)
};

class RegexVerifyConfig {
public:
    size_t max_chars_size = 0;
    std::vector<RegexDefs> regex_defs;

    // RegexVerifyConfig::configure (src/lib.rs:126-131): max_chars_size and regex_defs; `meta` / `gate` are halo2-side
    static RegexVerifyConfig configure(size_t max_chars_size, const std::vector<RegexDefs>& regex_defs, int device = 0) {
        RegexVerifyConfig c;
        c.max_chars_size = max_chars_size;
        c.regex_defs = regex_defs;
        std::vector<const b2r_allstr*> allstr;
        std::vector<std::vector<const b2r_substr*>> subs(regex_defs.size());
        std::vector<const b2r_substr* const*> sub_ptrs;
        std::vector<uint32_t> n_subs;
        for (size_t d = 0; d < regex_defs.size(); d++) {
            allstr.push_back(regex_defs[d].allstr.handle());
            for (const auto& s : regex_defs[d].substrs) subs[d].push_back(s.handle());
            sub_ptrs.push_back(subs[d].data());
            n_subs.push_back((uint32_t)subs[d].size());
        }
        b2r_config* h = nullptr;
        detail::check(b2r_config_new(allstr.data(), sub_ptrs.data(), n_subs.data(), (uint32_t)regex_defs.size(), max_chars_size, device, &h));
        c.h_ = std::shared_ptr<b2r_config>(h, b2r_config_free);
        return c;
    }
    // The same chip bound to several GPUs of one process (b2r_config_new_multi): match_batch shards the strings over them.
    static RegexVerifyConfig configure_multi(size_t max_chars_size, const std::vector<RegexDefs>& regex_defs, const std::vector<int>& devices) {
        RegexVerifyConfig c;
        c.max_chars_size = max_chars_size;
        c.regex_defs = regex_defs;
        std::vector<const b2r_allstr*> allstr;
        std::vector<std::vector<const b2r_substr*>> subs(regex_defs.size());
        std::vector<const b2r_substr* const*> sub_ptrs;
        std::vector<uint32_t> n_subs;
        for (size_t d = 0; d < regex_defs.size(); d++) {
            allstr.push_back(regex_defs[d].allstr.handle());
            for (const auto& s : regex_defs[d].substrs) subs[d].push_back(s.handle());
            sub_ptrs.push_back(subs[d].data());
            n_subs.push_back((uint32_t)subs[d].size());
        }
        b2r_config* h = nullptr;
        detail::check(b2r_config_new_multi(allstr.data(), sub_ptrs.data(), n_subs.data(), (uint32_t)regex_defs.size(), max_chars_size, devices.data(),
                                           (uint32_t)devices.size(), &h));
        c.h_ = std::shared_ptr<b2r_config>(h, b2r_config_free);
        return c;
    }

    // Every witness column of a batch of strings (the bulk form of match_substrs): row-major, `row_pitch` / `bitmap_pitch` bytes
    // per string, plus the lookup multiplicities per table row (b2r.h).
    struct BatchWitness {
        size_t n = 0, row_pitch = 0, bitmap_pitch = 0;
        std::vector<std::vector<uint8_t>> states, substr_ids, start_enable, end_enable;   // per def (states: state_width bytes per row)
        std::vector<uint8_t> masked_chars, masked_substr_ids;
        std::vector<b2r_string_status> status;
        std::vector<std::vector<uint64_t>> mult, endpoint_mult;
    };
    // chunked: b2r_match_batch_chunked_host, the same outputs with every string cut into 1 KiB chunks walked in parallel (batches of
    // few, long strings, such as e-mail bodies)
    BatchWitness match_batch(const std::vector<std::vector<uint8_t>>& strings, bool sparse_d2h = false, bool chunked = false) const {
        const size_t M = max_chars_size, D = regex_defs.size(), n = strings.size();
        BatchWitness w;
        w.n = n; w.row_pitch = (M + 31) & ~size_t(31); w.bitmap_pitch = ((M + 7) / 8 + 31) & ~size_t(31);
        std::vector<uint8_t> bytes;
        std::vector<uint64_t> offsets(n + 1, 0);
        for (size_t j = 0; j < n; j++) { bytes.insert(bytes.end(), strings[j].begin(), strings[j].end()); offsets[j + 1] = bytes.size(); }
        b2r_outputs out{};
        out.row_pitch = w.row_pitch; out.bitmap_pitch = w.bitmap_pitch; out.flags = sparse_d2h ? B2R_OUT_SPARSE_D2H : 0;
        w.states.resize(D); w.substr_ids.resize(D); w.start_enable.resize(D); w.end_enable.resize(D); w.mult.resize(D); w.endpoint_mult.resize(D);
        for (size_t d = 0; d < D; d++) {
            w.states[d].resize(n * w.row_pitch * b2r_config_state_width(h_.get(), (uint32_t)d)); w.substr_ids[d].resize(n * w.row_pitch);
            w.start_enable[d].resize(n * w.bitmap_pitch); w.end_enable[d].resize(n * w.bitmap_pitch);
            w.mult[d].resize(b2r_table_num_rows(h_.get(), (uint32_t)d)); w.endpoint_mult[d].resize(2 * b2r_endpoint_num_rows(h_.get(), (uint32_t)d));
            out.states[d] = w.states[d].data(); out.substr_ids[d] = w.substr_ids[d].data();
            out.start_enable[d] = w.start_enable[d].data(); out.end_enable[d] = w.end_enable[d].data();
            out.mult[d] = w.mult[d].data(); out.endpoint_mult[d] = w.endpoint_mult[d].data();
        }
        w.masked_chars.resize(n * w.row_pitch); w.masked_substr_ids.resize(n * w.row_pitch); w.status.resize(n);
        out.masked_chars = w.masked_chars.data(); out.masked_substr_ids = w.masked_substr_ids.data(); out.status = w.status.data();
        b2r_batch_status res{};
        const int rc = (chunked ? b2r_match_batch_chunked_host : b2r_match_batch_host)(h_.get(), bytes.data(), offsets.data(), n, &out, &res);
        if (rc == B2R_ERR_INVALID_TRANSITION) throw InvalidTransition(res);
        detail::check(rc);
        return w;
    }

    // The lookup multiplicities of every string of a batch, one list per string and def (b2r_match_batch_host_mult_packed): string
    // j's (row, count) pairs of def d are entries[d][row_start[d][j] .. row_start[d][j+1]), rows ascending, row 0 first;
    // endpoint_counts[d] holds 2*E_d counts per string.  chunked: b2r_match_batch_chunked_host_mult_packed.
    struct StringMult {
        std::vector<std::vector<b2r_row_count>> entries;
        std::vector<std::vector<uint64_t>> row_start;
        std::vector<std::vector<uint32_t>> endpoint_counts;
    };
    StringMult string_mult(const std::vector<std::vector<uint8_t>>& strings, bool chunked = false) const {
        const size_t M = max_chars_size, D = regex_defs.size(), n = strings.size();
        std::vector<uint8_t> bytes;
        std::vector<uint64_t> offsets(n + 1, 0);
        for (size_t j = 0; j < n; j++) { bytes.insert(bytes.end(), strings[j].begin(), strings[j].end()); offsets[j + 1] = bytes.size(); }
        b2r_outputs out{};
        out.row_pitch = (M + 31) & ~size_t(31); out.bitmap_pitch = ((M + 7) / 8 + 31) & ~size_t(31);
        size_t pitch = 1;                                                 // no list is longer than min(M, T_d)
        for (size_t d = 0; d < D; d++) pitch = std::max<size_t>(pitch, std::min<size_t>(M, b2r_table_num_rows(h_.get(), (uint32_t)d)));
        StringMult s;
        s.entries.resize(D); s.row_start.resize(D); s.endpoint_counts.resize(D);
        b2r_string_mult_packed_outputs pk{};
        pk.capacity = n * pitch;
        for (size_t d = 0; d < D; d++) {
            s.entries[d].resize(n * pitch); s.row_start[d].resize(n + 1); s.endpoint_counts[d].resize(n * 2 * b2r_endpoint_num_rows(h_.get(), (uint32_t)d));
            pk.entries[d] = s.entries[d].data(); pk.row_start[d] = s.row_start[d].data(); pk.endpoint_counts[d] = s.endpoint_counts[d].data();
        }
        b2r_batch_status res{};
        const int rc = (chunked ? b2r_match_batch_chunked_host_mult_packed : b2r_match_batch_host_mult_packed)(h_.get(), bytes.data(), offsets.data(), n,
                                                                                                             &out, &pk, &res);
        if (rc == B2R_ERR_INVALID_TRANSITION) throw InvalidTransition(res);
        detail::check(rc);
        for (size_t d = 0; d < D; d++) s.entries[d].resize(s.row_start[d][n]);
        return s;
    }

    // match_substrs (src/lib.rs:311-315): one &[u8] in, the assigned values out
    AssignedRegexResult match_substrs(const std::vector<uint8_t>& characters) const {
        const size_t M = max_chars_size, D = regex_defs.size(), bm = (M + 7) / 8;
        const size_t bp = (bm + 15) & ~size_t(15), rp = (M + 15) & ~size_t(15);
        AssignedRegexResult r;
        std::vector<std::vector<uint8_t>> st8(D), sid(D, std::vector<uint8_t>(rp)), se(D, std::vector<uint8_t>(bp)), ee(D, std::vector<uint8_t>(bp));
        std::vector<std::vector<uint16_t>> st16(D);
        std::vector<uint8_t> mc(rp), ms(rp);
        b2r_string_status status{};
        b2r_outputs out{};
        out.row_pitch = rp; out.bitmap_pitch = bp;
        for (size_t d = 0; d < D; d++) {
            if (b2r_config_state_width(h_.get(), (uint32_t)d) == 1) { st8[d].resize(rp); out.states[d] = st8[d].data(); }
            else { st16[d].resize(rp); out.states[d] = st16[d].data(); }
            out.substr_ids[d] = sid[d].data(); out.start_enable[d] = se[d].data(); out.end_enable[d] = ee[d].data();
        }
        out.masked_chars = mc.data(); out.masked_substr_ids = ms.data(); out.status = &status;
        b2r_batch_status res{};
        const int rc = b2r_match_substrs(h_.get(), characters.data(), characters.size(), &out, &res);
        if (rc == B2R_ERR_INVALID_TRANSITION) throw InvalidTransition(res);
        detail::check(rc);
        r.all_enable_flags.assign(M, 0); r.all_characters.assign(M, 0);
        for (size_t i = 0; i < characters.size(); i++) { r.all_enable_flags[i] = 1; r.all_characters[i] = characters[i]; }
        r.all_substr_ids.assign(ms.begin(), ms.begin() + M);
        r.masked_characters.assign(mc.begin(), mc.begin() + M);
        r.states.resize(D); r.substr_ids.resize(D); r.start_enable.resize(D); r.end_enable.resize(D);
        for (size_t d = 0; d < D; d++) {
            r.states[d].resize(M);
            for (size_t i = 0; i < M; i++) r.states[d][i] = st8[d].empty() ? st16[d][i] : st8[d][i];
            r.substr_ids[d].assign(sid[d].begin(), sid[d].begin() + M);
            r.start_enable[d].resize(M); r.end_enable[d].resize(M);
            for (size_t i = 0; i < M; i++) { r.start_enable[d][i] = (se[d][i >> 3] >> (i & 7)) & 1; r.end_enable[d][i] = (ee[d][i >> 3] >> (i & 7)) & 1; }
            r.accepted.push_back((status.flags & B2R_ST_ACCEPTED(d)) != 0);
        }
        return r;
    }

    // derive_states (src/lib.rs:804-823): per def, len + 1 states
    std::vector<std::vector<uint64_t>> derive_states(const std::vector<uint8_t>& characters) const {
        const AssignedRegexResult r = match_substrs(characters);
        std::vector<std::vector<uint64_t>> v(regex_defs.size());
        for (size_t d = 0; d < v.size(); d++) v[d].assign(r.states[d].begin(), r.states[d].begin() + characters.size() + 1);
        return v;
    }
    // derive_substr_ids (src/lib.rs:825-845): per def, len ids
    std::vector<std::vector<size_t>> derive_substr_ids(const std::vector<uint8_t>& characters) const {
        const AssignedRegexResult r = match_substrs(characters);
        std::vector<std::vector<size_t>> v(regex_defs.size());
        for (size_t d = 0; d < v.size(); d++) v[d].assign(r.substr_ids[d].begin(), r.substr_ids[d].begin() + characters.size());
        return v;
    }
    // derive_is_start_end (src/lib.rs:847-888): (is_starts, is_ends), per def len + 1 flags; is_starts ends with false, is_ends starts with false
    std::pair<std::vector<std::vector<bool>>, std::vector<std::vector<bool>>> derive_is_start_end(const std::vector<uint8_t>& characters) const {
        const AssignedRegexResult r = match_substrs(characters);
        const size_t L = characters.size(), D = regex_defs.size();
        std::vector<std::vector<bool>> is_starts(D), is_ends(D);
        for (size_t d = 0; d < D; d++) {
            for (size_t i = 0; i < L; i++) is_starts[d].push_back(r.start_enable[d][i] != 0);
            is_starts[d].push_back(false);
            is_ends[d].push_back(false);
            for (size_t i = 0; i < L; i++) is_ends[d].push_back(r.end_enable[d][i] != 0);
        }
        return {is_starts, is_ends};
    }
    // RegexTableConfig::load row order (src/table.rs:101-122): {char, cur_state, next_state, substr_id} per row of def d
    std::vector<std::array<uint64_t, 4>> table_rows(uint32_t d) const {
        std::vector<std::array<uint64_t, 4>> rows(b2r_table_num_rows(h_.get(), d));
        detail::check(b2r_table_rows(h_.get(), d, rows.empty() ? nullptr : rows[0].data(), rows.size()));
        return rows;
    }
    b2r_config* handle() const { return h_.get(); }

private:
    std::shared_ptr<b2r_config> h_;
};

}  // namespace halo2_regex
