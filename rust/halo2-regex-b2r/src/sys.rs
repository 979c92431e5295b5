//! Raw declarations of `include/b2r.h` (keep in step with that header; every entry point there cites the reference interface
//! it replaces).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct b2r_allstr { _p: [u8; 0] }
#[repr(C)] pub struct b2r_substr { _p: [u8; 0] }
#[repr(C)] pub struct b2r_config { _p: [u8; 0] }

pub const B2R_MAX_DEFS: usize = 4;
pub const B2R_OK: c_int = 0;
pub const B2R_ERR_PARSE: c_int = -1;
pub const B2R_ERR_INVALID_TRANSITION: c_int = -5;
pub const B2R_ERR_TOO_LONG: c_int = -6;
pub const B2R_OUT_ACCUMULATE_MULT: u32 = 1;
pub const B2R_OUT_SPARSE_D2H: u32 = 2;
pub const B2R_OUT_SPARSE_REUSE: u32 = 4;
pub const B2R_ST_OVERLAP: u32 = 1 << 8;
pub const B2R_COL_U8: u32 = 1;
pub const B2R_COL_U16: u32 = 2;
pub const B2R_COL_U64: u32 = 3;
pub const B2R_COL_BITMAP: u32 = 4;
pub const B2R_COL_CHARS: u32 = 5;
pub const B2R_COL_ENABLE: u32 = 6;

#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct b2r_string_status {
    pub flags: u32, pub err_pos: u32, pub err_state: u32, pub err_byte: u8, pub err_def: u8, pub reserved0: u16,
    pub n_records: u32, pub n_compact: u32, pub reserved1: [u32; 2],
}
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct b2r_substr_record { pub start: u32, pub len: u32, pub substr_id: u32, pub compact_off: u32 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct b2r_batch_status {
    pub code: i32, pub reserved: u32, pub string_idx: u64, pub pos: u32, pub state: u32,
    pub byte: u8, pub def: u8, pub reserved2: u16, pub n_overlap_lo: u32,
}
#[repr(C)]
pub struct b2r_outputs {
    pub row_pitch: u64, pub bitmap_pitch: u64,
    pub states: [*mut c_void; B2R_MAX_DEFS], pub substr_ids: [*mut u8; B2R_MAX_DEFS],
    pub start_enable: [*mut u8; B2R_MAX_DEFS], pub end_enable: [*mut u8; B2R_MAX_DEFS],
    pub masked_chars: *mut u8, pub masked_substr_ids: *mut u8,
    pub status: *mut b2r_string_status, pub records: *mut b2r_substr_record, pub max_records: u32, pub compact_pitch: u32,
    pub compact_bytes: *mut u8, pub mult: [*mut u64; B2R_MAX_DEFS], pub endpoint_mult: [*mut u64; B2R_MAX_DEFS],
    pub flags: u32, pub reserved: u32,
}
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct b2r_row_count { pub row: u32, pub count: u32 }
#[repr(C)]
pub struct b2r_string_mult_outputs {
    pub max_entries: u32, pub reserved: u32,
    pub entries: [*mut b2r_row_count; B2R_MAX_DEFS], pub n_entries: [*mut u32; B2R_MAX_DEFS],
    pub endpoint_counts: [*mut u32; B2R_MAX_DEFS],
}
#[repr(C)]
pub struct b2r_string_mult_packed_outputs {
    pub capacity: u64,
    pub entries: [*mut b2r_row_count; B2R_MAX_DEFS], pub row_start: [*mut u64; B2R_MAX_DEFS],
    pub endpoint_counts: [*mut u32; B2R_MAX_DEFS],
}

extern "C" {
    pub fn b2r_last_error() -> *const c_char;
    pub fn b2r_allstr_parse(text: *const c_char, len: usize, out: *mut *mut b2r_allstr, err_line: *mut u64) -> c_int;
    pub fn b2r_allstr_free(a: *mut b2r_allstr);
    pub fn b2r_substr_parse(text: *const c_char, len: usize, out: *mut *mut b2r_substr, err_line: *mut u64) -> c_int;
    pub fn b2r_substr_new(max_length: u64, min_position: u64, max_position: u64, pairs: *const u64, n_pairs: u64,
                          starts: *const u64, n_start: u64, ends: *const u64, n_end: u64, out: *mut *mut b2r_substr) -> c_int;
    pub fn b2r_substr_free(s: *mut b2r_substr);
    pub fn b2r_config_new(allstr: *const *const b2r_allstr, substrs: *const *const *const b2r_substr, n_substrs: *const u32,
                          n_defs: u32, max_chars_size: u64, device: c_int, out: *mut *mut b2r_config) -> c_int;
    pub fn b2r_config_new_multi(allstr: *const *const b2r_allstr, substrs: *const *const *const b2r_substr, n_substrs: *const u32,
                                n_defs: u32, max_chars_size: u64, device_ids: *const c_int, n_devices: u32, out: *mut *mut b2r_config) -> c_int;
    pub fn b2r_config_free(c: *mut b2r_config);
    pub fn b2r_config_state_width(c: *const b2r_config, d: u32) -> u32;
    pub fn b2r_config_recommended_row_pitch(c: *const b2r_config) -> u64;
    pub fn b2r_config_recommended_bitmap_pitch(c: *const b2r_config) -> u64;
    pub fn b2r_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn b2r_host_free(p: *mut c_void) -> c_int;
    pub fn b2r_host_register(p: *mut c_void, bytes: usize) -> c_int;
    pub fn b2r_host_unregister(p: *mut c_void) -> c_int;
    pub fn b2r_table_num_rows(c: *const b2r_config, d: u32) -> u64;
    pub fn b2r_table_rows(c: *const b2r_config, d: u32, out4: *mut u64, capacity_rows: u64) -> c_int;
    pub fn b2r_endpoint_num_rows(c: *const b2r_config, d: u32) -> u64;
    pub fn b2r_endpoint_rows(c: *const b2r_config, d: u32, out3: *mut u64, capacity_rows: u64) -> c_int;
    pub fn b2r_match_substrs(c: *mut b2r_config, characters: *const u8, len: u64, out: *const b2r_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_match_batch_host(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_match_batch_chunked_host(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                        result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_match_batch(c: *mut b2r_config, d_bytes: *const u8, d_offsets: *const u64, n: u64, total_bytes: u64,
                           d_out: *const b2r_outputs, cuda_stream: *mut c_void) -> c_int;
    pub fn b2r_match_batch_chunked(c: *mut b2r_config, d_bytes: *const u8, d_offsets: *const u64, n: u64, total_bytes: u64,
                                   d_out: *const b2r_outputs, cuda_stream: *mut c_void) -> c_int;
    pub fn b2r_match_long(c: *mut b2r_config, d_bytes: *const u8, len: u64, d_out: *const b2r_outputs, cuda_stream: *mut c_void) -> c_int;
    pub fn b2r_match_long_host(c: *mut b2r_config, h_bytes: *const u8, len: u64, h_out: *const b2r_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_string_mult(c: *mut b2r_config, d_bytes: *const u8, d_offsets: *const u64, n: u64, total_bytes: u64, max_chars_size: u64,
                           d_out: *const b2r_outputs, d_sm: *const b2r_string_mult_outputs, cuda_stream: *mut c_void) -> c_int;
    pub fn b2r_match_batch_host_mult(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                     sm: *const b2r_string_mult_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_match_batch_chunked_host_mult(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                             sm: *const b2r_string_mult_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_string_mult_packed(c: *mut b2r_config, d_bytes: *const u8, d_offsets: *const u64, n: u64, total_bytes: u64, max_chars_size: u64,
                                  d_out: *const b2r_outputs, d_pk: *const b2r_string_mult_packed_outputs, cuda_stream: *mut c_void) -> c_int;
    pub fn b2r_match_batch_host_mult_packed(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                            pk: *const b2r_string_mult_packed_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_match_batch_chunked_host_mult_packed(c: *mut b2r_config, bytes: *const u8, offsets: *const u64, n: u64, out: *const b2r_outputs,
                                                    pk: *const b2r_string_mult_packed_outputs, result: *mut b2r_batch_status) -> c_int;
    pub fn b2r_batch_result(c: *mut b2r_config, cuda_stream: *mut c_void, out: *mut b2r_batch_status) -> c_int;
    pub fn b2r_column_to_fr(c: *mut b2r_config, d_col: *const c_void, kind: u32, d_offsets: *const u64, n_strings: u64, rows: u64,
                            pitch: u64, d_fr: *mut u64, cuda_stream: *mut c_void) -> c_int;
}
