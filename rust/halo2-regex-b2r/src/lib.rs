//! Safe wrapper over `libb2r.so` with the shapes the reference's `RegexVerifyConfig` needs.
//!
//! What changes in zkemail/halo2-regex (`src/lib.rs` of the reference):
//!  * `RegexVerifyConfig` gains a private `b2r: Arc<Config>` built in `configure` from the unchanged `regex_defs`
//!    (`Config::from_texts` with the same lookup-text the crate already reads; `regex_defs` stays `pub`);
//!  * `match_substrs` (`:311-315`, signature unchanged) replaces `derive_states / derive_substr_ids / derive_is_start_end`
//!    (`:316-318`) and the value computations of `:339-348, 388-418, 427-519, 593-764` by ONE call, `Config::match_substrs`,
//!    and feeds `assign_advice` from the returned `Witness` (see `Witness::state_values` etc.); cell assignment, the FlexGate
//!    cells that re-derive the masks in-circuit and the constraint system stay as they are;
//!  * a prover with many strings calls `Config::match_batch` once instead of `match_substrs` per string.
//! An invalid transition re-raises the reference's panic text (`:817`).
pub mod sys;

use std::ffi::CStr;
use std::os::raw::c_void;
use std::ptr;
use sys::*;

fn last_error() -> String {
    unsafe { CStr::from_ptr(b2r_last_error()) }.to_string_lossy().into_owned()
}

/// Page-locked host memory from the library (`b2r_host_alloc`): the copies of the host-pointer entry points only overlap with
/// the kernels when source and destination are pinned.  Zero-initialised by the driver.
pub struct PinnedBuf { ptr: *mut u8, len: usize }
unsafe impl Send for PinnedBuf {}
impl PinnedBuf {
    pub fn new(len: usize) -> Self {
        let mut p: *mut c_void = ptr::null_mut();
        let rc = unsafe { b2r_host_alloc(len.max(1), &mut p) };
        assert_eq!(rc, B2R_OK, "b2r_host_alloc: {}", last_error());
        PinnedBuf { ptr: p as *mut u8, len }
    }
    pub fn as_slice(&self) -> &[u8] { unsafe { std::slice::from_raw_parts(self.ptr, self.len) } }
    pub fn as_mut_slice(&mut self) -> &mut [u8] { unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) } }
    pub fn as_mut_ptr(&mut self) -> *mut u8 { self.ptr }
}
impl Drop for PinnedBuf { fn drop(&mut self) { unsafe { b2r_host_free(self.ptr as *mut c_void); } } }

/// `AllstrRegexDef` + its `SubstrRegexDef`s as lookup text (the files `read_from_text` reads, reference src/defs.rs:54, 184).
pub struct DefTexts<'a> { pub allstr: &'a str, pub substrs: Vec<&'a str> }

/// One `RegexVerifyConfig` worth of packed tables on one or several GPUs.
pub struct Config { ptr: *mut b2r_config, n_defs: usize, max_chars_size: usize, state_width: usize }
unsafe impl Send for Config {}

/// The witness columns of ONE string, `max_chars_size` rows each, exactly the values the reference assigns.
pub struct Witness {
    pub len: usize,
    pub states: Vec<Vec<u64>>,            // per def: s_i, the final state at row len, dummy after (src/lib.rs:388-418)
    pub substr_ids: Vec<Vec<u64>>,        // per def, unmasked (src/lib.rs:825-845)
    pub start_enable: Vec<Vec<bool>>,     // enable[i] * is_start_d[i]       (src/lib.rs:482-493)
    pub end_enable: Vec<Vec<bool>>,       // enable[i] * is_end_d[i+1]       (src/lib.rs:501-513)
    pub masked_characters: Vec<u64>,      // AssignedRegexResult.masked_characters (src/lib.rs:740-764)
    pub all_substr_ids: Vec<u64>,         // AssignedRegexResult.all_substr_ids
    pub accepted: Vec<bool>,              // per def: state[len] == accepted_state_val (src/lib.rs:427-457)
    pub overlap: bool,                    // two defs flagged the same row: outside the reference's boolean domain
}

impl Config {
    /// `RegexVerifyConfig::configure` for the witness side: `devices` = CUDA device ids (one: `b2r_config_new`, several: the
    /// single-process multi-GPU handle `b2r_config_new_multi`).
    pub fn from_texts(max_chars_size: usize, defs: &[DefTexts], devices: &[i32]) -> Result<Self, String> {
        assert!(!defs.is_empty() && defs.len() <= B2R_MAX_DEFS && !devices.is_empty());
        let mut allstr: Vec<*const b2r_allstr> = Vec::new();
        let mut subs: Vec<Vec<*const b2r_substr>> = Vec::new();
        let mut cleanup = |allstr: &Vec<*const b2r_allstr>, subs: &Vec<Vec<*const b2r_substr>>| unsafe {
            for a in allstr { b2r_allstr_free(*a as *mut _); }
            for v in subs { for s in v { b2r_substr_free(*s as *mut _); } }
        };
        for d in defs {
            let (mut a, mut line) = (ptr::null_mut(), 0u64);
            if unsafe { b2r_allstr_parse(d.allstr.as_ptr() as *const _, d.allstr.len(), &mut a, &mut line) } != B2R_OK {
                cleanup(&allstr, &subs);
                return Err(format!("allstr text, line {line}: {}", last_error()));
            }
            allstr.push(a);
            let mut v = Vec::new();
            for s in &d.substrs {
                let mut p = ptr::null_mut();
                if unsafe { b2r_substr_parse(s.as_ptr() as *const _, s.len(), &mut p, &mut line) } != B2R_OK {
                    subs.push(v);
                    cleanup(&allstr, &subs);
                    return Err(format!("substr text, line {line}: {}", last_error()));
                }
                v.push(p as *const b2r_substr);
            }
            subs.push(v);
        }
        let sub_ptrs: Vec<*const *const b2r_substr> = subs.iter().map(|v| v.as_ptr()).collect();
        let n_subs: Vec<u32> = subs.iter().map(|v| v.len() as u32).collect();
        let mut c = ptr::null_mut();
        let rc = unsafe {
            if devices.len() == 1 {
                b2r_config_new(allstr.as_ptr(), sub_ptrs.as_ptr(), n_subs.as_ptr(), defs.len() as u32, max_chars_size as u64, devices[0], &mut c)
            } else {
                b2r_config_new_multi(allstr.as_ptr(), sub_ptrs.as_ptr(), n_subs.as_ptr(), defs.len() as u32, max_chars_size as u64,
                                     devices.as_ptr(), devices.len() as u32, &mut c)
            }
        };
        cleanup(&allstr, &subs);                       // the handle keeps its own packed copy
        if rc != B2R_OK { return Err(last_error()); }
        let state_width = unsafe { b2r_config_state_width(c, 0) } as usize;
        Ok(Config { ptr: c, n_defs: defs.len(), max_chars_size, state_width })
    }

    /// Replaces reference src/lib.rs:316-318 + the value computations behind them for one string.
    /// Panics with the reference's text on an invalid transition (src/lib.rs:817).
    pub fn match_substrs(&self, characters: &[u8]) -> Witness {
        let (m, d, w) = (self.max_chars_size, self.n_defs, self.state_width);
        let rp = (m + 15) & !15;
        let bp = ((m + 7) / 8 + 15) & !15;
        let mut states = vec![vec![0u8; rp * w]; d];
        let mut sids = vec![vec![0u8; rp]; d];
        let mut se = vec![vec![0u8; bp]; d];
        let mut ee = vec![vec![0u8; bp]; d];
        let (mut mc, mut ms) = (vec![0u8; rp], vec![0u8; rp]);
        let mut status = b2r_string_status::default();
        let mut out: b2r_outputs = unsafe { std::mem::zeroed() };
        out.row_pitch = rp as u64;
        out.bitmap_pitch = bp as u64;
        for i in 0..d {
            out.states[i] = states[i].as_mut_ptr() as *mut c_void;
            out.substr_ids[i] = sids[i].as_mut_ptr();
            out.start_enable[i] = se[i].as_mut_ptr();
            out.end_enable[i] = ee[i].as_mut_ptr();
        }
        out.masked_chars = mc.as_mut_ptr();
        out.masked_substr_ids = ms.as_mut_ptr();
        out.status = &mut status;
        let mut res = b2r_batch_status::default();
        let rc = unsafe { b2r_match_substrs(self.ptr, characters.as_ptr(), characters.len() as u64, &out, &mut res) };
        if rc == B2R_ERR_INVALID_TRANSITION {
            panic!("The transition from {} by {} is invalid!", res.state, res.byte);   // reference src/lib.rs:817
        }
        assert_eq!(rc, B2R_OK, "{}", last_error());
        let bit = |v: &Vec<u8>, i: usize| (v[i >> 3] >> (i & 7)) & 1 == 1;
        let st = |v: &Vec<u8>, i: usize| if w == 1 { v[i] as u64 } else { u16::from_le_bytes([v[2 * i], v[2 * i + 1]]) as u64 };
        Witness {
            len: characters.len(),
            states: states.iter().map(|v| (0..m).map(|i| st(v, i)).collect()).collect(),
            substr_ids: sids.iter().map(|v| v[..m].iter().map(|&x| x as u64).collect()).collect(),
            start_enable: se.iter().map(|v| (0..m).map(|i| bit(v, i)).collect()).collect(),
            end_enable: ee.iter().map(|v| (0..m).map(|i| bit(v, i)).collect()).collect(),
            masked_characters: mc[..m].iter().map(|&x| x as u64).collect(),
            all_substr_ids: ms[..m].iter().map(|&x| x as u64).collect(),
            accepted: (0..d).map(|i| status.flags & (1 << i) != 0).collect(),
            overlap: status.flags & B2R_ST_OVERLAP != 0,
        }
    }

    /// Whole batches: `bytes` = the strings back to back, `offsets` = N+1 offsets; `out` as described in include/b2r.h (host
    /// pointers; use `PinnedBuf`s and `B2R_OUT_SPARSE_D2H | B2R_OUT_SPARSE_REUSE` when the same buffers are filled batch after batch).
    pub fn match_batch(&self, bytes: &[u8], offsets: &[u64], out: &b2r_outputs) -> Result<b2r_batch_status, (i32, b2r_batch_status)> {
        let mut res = b2r_batch_status::default();
        let rc = unsafe { b2r_match_batch_host(self.ptr, bytes.as_ptr(), offsets.as_ptr(), offsets.len() as u64 - 1, out, &mut res) };
        if rc == B2R_OK { Ok(res) } else { Err((rc, res)) }
    }

    /// `match_batch` for batches of few, long strings (e-mail bodies): the same arguments, result and outputs, with every string
    /// cut into 1 KiB chunks that are walked in parallel on the device (`b2r_match_batch_chunked_host`).
    pub fn match_batch_chunked(&self, bytes: &[u8], offsets: &[u64], out: &b2r_outputs) -> Result<b2r_batch_status, (i32, b2r_batch_status)> {
        let mut res = b2r_batch_status::default();
        let rc = unsafe { b2r_match_batch_chunked_host(self.ptr, bytes.as_ptr(), offsets.as_ptr(), offsets.len() as u64 - 1, out, &mut res) };
        if rc == B2R_OK { Ok(res) } else { Err((rc, res)) }
    }

    /// `RegexTableConfig::load` row order (reference src/table.rs:101-122): rows of {char, cur_state, next_state, substr_id};
    /// multiplicity counter r of `b2r_outputs.mult[d]` belongs to row r.
    pub fn table_rows(&self, d: usize) -> Vec<[u64; 4]> {
        let n = unsafe { b2r_table_num_rows(self.ptr, d as u32) } as usize;
        let mut v = vec![[0u64; 4]; n];
        assert_eq!(unsafe { b2r_table_rows(self.ptr, d as u32, v.as_mut_ptr() as *mut u64, n as u64) }, B2R_OK);
        v
    }

    pub fn raw(&self) -> *mut b2r_config { self.ptr }
}
impl Drop for Config { fn drop(&mut self) { unsafe { b2r_config_free(self.ptr) } } }

/// `b2r_column_to_fr` writes Fr cells in the in-memory layout of `halo2curves::bn256::Fr` (four little-endian u64 limbs in
/// Montgomery form): a host copy of such a buffer IS a `[Fr]`.
#[cfg(feature = "fr")]
pub fn limbs_as_fr(limbs: &[u64]) -> &[halo2curves::bn256::Fr] {
    assert_eq!(limbs.len() % 4, 0);
    assert_eq!(std::mem::size_of::<halo2curves::bn256::Fr>(), 32);
    unsafe { std::slice::from_raw_parts(limbs.as_ptr() as *const halo2curves::bn256::Fr, limbs.len() / 4) }
}
