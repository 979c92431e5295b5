"""Loads halo2_regex_b200/libb2r.so (the C ABI of include/b2r.h) and declares its signatures.

There is no CPU fallback: importing this module fails loudly when the CUDA extension has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C halo2_regex_b200/csrc`).
"""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2R_LIB") or os.path.join(_HERE, "libb2r.so")   # B2R_LIB: an instrumented build of the same library (development aid)

# every symbol include/b2r.h declares (tests check the export list against the header)
SYMBOLS = """
b2r_last_error b2r_version
b2r_allstr_parse b2r_allstr_read_from_text b2r_allstr_free b2r_allstr_first_state_val b2r_allstr_accepted_state_val
b2r_allstr_largest_state_val b2r_allstr_num_transitions b2r_allstr_lookup b2r_allstr_entries
b2r_substr_parse b2r_substr_read_from_text b2r_substr_new b2r_substr_free b2r_substr_max_length b2r_substr_min_position
b2r_substr_max_position b2r_substr_num_transitions b2r_substr_num_start_states b2r_substr_num_end_states
b2r_substr_transitions b2r_substr_start_states b2r_substr_end_states b2r_substr_contains
b2r_config_new b2r_config_free b2r_config_num_defs b2r_config_max_chars_size b2r_config_device b2r_config_state_width
b2r_config_dummy_state b2r_config_substr_id_offset b2r_config_num_byte_classes b2r_config_recommended_row_pitch
b2r_config_recommended_bitmap_pitch b2r_table_num_rows b2r_table_rows b2r_endpoint_num_rows b2r_endpoint_rows
b2r_match_batch b2r_match_batch_chunked b2r_batch_result b2r_match_batch_host b2r_match_batch_chunked_host b2r_match_substrs b2r_match_long b2r_match_long_host b2r_last_launch_count
b2r_config_set_timing b2r_last_kernel_ms b2r_last_stage_ms b2r_last_plan
b2r_config_new_multi b2r_config_num_devices b2r_config_set_option b2r_host_alloc b2r_host_free b2r_host_register b2r_host_unregister
b2r_last_host_bytes b2r_column_to_fr
b2r_string_mult b2r_match_batch_host_mult b2r_match_batch_chunked_host_mult
b2r_string_mult_packed b2r_match_batch_host_mult_packed b2r_match_batch_chunked_host_mult_packed
""".split()


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a CUDA extension has not been built and there is no CPU fallback. "
            "Run `make -C halo2_regex_b200/csrc -j8` (or __graft_entry__.build()).")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32, sz = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_size_t
    pvp, pu64 = C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)

    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype, f.argtypes = res, list(args)

    sig("b2r_last_error", C.c_char_p)
    sig("b2r_version", C.c_char_p)
    sig("b2r_allstr_parse", i32, C.c_char_p, sz, pvp, pu64)
    sig("b2r_allstr_read_from_text", i32, C.c_char_p, pvp, pu64)
    sig("b2r_allstr_free", None, vp)
    for n in ("first_state_val", "accepted_state_val", "largest_state_val", "num_transitions"):
        sig("b2r_allstr_" + n, u64, vp)
    sig("b2r_allstr_lookup", i32, vp, C.c_uint8, u64, pu64, pu64)
    sig("b2r_allstr_entries", i32, vp, vp, u64)
    sig("b2r_substr_parse", i32, C.c_char_p, sz, pvp, pu64)
    sig("b2r_substr_read_from_text", i32, C.c_char_p, pvp, pu64)
    sig("b2r_substr_new", i32, u64, u64, u64, vp, u64, vp, u64, vp, u64, pvp)
    sig("b2r_substr_free", None, vp)
    for n in ("max_length", "min_position", "max_position", "num_transitions", "num_start_states", "num_end_states"):
        sig("b2r_substr_" + n, u64, vp)
    for n in ("transitions", "start_states", "end_states"):
        sig("b2r_substr_" + n, i32, vp, vp, u64)
    sig("b2r_substr_contains", i32, vp, u64, u64)
    sig("b2r_config_new", i32, pvp, C.POINTER(pvp), C.POINTER(u32), u32, u64, i32, pvp)
    sig("b2r_config_free", None, vp)
    sig("b2r_config_num_defs", u32, vp)
    sig("b2r_config_max_chars_size", u64, vp)
    sig("b2r_config_device", i32, vp)
    sig("b2r_config_state_width", u32, vp, u32)
    sig("b2r_config_dummy_state", u64, vp, u32)
    sig("b2r_config_substr_id_offset", u32, vp, u32)
    sig("b2r_config_num_byte_classes", u32, vp, u32)
    sig("b2r_config_recommended_row_pitch", u64, vp)
    sig("b2r_config_recommended_bitmap_pitch", u64, vp)
    sig("b2r_table_num_rows", u64, vp, u32)
    sig("b2r_table_rows", i32, vp, u32, vp, u64)
    sig("b2r_endpoint_num_rows", u64, vp, u32)
    sig("b2r_endpoint_rows", i32, vp, u32, vp, u64)
    sig("b2r_match_batch", i32, vp, vp, vp, u64, u64, C.POINTER(_abi.Outputs), vp)
    sig("b2r_match_batch_chunked", i32, vp, vp, vp, u64, u64, C.POINTER(_abi.Outputs), vp)
    sig("b2r_batch_result", i32, vp, vp, C.POINTER(_abi.BatchStatus))
    sig("b2r_match_batch_host", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.BatchStatus))
    sig("b2r_match_batch_chunked_host", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.BatchStatus))
    sig("b2r_match_substrs", i32, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.BatchStatus))
    sig("b2r_match_long", i32, vp, vp, u64, C.POINTER(_abi.Outputs), vp)
    sig("b2r_match_long_host", i32, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.BatchStatus))
    sig("b2r_last_launch_count", u32, vp)
    sig("b2r_config_set_timing", i32, vp, i32)
    sig("b2r_last_kernel_ms", i32, vp, C.POINTER(C.c_float), C.POINTER(C.c_float))
    sig("b2r_last_stage_ms", i32, vp, C.POINTER(C.c_float))
    sig("b2r_last_plan", i32, vp, C.POINTER(u32), C.POINTER(u32))
    sig("b2r_config_new_multi", i32, pvp, C.POINTER(pvp), C.POINTER(u32), u32, u64, C.POINTER(i32), u32, pvp)
    sig("b2r_config_num_devices", u32, vp)
    sig("b2r_config_set_option", i32, vp, C.c_char_p, C.c_char_p)
    sig("b2r_host_alloc", i32, sz, pvp)
    sig("b2r_host_free", i32, vp)
    sig("b2r_host_register", i32, vp, sz)
    sig("b2r_host_unregister", i32, vp)
    sig("b2r_last_host_bytes", i32, vp, pu64, pu64)
    sig("b2r_column_to_fr", i32, vp, vp, u32, vp, u64, u64, u64, vp, vp)
    sig("b2r_string_mult", i32, vp, vp, vp, u64, u64, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultStruct), vp)
    sig("b2r_match_batch_host_mult", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultStruct), C.POINTER(_abi.BatchStatus))
    sig("b2r_match_batch_chunked_host_mult", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultStruct),
        C.POINTER(_abi.BatchStatus))
    sig("b2r_string_mult_packed", i32, vp, vp, vp, u64, u64, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultPackedStruct), vp)
    sig("b2r_match_batch_host_mult_packed", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultPackedStruct),
        C.POINTER(_abi.BatchStatus))
    sig("b2r_match_batch_chunked_host_mult_packed", i32, vp, vp, vp, u64, C.POINTER(_abi.Outputs), C.POINTER(_abi.StringMultPackedStruct),
        C.POINTER(_abi.BatchStatus))
    return L


lib = _load()


def last_error():
    return lib.b2r_last_error().decode("utf-8", "replace")
