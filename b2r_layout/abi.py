"""ctypes mirror of include/b2r.h (struct layouts and constants only; loads nothing)."""
import ctypes as C

B2R_MAX_DEFS = 4

B2R_OK = 0
B2R_ERR_PARSE = -1
B2R_ERR_IO = -2
B2R_ERR_INVALID_ARG = -3
B2R_ERR_CUDA = -4
B2R_ERR_INVALID_TRANSITION = -5
B2R_ERR_TOO_LONG = -6
B2R_ERR_UNSUPPORTED = -7
B2R_ERR_ALIGNMENT = -8

B2R_ST_OVERLAP = 1 << 8
B2R_ST_INVALID_TRANSITION = 1 << 9
B2R_ST_TOO_LONG = 1 << 10
B2R_ST_RECORDS_TRUNCATED = 1 << 11
B2R_ST_COMPACT_TRUNCATED = 1 << 12

B2R_OUT_ACCUMULATE_MULT = 1
B2R_OUT_SPARSE_D2H = 2
B2R_OUT_SPARSE_REUSE = 4

B2R_COL_U8, B2R_COL_U16, B2R_COL_U64, B2R_COL_BITMAP, B2R_COL_CHARS, B2R_COL_ENABLE = 1, 2, 3, 4, 5, 6


def B2R_ST_ACCEPTED(d):
    return 1 << d


class StringStatus(C.Structure):
    _fields_ = [
        ("flags", C.c_uint32),
        ("err_pos", C.c_uint32),
        ("err_state", C.c_uint32),
        ("err_byte", C.c_uint8),
        ("err_def", C.c_uint8),
        ("reserved0", C.c_uint16),
        ("n_records", C.c_uint32),
        ("n_compact", C.c_uint32),
        ("reserved1", C.c_uint32 * 2),
    ]


class SubstrRecord(C.Structure):
    _fields_ = [
        ("start", C.c_uint32),
        ("len", C.c_uint32),
        ("substr_id", C.c_uint32),
        ("compact_off", C.c_uint32),
    ]


class BatchStatus(C.Structure):
    _fields_ = [
        ("code", C.c_int32),
        ("reserved", C.c_uint32),
        ("string_idx", C.c_uint64),
        ("pos", C.c_uint32),
        ("state", C.c_uint32),
        ("byte", C.c_uint8),
        ("defidx", C.c_uint8),
        ("reserved2", C.c_uint16),
        ("n_overlap_lo", C.c_uint32),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("row_pitch", C.c_uint64),
        ("bitmap_pitch", C.c_uint64),
        ("states", C.c_void_p * B2R_MAX_DEFS),
        ("substr_ids", C.c_void_p * B2R_MAX_DEFS),
        ("start_enable", C.c_void_p * B2R_MAX_DEFS),
        ("end_enable", C.c_void_p * B2R_MAX_DEFS),
        ("masked_chars", C.c_void_p),
        ("masked_substr_ids", C.c_void_p),
        ("status", C.c_void_p),
        ("records", C.c_void_p),
        ("max_records", C.c_uint32),
        ("compact_pitch", C.c_uint32),
        ("compact_bytes", C.c_void_p),
        ("mult", C.c_void_p * B2R_MAX_DEFS),
        ("endpoint_mult", C.c_void_p * B2R_MAX_DEFS),
        ("flags", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class RowCount(C.Structure):
    _fields_ = [("row", C.c_uint32), ("count", C.c_uint32)]


class StringMultStruct(C.Structure):
    """b2r_string_mult_outputs"""
    _fields_ = [
        ("max_entries", C.c_uint32),
        ("reserved", C.c_uint32),
        ("entries", C.c_void_p * B2R_MAX_DEFS),
        ("n_entries", C.c_void_p * B2R_MAX_DEFS),
        ("endpoint_counts", C.c_void_p * B2R_MAX_DEFS),
    ]


class StringMultPackedStruct(C.Structure):
    """b2r_string_mult_packed_outputs"""
    _fields_ = [
        ("capacity", C.c_uint64),
        ("entries", C.c_void_p * B2R_MAX_DEFS),
        ("row_start", C.c_void_p * B2R_MAX_DEFS),
        ("endpoint_counts", C.c_void_p * B2R_MAX_DEFS),
    ]


assert C.sizeof(StringStatus) == 32
assert C.sizeof(RowCount) == 8
assert C.sizeof(SubstrRecord) == 16
assert C.sizeof(BatchStatus) == 32

STATUS_DTYPE = [
    ("flags", "<u4"),
    ("err_pos", "<u4"),
    ("err_state", "<u4"),
    ("err_byte", "u1"),
    ("err_def", "u1"),
    ("reserved0", "<u2"),
    ("n_records", "<u4"),
    ("n_compact", "<u4"),
    ("reserved1", "<u4", (2,)),
]
RECORD_DTYPE = [("start", "<u4"), ("len", "<u4"), ("substr_id", "<u4"), ("compact_off", "<u4")]
