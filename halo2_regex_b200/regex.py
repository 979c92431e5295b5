"""`RegexVerifyConfig` — host mirror of the reference chip's witness-generation interface (src/lib.rs:97-131, 311-315,
779-785, 804-888) on top of the C ABI (include/b2r.h).  Same names, argument meaning and error behaviour for the path
this repo replaces; the halo2 constraint system / cell assignment is out of scope and stays in the host prover.
"""
import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _abi
from ._ffi import last_error, lib
from .buffers import HostOutputs, round_up
from .defs import RegexDefs


class InvalidTransitionError(RuntimeError):
    """The reference panics with this exact text (src/lib.rs:817)."""

    def __init__(self, state, char, string_idx=0, pos=0, defidx=0):
        super().__init__(f"The transition from {state} by {char} is invalid!")
        self.state, self.char, self.string_idx, self.pos, self.defidx = state, char, string_idx, pos, defidx


class StringTooLongError(ValueError):
    pass


def _raise(rc, res=None):
    if rc == 0:
        return
    if rc == _abi.B2R_ERR_INVALID_TRANSITION and res is not None:
        raise InvalidTransitionError(res.state, res.byte, res.string_idx, res.pos, res.defidx)
    if rc == _abi.B2R_ERR_TOO_LONG:
        raise StringTooLongError(last_error())
    raise RuntimeError(f"b2r error {rc}: {last_error()}")


@dataclass
class AssignedRegexResult:
    """Values of the reference's `AssignedRegexResult` (src/lib.rs:79-93), one entry per row (max_chars_size rows),
    plus the other witness columns of the same call."""
    all_enable_flags: np.ndarray
    all_characters: np.ndarray
    all_substr_ids: np.ndarray       # masked substr ids, as in the reference (src/lib.rs:766-771)
    masked_characters: np.ndarray
    states: list = field(default_factory=list)        # per def, M rows (final state at row len, dummy after)
    substr_ids: list = field(default_factory=list)    # per def, unmasked
    start_enable: list = field(default_factory=list)  # per def, bool
    end_enable: list = field(default_factory=list)
    accepted: list = field(default_factory=list)      # per def: state[len] == accepted_state_val (src/lib.rs:427-457)
    records: np.ndarray = None
    substr_bytes: bytes = b""


class DeviceOutputs:
    """Caller-owned DEVICE buffers (torch tensors) for one batch, laid out as include/b2r.h `b2r_outputs` describes."""

    def __init__(self, cfg, n_strings, row_pitch=None, bitmap_pitch=None, max_records=8, compact_pitch=64, want=None, device=None, max_chars_size=None):
        import torch
        self.cfg, self.n, self.m = cfg, int(n_strings), int(max_chars_size) if max_chars_size else cfg.max_chars_size   # max_chars_size: match_long (len + 1)
        self.row_pitch = int(row_pitch) if row_pitch else round_up(self.m, 32)
        self.bitmap_pitch = int(bitmap_pitch) if bitmap_pitch else round_up((self.m + 7) // 8, 32)
        want = set(want) if want else {"states", "substr_ids", "start_enable", "end_enable", "masked_chars", "masked_substr_ids",
                                       "status", "records", "compact_bytes", "mult", "endpoint_mult"}
        self.want = want
        dev = device if device is not None else torch.device("cuda", cfg.device)
        n, rp, bp = self.n, self.row_pitch, self.bitmap_pitch
        self.max_records, self.compact_pitch = int(max_records), int(compact_pitch)

        def z(shape, dtype=torch.uint8):
            return torch.empty(shape, dtype=dtype, device=dev)

        D = cfg.n_defs
        self.states = [z((n, rp), torch.uint8 if cfg.state_widths[d] == 1 else torch.int16) if "states" in want else None for d in range(D)]
        self.substr_ids = [z((n, rp)) if "substr_ids" in want else None for d in range(D)]
        self.start_enable = [z((n, bp)) if "start_enable" in want else None for d in range(D)]
        self.end_enable = [z((n, bp)) if "end_enable" in want else None for d in range(D)]
        # every multiplicity counter of the batch lives in ONE flat u64 buffer, so that the multi-GPU path all-reduces it with
        # a single collective and the finalisation kernel writes straight into the collective's buffer
        sizes = [cfg.table_num_rows[d] if "mult" in want else 0 for d in range(D)] + [2 * cfg.endpoint_num_rows[d] if "endpoint_mult" in want else 0 for d in range(D)]
        self.mult_all = torch.zeros(max(sum(sizes), 1), dtype=torch.int64, device=dev)
        views, o = [], 0
        for sz in sizes:
            views.append(self.mult_all[o:o + sz] if sz else None)
            o += sz
        self.mult, self.endpoint_mult = views[:D], views[D:]
        self.masked_chars = z((n, rp)) if "masked_chars" in want else None
        self.masked_substr_ids = z((n, rp)) if "masked_substr_ids" in want else None
        self.status = z((n, 32)) if "status" in want else None
        self.records = z((n, self.max_records, 16)) if "records" in want else None
        self.compact_bytes = z((n, self.compact_pitch)) if "compact_bytes" in want else None

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    def struct(self, flags=0):
        o = _abi.Outputs()
        o.row_pitch, o.bitmap_pitch = self.row_pitch, self.bitmap_pitch
        for d in range(self.cfg.n_defs):
            o.states[d] = self._p(self.states[d])
            o.substr_ids[d] = self._p(self.substr_ids[d])
            o.start_enable[d] = self._p(self.start_enable[d])
            o.end_enable[d] = self._p(self.end_enable[d])
            o.mult[d] = self._p(self.mult[d])
            o.endpoint_mult[d] = self._p(self.endpoint_mult[d])
        o.masked_chars = self._p(self.masked_chars)
        o.masked_substr_ids = self._p(self.masked_substr_ids)
        o.status = self._p(self.status)
        o.records = self._p(self.records)
        o.max_records = self.max_records if self.records is not None else 0
        o.compact_pitch = self.compact_pitch if self.compact_bytes is not None else 0
        o.compact_bytes = self._p(self.compact_bytes)
        o.flags = flags
        return o

    def to_host(self):
        """Copies every column into a HostOutputs (for comparison against the oracle)."""
        cfg = self.cfg
        h = HostOutputs(self.n, self.m, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, row_pitch=self.row_pitch,
                        bitmap_pitch=self.bitmap_pitch, max_records=self.max_records, compact_pitch=self.compact_pitch, want=self.want)

        def cp(dst, src):
            if dst is not None and src is not None:
                dst.view(np.uint8).reshape(-1)[:] = src.contiguous().view(-1).view(dtype=__import__("torch").uint8).cpu().numpy()

        for d in range(cfg.n_defs):
            cp(h.states[d], self.states[d]); cp(h.substr_ids[d], self.substr_ids[d])
            cp(h.start_enable[d], self.start_enable[d]); cp(h.end_enable[d], self.end_enable[d])
            cp(h.mult[d], self.mult[d]); cp(h.endpoint_mult[d], self.endpoint_mult[d])
        cp(h.masked_chars, self.masked_chars); cp(h.masked_substr_ids, self.masked_substr_ids)
        cp(h.status, self.status); cp(h.records, self.records); cp(h.compact_bytes, self.compact_bytes)
        return h

    def written_bytes(self):
        """Algorithmic witness bytes this batch writes: M defined rows per string per column (SURVEY 8(d))."""
        n, m, bm = self.n, self.m, (self.m + 7) // 8
        tot = 0
        for d in range(self.cfg.n_defs):
            tot += n * m * self.cfg.state_widths[d] if self.states[d] is not None else 0
            tot += n * m if self.substr_ids[d] is not None else 0
            tot += n * bm if self.start_enable[d] is not None else 0
            tot += n * bm if self.end_enable[d] is not None else 0
            tot += 8 * self.cfg.table_num_rows[d] if self.mult[d] is not None else 0
            tot += 16 * self.cfg.endpoint_num_rows[d] if self.endpoint_mult[d] is not None else 0
        tot += n * m if self.masked_chars is not None else 0
        tot += n * m if self.masked_substr_ids is not None else 0
        tot += n * 32 if self.status is not None else 0
        return tot


class StringMultOutputs:
    """Per-string lookup multiplicities (include/b2r.h `b2r_string_mult_outputs`) as torch tensors: per def `entries[d]`
    (n, max_entries, 2) int32 holding (row, count) pairs as u32, `n_entries[d]` (n,), `endpoint_counts[d]` (n, 2*E_d).
    `device`: the handle's GPU by default (b2r_string_mult), "cpu" for the host entry points (`pin=True`: page-locked).
    `max_entries` defaults to max_d min(M, T_d), which never truncates; `fill`: a byte pattern for every buffer."""

    WANT = ("entries", "n_entries", "endpoint_counts")

    def __init__(self, cfg, n, max_entries=None, device=None, want=WANT, fill=None, pin=False, max_chars_size=None):
        import torch
        self.cfg, self.n = cfg, int(n)
        self.m = int(max_chars_size) if max_chars_size else cfg.max_chars_size
        self.max_entries = int(max_entries) if max_entries is not None else max(min(self.m, t) for t in cfg.table_num_rows)
        if device is None:
            device = torch.device("cuda", cfg.device) if cfg.device >= 0 else "cpu"
        dev = torch.device(device)
        self.want = set(want)

        def z(shape):
            t = torch.empty(shape, dtype=torch.int32, device=dev, pin_memory=pin and dev.type == "cpu")
            if fill is not None:
                t.view(torch.uint8).fill_(fill)
            return t

        D = cfg.n_defs
        self.entries = [z((self.n, self.max_entries, 2)) if "entries" in self.want else None for _ in range(D)]
        self.n_entries = [z((self.n,)) if "n_entries" in self.want or "entries" in self.want else None for _ in range(D)]
        self.endpoint_counts = [z((self.n, 2 * cfg.endpoint_num_rows[d])) if "endpoint_counts" in self.want else None for d in range(D)]

    def struct(self):
        s = _abi.StringMultStruct()
        s.max_entries = self.max_entries
        for d in range(self.cfg.n_defs):
            for name in ("entries", "n_entries", "endpoint_counts"):
                t = getattr(self, name)[d]
                getattr(s, name)[d] = None if t is None else t.data_ptr()
        return s

    def to_host(self):
        """A copy of every buffer in host memory."""
        h = StringMultOutputs.__new__(StringMultOutputs)
        h.cfg, h.n, h.m, h.max_entries, h.want = self.cfg, self.n, self.m, self.max_entries, set(self.want)
        for name in ("entries", "n_entries", "endpoint_counts"):
            setattr(h, name, [None if t is None else t.cpu() for t in getattr(self, name)])
        return h

    def dense(self, j, d):
        """The T_d-long count vector of string j (uint64): the mult[d] of a one-string batch of that string."""
        out = np.zeros(self.cfg.table_num_rows[d], dtype=np.uint64)
        k = min(int(self.n_entries[d][j]), self.max_entries)
        e = self.entries[d][j, :k].cpu().numpy().view(np.uint32)
        out[e[:, 0]] = e[:, 1]
        return out


class StringMultPacked:
    """Per-string lookup multiplicities in the packed layout (include/b2r.h `b2r_string_mult_packed_outputs`) as torch tensors:
    per def `entries[d]` (capacity, 2) int32 holding (row, count) pairs as u32, string j's list at
    entries[d][row_start[d][j] : row_start[d][j + 1]]; `row_start[d]` (n + 1,) int64; `endpoint_counts[d]` (n, 2*E_d).
    `capacity` defaults to the worst case n * max_d min(M, T_d), so every list is stored; a list is stored only when
    row_start[d][j + 1] <= capacity.  `device`, `pin`, `fill`, `max_chars_size`: as for StringMultOutputs."""

    WANT = ("entries", "row_start", "endpoint_counts")

    def __init__(self, cfg, n, capacity=None, device=None, want=WANT, fill=None, pin=False, max_chars_size=None):
        import torch
        self.cfg, self.n = cfg, int(n)
        self.m = int(max_chars_size) if max_chars_size else cfg.max_chars_size
        self.capacity = int(capacity) if capacity is not None else self.n * max(min(self.m, t) for t in cfg.table_num_rows)
        if device is None:
            device = torch.device("cuda", cfg.device) if cfg.device >= 0 else "cpu"
        dev = torch.device(device)
        self.want = set(want)

        def z(shape, dtype=torch.int32):
            t = torch.empty(shape, dtype=dtype, device=dev, pin_memory=pin and dev.type == "cpu")
            if fill is not None:
                t.view(torch.uint8).fill_(fill)
            return t

        D = cfg.n_defs
        self.entries = [z((self.capacity, 2)) if "entries" in self.want else None for _ in range(D)]
        self.row_start = [z((self.n + 1,), torch.int64) if "row_start" in self.want or "entries" in self.want else None for _ in range(D)]
        self.endpoint_counts = [z((self.n, 2 * cfg.endpoint_num_rows[d])) if "endpoint_counts" in self.want else None for d in range(D)]

    def struct(self):
        s = _abi.StringMultPackedStruct()
        s.capacity = self.capacity
        for d in range(self.cfg.n_defs):
            for name in ("entries", "row_start", "endpoint_counts"):
                t = getattr(self, name)[d]
                getattr(s, name)[d] = None if t is None or t.numel() == 0 else t.data_ptr()
        return s

    def to_host(self):
        """A copy of every buffer in host memory."""
        h = StringMultPacked.__new__(StringMultPacked)
        h.cfg, h.n, h.m, h.capacity, h.want = self.cfg, self.n, self.m, self.capacity, set(self.want)
        for name in ("entries", "row_start", "endpoint_counts"):
            setattr(h, name, [None if t is None else t.cpu() for t in getattr(self, name)])
        return h

    def stored(self, j, d):
        """True when string j's list of def d is in `entries` (row_start[d][j + 1] <= capacity)."""
        return self.entries[d] is not None and int(self.row_start[d][j + 1]) <= self.capacity

    def entries_of(self, j, d):
        """The (row, count) list of string j and def d as a (k, 2) uint32 array, rows ascending.  LookupError when it is not
        stored (the capacity ran out before it)."""
        if not self.stored(j, d):
            raise LookupError(f"string {j}, def {d}: list not stored (row_start[{j + 1}] > capacity {self.capacity})")
        a, b = int(self.row_start[d][j]), int(self.row_start[d][j + 1])
        return self.entries[d][a:b].cpu().numpy().view(np.uint32)

    def dense(self, j, d):
        """The T_d-long count vector of string j (uint64): the mult[d] of a one-string batch of that string."""
        out = np.zeros(self.cfg.table_num_rows[d], dtype=np.uint64)
        e = self.entries_of(j, d)
        out[e[:, 0]] = e[:, 1]
        return out


class RegexVerifyConfig:
    """reference src/lib.rs:97-113.  `configure` takes the two parameters that matter for witness generation
    (`max_chars_size`, `regex_defs`, src/lib.rs:126-131); `meta` / `gate` belong to the halo2 side and are ignored."""

    def __init__(self, max_chars_size, regex_defs, device=None, devices=None):
        self.max_chars_size = int(max_chars_size)
        self.regex_defs = list(regex_defs)
        for rd in self.regex_defs:
            assert isinstance(rd, RegexDefs)
        self.devices = [int(x) for x in devices] if devices is not None else None
        if self.devices is not None:
            device = -1           # multi-device handle (b2r_config_new_multi): one process, several GPUs
        if device is None:
            try:
                import torch
                device = torch.cuda.current_device() if torch.cuda.is_available() else -1
            except ImportError:  # pragma: no cover
                device = -1
        self.device = int(device)
        D = len(self.regex_defs)
        allstr = (C.c_void_p * D)(*[rd.allstr._h for rd in self.regex_defs])
        sub_arrays = [(C.c_void_p * max(1, len(rd.substrs)))(*[s._h for s in rd.substrs]) for rd in self.regex_defs]
        subs = (C.POINTER(C.c_void_p) * D)(*[C.cast(a, C.POINTER(C.c_void_p)) for a in sub_arrays])
        ns = (C.c_uint32 * D)(*[len(rd.substrs) for rd in self.regex_defs])
        h = C.c_void_p()
        if self.devices is not None:
            ids = (C.c_int * len(self.devices))(*self.devices)
            rc = lib.b2r_config_new_multi(allstr, subs, ns, D, self.max_chars_size, ids, len(self.devices), C.byref(h))
        else:
            rc = lib.b2r_config_new(allstr, subs, ns, D, self.max_chars_size, self.device, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"b2r_config_new failed ({rc}): {last_error()}")
        self._h = h
        self.n_defs = D
        self.state_widths = [lib.b2r_config_state_width(h, d) for d in range(D)]
        self.dummy_states = [lib.b2r_config_dummy_state(h, d) for d in range(D)]
        self.substr_id_offsets = [lib.b2r_config_substr_id_offset(h, d) for d in range(D)]
        self.table_num_rows = [lib.b2r_table_num_rows(h, d) for d in range(D)]
        self.endpoint_num_rows = [lib.b2r_endpoint_num_rows(h, d) for d in range(D)]
        self.num_byte_classes = [lib.b2r_config_num_byte_classes(h, d) for d in range(D)]

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib.b2r_config_free(h)

    @classmethod
    def configure(cls, max_chars_size, regex_defs, meta=None, gate=None, device=None, devices=None):
        return cls(max_chars_size, regex_defs, device=device, devices=devices)

    def set_option(self, name, value):
        """Testing / tuning knobs of the handle (b2r_config_set_option): "table_mode", "hist_mode", "fuse", "slices", ..."""
        _raise(lib.b2r_config_set_option(self._h, str(name).encode(), str(value).encode()))

    def last_host_bytes(self):
        """(host->device, device->host) bytes the last host-pointer call moved over PCIe."""
        a, b = C.c_uint64(), C.c_uint64()
        _raise(lib.b2r_last_host_bytes(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # ---- RegexVerifyConfig::load → RegexTableConfig::load (src/lib.rs:779-785, src/table.rs:61-198) -----------------
    def table_rows(self, d):
        out = np.zeros((self.table_num_rows[d], 4), dtype=np.uint64)
        _raise(lib.b2r_table_rows(self._h, d, out.ctypes.data, len(out)))
        return out

    def endpoint_rows(self, d):
        out = np.zeros((self.endpoint_num_rows[d], 3), dtype=np.uint64)
        _raise(lib.b2r_endpoint_rows(self._h, d, out.ctypes.data, len(out)))
        return out

    def load(self):
        """Rows of the fixed lookup tables in the reference's order, per def: [(transition_rows, endpoint_rows), ...]"""
        return [(self.table_rows(d), self.endpoint_rows(d)) for d in range(self.n_defs)]

    # ---- batches --------------------------------------------------------------------------------------------------
    def new_host_outputs(self, n, **kw):
        return HostOutputs(n, self.max_chars_size, self.state_widths, self.table_num_rows, self.endpoint_num_rows, **kw)

    def match_batch_host(self, data, offsets, out=None, flags=0, check=True, sparse=False, reuse=False, **kw):
        """Host buffers in, host buffers out (H2D, kernels, D2H inside): the call a drop-in shim makes.
        sparse=True: B2R_OUT_SPARSE_D2H — the zero-dominated columns cross PCIe compacted and are expanded by host threads.
        reuse=True: B2R_OUT_SPARSE_REUSE — `out` is what the previous call on this handle filled: only its sectors are cleared."""
        return self._host_call(lib.b2r_match_batch_host, data, offsets, out, flags, check, sparse, reuse, kw)

    def match_batch_chunked_host(self, data, offsets, out=None, flags=0, check=True, sparse=False, reuse=False, **kw):
        """b2r_match_batch_chunked_host: the call and the outputs of match_batch_host, with the kernels of
        match_batch_chunked_device (every string cut into 1 KiB chunks walked in parallel) — for batches of few, long strings."""
        return self._host_call(lib.b2r_match_batch_chunked_host, data, offsets, out, flags, check, sparse, reuse, kw)

    def _host_call(self, fn, data, offsets, out, flags, check, sparse, reuse, kw):
        if sparse:
            flags |= _abi.B2R_OUT_SPARSE_D2H
        if reuse:
            flags |= _abi.B2R_OUT_SPARSE_REUSE
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        if out is None:
            out = self.new_host_outputs(n, **kw)
        st = out.struct(flags)
        res = _abi.BatchStatus()
        rc = fn(self._h, data.ctypes.data, offsets.ctypes.data, n, C.byref(st), C.byref(res))
        if check:
            _raise(rc, res)
        return out, res

    def match_batch_host_mult(self, data, offsets, out=None, sm=None, flags=0, check=True, sparse=False, reuse=False, max_entries=None, **kw):
        """b2r_match_batch_host_mult: match_batch_host plus the per-string lookup multiplicities into `sm` (a host
        StringMultOutputs, allocated here if not given).  Returns (out, sm, batch result)."""
        return self._host_call_mult(lib.b2r_match_batch_host_mult, data, offsets, out, sm, flags, check, sparse, reuse, max_entries, kw)

    def match_batch_chunked_host_mult(self, data, offsets, out=None, sm=None, flags=0, check=True, sparse=False, reuse=False, max_entries=None, **kw):
        """b2r_match_batch_chunked_host_mult: match_batch_chunked_host plus the per-string lookup multiplicities."""
        return self._host_call_mult(lib.b2r_match_batch_chunked_host_mult, data, offsets, out, sm, flags, check, sparse, reuse, max_entries, kw)

    def _host_call_mult(self, fn, data, offsets, out, sm, flags, check, sparse, reuse, max_entries, kw):
        n = len(offsets) - 1
        if sm is None:
            sm = StringMultOutputs(self, n, max_entries=max_entries, device="cpu")
        s = sm.struct()
        call = lambda h, b, o, n_, st, res: fn(h, b, o, n_, st, C.byref(s), res)  # noqa: E731
        out, res = self._host_call(call, data, offsets, out, flags, check, sparse, reuse, kw)
        return out, sm, res

    def match_batch_host_mult_packed(self, data, offsets, out=None, pk=None, flags=0, check=True, sparse=False, reuse=False, capacity=None, **kw):
        """b2r_match_batch_host_mult_packed: match_batch_host plus the per-string lookup multiplicities in the packed layout
        into `pk` (a host StringMultPacked, allocated here if not given).  Returns (out, pk, batch result)."""
        return self._host_call_packed(lib.b2r_match_batch_host_mult_packed, data, offsets, out, pk, flags, check, sparse, reuse, capacity, kw)

    def match_batch_chunked_host_mult_packed(self, data, offsets, out=None, pk=None, flags=0, check=True, sparse=False, reuse=False, capacity=None,
                                             **kw):
        """b2r_match_batch_chunked_host_mult_packed: match_batch_chunked_host plus the packed per-string lookup multiplicities."""
        return self._host_call_packed(lib.b2r_match_batch_chunked_host_mult_packed, data, offsets, out, pk, flags, check, sparse, reuse, capacity, kw)

    def _host_call_packed(self, fn, data, offsets, out, pk, flags, check, sparse, reuse, capacity, kw):
        n = len(offsets) - 1
        if pk is None:
            pk = StringMultPacked(self, n, capacity=capacity, device="cpu")
        s = pk.struct()
        call = lambda h, b, o, n_, st, res: fn(h, b, o, n_, st, C.byref(s), res)  # noqa: E731
        out, res = self._host_call(call, data, offsets, out, flags, check, sparse, reuse, kw)
        return out, pk, res

    def string_mult_packed_device(self, d_bytes, d_offsets, out, pk=None, max_chars_size=0, stream=None, capacity=None):
        """b2r_string_mult_packed: string_mult_device's counts in the packed layout (StringMultPacked, on the device).
        Asynchronous on `stream`.  Returns `pk`."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(d_bytes.device)
        n = d_offsets.numel() - 1
        if pk is None:
            pk = StringMultPacked(self, n, capacity=capacity, device=d_bytes.device, max_chars_size=max_chars_size or None)
        rc = lib.b2r_string_mult_packed(self._h, d_bytes.data_ptr(), d_offsets.data_ptr(), n, d_bytes.numel(), int(max_chars_size),
                                        C.byref(out.struct()), C.byref(pk.struct()), stream.cuda_stream)
        _raise(rc)
        return pk

    def string_mult_device(self, d_bytes, d_offsets, out, sm=None, max_chars_size=0, stream=None, max_entries=None):
        """b2r_string_mult: per-string lookup multiplicities from the state columns and status that an earlier
        match_batch_device / match_batch_chunked_device / match_long_device call wrote into `out` (same bytes and offsets;
        after match_long_device pass max_chars_size = len + 1 and offsets [0, len]).  Asynchronous on `stream`.  Returns `sm`."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(d_bytes.device)
        n = d_offsets.numel() - 1
        if sm is None:
            sm = StringMultOutputs(self, n, max_entries=max_entries, device=d_bytes.device, max_chars_size=max_chars_size or None)
        rc = lib.b2r_string_mult(self._h, d_bytes.data_ptr(), d_offsets.data_ptr(), n, d_bytes.numel(), int(max_chars_size),
                                 C.byref(out.struct()), C.byref(sm.struct()), stream.cuda_stream)
        _raise(rc)
        return sm

    def match_strings(self, strings, **kw):
        data = np.frombuffer(b"".join(strings), dtype=np.uint8) if strings else np.zeros(0, np.uint8)
        offs = np.zeros(len(strings) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(s) for s in strings])
        return self.match_batch_host(data, offs, **kw)

    def match_batch_device(self, d_bytes, d_offsets, out, flags=0, stream=None):
        """Device tensors in/out, asynchronous on `stream` (torch.cuda.Stream or None = current stream)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(d_bytes.device)
        n = d_offsets.numel() - 1
        st = out.struct(flags)
        rc = lib.b2r_match_batch(self._h, d_bytes.data_ptr(), d_offsets.data_ptr(), n, d_bytes.numel(), C.byref(st), stream.cuda_stream)
        _raise(rc)
        return out

    def match_batch_chunked_device(self, d_bytes, d_offsets, out, flags=0, stream=None):
        """b2r_match_batch_chunked: the same call and the same outputs as match_batch_device, with every string cut into 1 KiB
        chunks that are walked in parallel (batches of few, long strings).  Asynchronous on `stream`."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(d_bytes.device)
        n = d_offsets.numel() - 1
        st = out.struct(flags)
        rc = lib.b2r_match_batch_chunked(self._h, d_bytes.data_ptr(), d_offsets.data_ptr(), n, d_bytes.numel(), C.byref(st), stream.cuda_stream)
        _raise(rc)
        return out

    def match_long_device(self, d_bytes, out, flags=0, stream=None):
        """b2r_match_long: ONE string (the whole of `d_bytes`, a device tensor) with max_chars_size = len + 1; `out` is a
        DeviceOutputs(cfg, 1, max_chars_size=len + 1); `flags`: B2R_OUT_* (B2R_OUT_ACCUMULATE_MULT adds into out's counters).
        Asynchronous on `stream`."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(d_bytes.device)
        st = out.struct(flags)
        rc = lib.b2r_match_long(self._h, d_bytes.data_ptr(), d_bytes.numel(), C.byref(st), stream.cuda_stream)
        _raise(rc)
        return out

    def match_long_host(self, data, out=None, flags=0, check=True, **kw):
        """b2r_match_long_host: ONE string (host bytes) through the chunked long-string path, max_chars_size = len + 1;
        host buffers out (`out`: HostOutputs(1, len + 1, ...), allocated here if not given); `flags`: B2R_OUT_*
        (B2R_OUT_ACCUMULATE_MULT adds into out's counters)."""
        data = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data, dtype=np.uint8)
        if out is None:
            out = HostOutputs(1, len(data) + 1, self.state_widths, self.table_num_rows, self.endpoint_num_rows, **kw)
        st = out.struct(flags)
        res = _abi.BatchStatus()
        rc = lib.b2r_match_long_host(self._h, data.ctypes.data, len(data), C.byref(st), C.byref(res))
        if check:
            _raise(rc, res)
        return out, res

    # ---- the step after the path: columns as BN254 Fr cells (src/lib.rs:342-347, 388-418: Value::known(F::from(x))) -----------
    def column_to_fr(self, col, kind=None, rows=None, offsets=None, stream=None):
        """b2r_column_to_fr: a device column (torch tensor (n, pitch): uint8 -> B2R_COL_U8, int16 -> _U16, int64 -> _U64;
        kind="bitmap": an LSB-first bitmap column; kind="chars" / "enable": `col` = the input bytes, `offsets` the N+1 offsets) ->
        int64 tensor (n, rows, 4): little-endian Montgomery limbs of halo2curves::bn256::Fr::from(value)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(col.device)
        rows = int(rows) if rows else self.max_chars_size
        kinds = {"u8": _abi.B2R_COL_U8, "u16": _abi.B2R_COL_U16, "u64": _abi.B2R_COL_U64, "bitmap": _abi.B2R_COL_BITMAP,
                 "chars": _abi.B2R_COL_CHARS, "enable": _abi.B2R_COL_ENABLE}
        if kind is None:
            kind = {torch.uint8: "u8", torch.int16: "u16", torch.int64: "u64"}[col.dtype]
        if kind in ("chars", "enable"):
            n, pitch = offsets.numel() - 1, 0
        else:
            n, pitch = col.shape[0], col.shape[1]
        out = torch.empty((n, rows, 4), dtype=torch.int64, device=col.device)
        rc = lib.b2r_column_to_fr(self._h, col.data_ptr(), kinds[kind], offsets.data_ptr() if offsets is not None else None, n, rows, pitch,
                                  out.data_ptr(), stream.cuda_stream)
        _raise(rc)
        return out

    def batch_result(self, stream=None, check=True):
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(torch.device("cuda", self.device))
        res = _abi.BatchStatus()
        rc = lib.b2r_batch_result(self._h, stream.cuda_stream, C.byref(res))
        if check:
            _raise(rc, res)
        return res

    def last_launch_count(self):
        return lib.b2r_last_launch_count(self._h)

    def set_timing(self, enable=True):
        _raise(lib.b2r_config_set_timing(self._h, 1 if enable else 0))

    def last_kernel_ms(self):
        w, t = C.c_float(), C.c_float()
        _raise(lib.b2r_last_kernel_ms(self._h, C.byref(w), C.byref(t)))
        return w.value, t.value

    def last_stage_ms(self):
        """(walk_kernel, emit_kernel, finalize_kernel) device times of the last call, in ms."""
        ms = (C.c_float * 3)()
        _raise(lib.b2r_last_stage_ms(self._h, ms))
        return ms[0], ms[1], ms[2]

    def last_plan(self):
        """(table placement, bin placement) chosen by the last call: see b2r_last_plan in include/b2r.h."""
        t, h = C.c_uint32(), C.c_uint32()
        _raise(lib.b2r_last_plan(self._h, C.byref(t), C.byref(h)))
        return ("repl", "plain", "global", "plain16", "repl16")[t.value], ("none", "smem", "global")[h.value]

    # ---- match_substrs (src/lib.rs:311-773): one string ------------------------------------------------------------
    def match_substrs(self, characters, ctx=None):
        characters = bytes(characters)
        out, _ = self.match_strings([characters], max_records=64, compact_pitch=max(64, self.max_chars_size))
        M, L = self.max_chars_size, len(characters)
        enable = np.zeros(M, dtype=np.uint8)
        enable[:L] = 1
        chars = np.zeros(M, dtype=np.uint8)
        chars[:L] = np.frombuffer(characters, dtype=np.uint8)
        flags = int(out.status["flags"][0])
        nrec = min(int(out.status["n_records"][0]), out.max_records)
        return AssignedRegexResult(
            all_enable_flags=enable, all_characters=chars,
            all_substr_ids=out.masked_substr_ids[0, :M].copy(), masked_characters=out.masked_chars[0, :M].copy(),
            states=[out.states[d][0, :M].copy() for d in range(self.n_defs)],
            substr_ids=[out.substr_ids[d][0, :M].copy() for d in range(self.n_defs)],
            start_enable=[out.bits(out.start_enable[d])[0] for d in range(self.n_defs)],
            end_enable=[out.bits(out.end_enable[d])[0] for d in range(self.n_defs)],
            accepted=[bool(flags & _abi.B2R_ST_ACCEPTED(d)) for d in range(self.n_defs)],
            records=out.records[0, :nrec].copy(),
            substr_bytes=bytes(out.compact_bytes[0, :min(int(out.status["n_compact"][0]), out.compact_pitch)]),
        )

    # ---- the three derive_* helpers of the reference (src/lib.rs:804-888), same return shapes ------------------------
    def derive_states(self, characters):
        r = self.match_substrs(characters)
        L = len(characters)
        return [[int(x) for x in r.states[d][:L + 1]] for d in range(self.n_defs)]

    def derive_substr_ids(self, characters):
        r = self.match_substrs(characters)
        L = len(characters)
        return [[int(x) for x in r.substr_ids[d][:L]] for d in range(self.n_defs)]

    def derive_is_start_end(self, characters):
        r = self.match_substrs(characters)
        L = len(characters)
        is_starts = [[bool(x) for x in r.start_enable[d][:L]] + [False] for d in range(self.n_defs)]
        is_ends = [[False] + [bool(x) for x in r.end_enable[d][:L]] for d in range(self.n_defs)]
        return is_starts, is_ends
