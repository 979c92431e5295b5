"""Per-string lookup multiplicities in the packed layout: b2r_string_mult_packed (device) and b2r_match_batch_host_mult_packed /
b2r_match_batch_chunked_host_mult_packed.  The contract (include/b2r.h): string j's list is exactly the list b2r_string_mult writes
with max_entries >= min(M, T_d), at entries[row_start[j] .. row_start[j+1]); row_start is always complete; a list is stored only
when row_start[j+1] <= capacity, and every other entry slot is left untouched.  The slot call is the reference here; a subset is
also checked against one-string oracle batches."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, product_config
from test_batch_chunked import ALPHA, _strings, _to_device
from test_dfa_shapes import _product, make_dfa
from test_gpu_parity import _pack
from test_string_mult import _config1_like, _expected, _ragged

FILL = 0x5A
FILL_WORD = 0x5A5A5A5A


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_packed_struct_layout():
    from halo2_regex_b200 import _abi
    S = _abi.StringMultPackedStruct
    assert C.sizeof(S) == 8 + 3 * 4 * 8
    assert (S.capacity.offset, S.entries.offset, S.row_start.offset, S.endpoint_counts.offset) == (0, 8, 40, 72)


def test_packed_symbols_exported():
    import subprocess
    import halo2_regex_b200 as H
    out = subprocess.check_output(["nm", "-D", H.LIB_PATH]).decode()
    for name in ("b2r_string_mult_packed", "b2r_match_batch_host_mult_packed", "b2r_match_batch_chunked_host_mult_packed"):
        assert f" T {name}\n" in out


def _pk_struct(cfg, entries=True, row_start=True, ep=True, capacity=16, base=0x10000):
    from halo2_regex_b200 import _abi
    s = _abi.StringMultPackedStruct()
    s.capacity = capacity
    for d in range(cfg.n_defs):
        s.entries[d] = base + 0x1000 * d if entries else None
        s.row_start[d] = base + 0x100000 + 0x1000 * d if row_start else None
        s.endpoint_counts[d] = base + 0x200000 + 0x1000 * d if ep else None
    return s


def _dev_out(cfg, states=True, status=True):
    from halo2_regex_b200 import _abi
    o = _abi.Outputs()
    o.row_pitch = 1056
    o.bitmap_pitch = 160
    for d in range(cfg.n_defs):
        o.states[d] = 0x400000 + 0x10000 * d if states else None
    o.status = 0x800000 if status else None
    return o


def _calls(cfg, out, pk):
    from halo2_regex_b200 import _abi
    from halo2_regex_b200._ffi import lib
    data = np.zeros(16, np.uint8)
    offs = np.array([0, 3], np.uint64)
    res = _abi.BatchStatus()
    return [lib.b2r_string_mult_packed(cfg._h, 0x1000, 0x2000, 1, 3, 0, C.byref(out), C.byref(pk), None),
            lib.b2r_match_batch_host_mult_packed(cfg._h, data.ctypes.data, offs.ctypes.data, 1, C.byref(out), C.byref(pk), C.byref(res)),
            lib.b2r_match_batch_chunked_host_mult_packed(cfg._h, data.ctypes.data, offs.ctypes.data, 1, C.byref(out), C.byref(pk), C.byref(res))]


def test_packed_deviceless_handle_and_argument_errors():
    from halo2_regex_b200 import _abi
    from halo2_regex_b200._ffi import lib
    cfg = product_config("three", 1025, device=-1)
    ok = _pk_struct(cfg)
    assert _calls(cfg, _dev_out(cfg), ok) == [_abi.B2R_ERR_CUDA] * 3
    # entries without row_start; capacity 0 and offsets only are fine
    assert _calls(cfg, _dev_out(cfg), _pk_struct(cfg, row_start=False)) == [_abi.B2R_ERR_INVALID_ARG] * 3
    assert _calls(cfg, _dev_out(cfg), _pk_struct(cfg, capacity=0)) == [_abi.B2R_ERR_CUDA] * 3
    assert _calls(cfg, _dev_out(cfg), _pk_struct(cfg, entries=False, capacity=0)) == [_abi.B2R_ERR_CUDA] * 3
    # the device entry reads the state columns and the status; the host entries use scratch ones
    assert _calls(cfg, _dev_out(cfg, states=False), ok) == [_abi.B2R_ERR_INVALID_ARG, _abi.B2R_ERR_CUDA, _abi.B2R_ERR_CUDA]
    assert _calls(cfg, _dev_out(cfg, status=False), ok) == [_abi.B2R_ERR_INVALID_ARG, _abi.B2R_ERR_CUDA, _abi.B2R_ERR_CUDA]
    assert _calls(cfg, _dev_out(cfg, states=False, status=False), _pk_struct(cfg, False, False, False))[0] == _abi.B2R_ERR_CUDA
    # alignment: entries and row_start 8 bytes, endpoint counts 4
    for field, off in (("entries", 4), ("row_start", 4), ("endpoint_counts", 2)):
        s = _pk_struct(cfg)
        getattr(s, field)[1] += off
        assert _calls(cfg, _dev_out(cfg), s) == [_abi.B2R_ERR_ALIGNMENT] * 3, field
    s = _pk_struct(cfg)
    s.endpoint_counts[2] += 4
    assert _calls(cfg, _dev_out(cfg), s) == [_abi.B2R_ERR_CUDA] * 3
    assert lib.b2r_string_mult_packed(cfg._h, None, None, 0, 0, 0, None, C.byref(ok), None) == _abi.B2R_ERR_INVALID_ARG
    assert lib.b2r_string_mult_packed(None, None, None, 0, 0, 0, None, None, None) == _abi.B2R_ERR_INVALID_ARG


def test_packed_holder_on_host():
    import torch
    import halo2_regex_b200 as H
    cfg = product_config("regex1", 1025, device=-1)
    pk = H.StringMultPacked(cfg, 3, device="cpu", capacity=5)
    assert pk.row_start[0].shape == (4,) and pk.entries[0].shape == (5, 2)
    assert H.StringMultPacked(cfg, 3, device="cpu").capacity == 3 * min(1025, cfg.table_num_rows[0])
    pk.row_start[0][:] = torch.tensor([0, 3, 3, 6])
    pk.entries[0][:3] = torch.tensor([[0, 1000], [5, 20], [7, 5]], dtype=torch.int32)
    v = pk.dense(0, 0)
    assert len(v) == cfg.table_num_rows[0] and v[0] == 1000 and v[5] == 20 and v[7] == 5 and v.sum() == 1025
    assert len(pk.entries_of(1, 0)) == 0 and pk.stored(1, 0) and not pk.stored(2, 0)
    with pytest.raises(LookupError):
        pk.entries_of(2, 0)


# ---- helpers of the GPU cases ----------------------------------------------------------------------------------------------
def _np(t, dtype=np.uint32):
    return None if t is None else t.cpu().numpy().view(dtype)


def _slot_lists(sm, d):
    """The slot call's lists of def d: (n_entries, [per string (k, 2) uint32])"""
    ent, ne = _np(sm.entries[d]), _np(sm.n_entries[d])
    assert (ne <= sm.max_entries).all()
    return ne, [ent[j, :ne[j]] for j in range(len(ne))]


def _vs_slot(pk, sm, ep=True):
    """packed == slot call with max_entries >= min(M, T_d): row_start is the prefix of n_entries, every list equal"""
    for d in range(pk.cfg.n_defs):
        ne, lists = _slot_lists(sm, d)
        rs = _np(pk.row_start[d], np.uint64)
        assert rs[0] == 0 and np.array_equal(np.diff(rs.astype(np.int64)), ne.astype(np.int64)), d
        if pk.entries[d] is not None:
            e = _np(pk.entries[d])
            assert int(rs[-1]) <= pk.capacity
            for j in range(len(ne)):
                assert np.array_equal(e[rs[j]:rs[j + 1]], lists[j]), (d, j)
        if ep:
            assert np.array_equal(_np(pk.endpoint_counts[d]), _np(sm.endpoint_counts[d])), d


def _device_pair(cfg, data, offs, chunked=False, M=0, capacity=None, **pkw):
    """match on the device, then the slot call (max_entries = max_d min(M, T_d)) and the packed call on the same columns"""
    import torch
    import halo2_regex_b200 as H
    d_bytes, d_offs = _to_device(data, offs)
    n = len(offs) - 1
    out = H.DeviceOutputs(cfg, n, want={"states", "status", "mult", "endpoint_mult"})
    (cfg.match_batch_chunked_device if chunked else cfg.match_batch_device)(d_bytes, d_offs, out)
    sm = cfg.string_mult_device(d_bytes, d_offs, out, max_chars_size=M)
    pk = H.StringMultPacked(cfg, n, fill=FILL, capacity=capacity, max_chars_size=M or None, **pkw)
    cfg.string_mult_packed_device(d_bytes, d_offs, out, pk, max_chars_size=M)
    torch.cuda.synchronize()
    return out, sm, pk, (d_bytes, d_offs)


def _dfa_set(which, M):
    import halo2_regex_b200 as H
    from halo2_regex_b200 import workloads as W
    if which in ("regex1", "three"):
        return product_config(which, M), None
    if which == "large_dfa":
        allstr, substr, _ = W.large_dfa_texts()
        cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
        return cfg, None
    dfas = [make_dfa(300, 4, 0, 7, "perm", seed=3, alphabet=b"xyz."), make_dfa(40, 3, 1, 5, "collapse_2", seed=4, alphabet=b"xyz.")]
    return _product(dfas, M), b"xyz."


def _set_strings(which, M, n, seed):
    """ragged lengths with 0 and M - 1, some invalid bytes, two strings too long"""
    from halo2_regex_b200 import workloads as W
    if which in ("regex1", "three"):
        return _ragged(which, M, n, seed)
    rng = np.random.default_rng(seed)
    if which == "large_dfa":
        rows, _ = W.config4_numpy(n, M - 1)
    else:
        rows = np.frombuffer(b"xyz.", np.uint8)[rng.integers(0, 4, size=(n, M - 1))]
    lens = rng.integers(0, M, size=n)
    lens[:3] = [0, M - 1, 1]
    strings = [bytes(rows[j, :lens[j]]) for j in range(n)]
    for k in range(5, n, 31):
        if strings[k]:
            s = bytearray(strings[k])
            s[len(s) // 2] = 0xFF
            strings[k] = bytes(s)
    return strings + [b"x" * M, b"." * (M + 7)]


# ---- 1. equal to the slot call, and to the oracle on a subset --------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["regex1", "three", "mixed_widths", "large_dfa"])
def test_packed_equals_slot_call(which):
    M = 1025
    cfg, _ = _dfa_set(which, M)
    strings = _set_strings(which, M, 300, zlib.crc32(which.encode()))
    data, offs = _pack(strings, lead=3)
    out, sm, pk, _ = _device_pair(cfg, data, offs)
    _vs_slot(pk, sm)
    assert cfg.last_launch_count() == 3                                   # count, scan, pack: one pass
    flagged = _np(out.status)[:, 0] & ((1 << 9) | (1 << 10))
    assert flagged.any()
    for d in range(cfg.n_defs):                                           # a flagged string has an empty list and zero endpoint counts
        rs = _np(pk.row_start[d], np.uint64)
        assert (np.diff(rs.astype(np.int64))[flagged != 0] == 0).all()
        assert not _np(pk.endpoint_counts[d])[flagged != 0].any()
    if which in DEF_SETS:
        sub = 60
        exp = _expected(oracle_config(which, M), data, offs[:sub + 1])
        for j, (dead, mults, eps) in enumerate(exp):
            for d in range(cfg.n_defs):
                if dead:
                    assert pk.row_start[d][j + 1] == pk.row_start[d][j]
                    continue
                assert np.array_equal(pk.dense(j, d), mults[d].astype(np.uint64)), (j, d)
                assert np.array_equal(_np(pk.endpoint_counts[d])[j], eps[d].astype(np.uint32)), (j, d)


# ---- 2. the per-string counts sum to the batch counters --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["regex1", "three"])
def test_packed_sums_to_batch_counters(which):
    cfg = product_config(which, 1025)
    data, offs = _config1_like(1 << 12, 21)
    out, sm, pk, _ = _device_pair(cfg, data, offs)
    assert cfg.batch_result(check=False).code == 0
    for d in range(cfg.n_defs):
        rs = _np(pk.row_start[d], np.uint64)
        e = _np(pk.entries[d])[:int(rs[-1])]
        tot = np.zeros(cfg.table_num_rows[d], np.uint64)
        np.add.at(tot, e[:, 0].astype(np.int64), e[:, 1].astype(np.uint64))
        assert np.array_equal(tot, out.mult[d].cpu().numpy().astype(np.uint64)), d
        assert np.array_equal(_np(pk.endpoint_counts[d]).astype(np.uint64).sum(axis=0), out.endpoint_mult[d].cpu().numpy().astype(np.uint64))
        assert (e[rs[:-1].astype(np.int64), 0] == 0).all()                 # row 0 first in every list


# ---- 3. many passes --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_packed_many_passes():
    M = 1025
    cfg = product_config("three", M)
    strings = _ragged("three", M, 500, 99)
    data, offs = _pack(strings, lead=1)
    _, sm, one, _ = _device_pair(cfg, data, offs)
    assert cfg.last_launch_count() == 3
    cfg.set_option("chunked_max_maps", 100_000)                           # a few strings a pass
    _, sm2, many, _ = _device_pair(cfg, data, offs)
    n = len(strings)
    pitch = max(min(M, t) for t in cfg.table_num_rows)
    per_pass = max(1, 100_000 // (cfg.n_defs * (pitch * 8 + 4)))
    assert per_pass < 20
    assert cfg.last_launch_count() == 3 * -(-n // per_pass)               # count, scan and pack per pass
    _vs_slot(many, sm)
    for d in range(cfg.n_defs):
        assert np.array_equal(_np(one.row_start[d], np.uint64), _np(many.row_start[d], np.uint64))
        assert np.array_equal(_np(one.entries[d]), _np(many.entries[d]))


@pytest.mark.gpu
def test_packed_after_chunked_batch_multi_segment():
    """M = 65537: strings longer than 4096 bytes are counted in segments and compacted; many passes of both workspaces."""
    M = 65537
    rng = random.Random(65537)
    lens = [0, 1, 4095, 4096, 4097, 8192, 8193, M - 1] + [rng.randrange(0, M) for _ in range(28)]
    strings = _strings(rng, M, lens) + [b"a" * M]
    strings[5] = strings[5][:100] + b"\xff" + strings[5][101:]
    data, offs = _pack(strings, lead=7)
    cfg = product_config("three", M)
    _, sm, pk, _ = _device_pair(cfg, data, offs, chunked=True)
    _vs_slot(pk, sm)
    cfg.set_option("chunked_max_maps", 300_000)
    _, _, pk2, _ = _device_pair(cfg, data, offs, chunked=True)
    assert cfg.last_launch_count() > 8
    _vs_slot(pk2, sm)
    exp = _expected(oracle_config("three", M), data, offs[:13])
    for j, (dead, mults, _) in enumerate(exp):
        for d in range(cfg.n_defs):
            assert dead or np.array_equal(pk2.dense(j, d), mults[d].astype(np.uint64)), (j, d)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1024, 4097, 65537])
def test_packed_after_long_string(L):
    import torch
    import halo2_regex_b200 as H
    cfg = product_config("regex1", 1025)
    rng = np.random.default_rng(L)
    s = np.frombuffer(ALPHA, np.uint8)[rng.integers(0, len(ALPHA), size=L)].copy()
    d_bytes = torch.from_numpy(s).cuda() if L else torch.zeros(0, dtype=torch.uint8, device="cuda")
    out = H.DeviceOutputs(cfg, 1, max_chars_size=L + 1, want={"states", "status", "mult", "endpoint_mult"})
    cfg.match_long_device(d_bytes, out)
    d_offs = torch.tensor([0, L], dtype=torch.int64, device="cuda")
    sm = cfg.string_mult_device(d_bytes, d_offs, out, max_chars_size=L + 1)
    pk = cfg.string_mult_packed_device(d_bytes, d_offs, out, max_chars_size=L + 1)
    torch.cuda.synchronize()
    _vs_slot(pk, sm)
    assert np.array_equal(pk.dense(0, 0), out.mult[0].cpu().numpy().astype(np.uint64))


# ---- 4. capacity -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_packed_capacity():
    import halo2_regex_b200 as H
    M = 1025
    cfg = product_config("three", M)
    strings = _ragged("three", M, 120, 5)
    data, offs = _pack(strings)
    n = len(strings)
    _, sm, full, (d_bytes, d_offs) = _device_pair(cfg, data, offs)
    out = H.DeviceOutputs(cfg, n, want={"states", "status"})
    cfg.match_batch_device(d_bytes, d_offs, out)
    rs0 = _np(full.row_start[0], np.uint64).astype(np.int64)
    k = n // 2
    for cap in (0, int(rs0[k]), int(rs0[k]) - 1, int(rs0[-1]), int(rs0[-1]) + 5):
        pk = H.StringMultPacked(cfg, n, capacity=max(cap, 1), fill=FILL)
        s = pk.struct()
        s.capacity = cap
        from halo2_regex_b200._ffi import lib
        import torch
        rc = lib.b2r_string_mult_packed(cfg._h, d_bytes.data_ptr(), d_offs.data_ptr(), n, d_bytes.numel(), 0, C.byref(out.struct()), C.byref(s),
                                        torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        for d in range(cfg.n_defs):
            rs = _np(pk.row_start[d], np.uint64).astype(np.int64)
            assert np.array_equal(rs, _np(full.row_start[d], np.uint64).astype(np.int64)), (cap, d)   # always complete
            e = _np(pk.entries[d])
            stored = rs[1:] <= cap
            assert (np.flatnonzero(~stored) > np.flatnonzero(stored).max(initial=-1)).all()         # a prefix
            top = int(rs[1:][stored].max(initial=0))
            ref = _np(full.entries[d])
            assert np.array_equal(e[:top], ref[:top]), (cap, d)
            assert (e[top:] == FILL_WORD).all(), (cap, d)                 # nothing else written, no list in part
    # entries NULL: offsets only
    pk = H.StringMultPacked(cfg, n, fill=FILL, want=("row_start",))
    cfg.string_mult_packed_device(d_bytes, d_offs, out, pk)
    for d in range(cfg.n_defs):
        assert np.array_equal(_np(pk.row_start[d], np.uint64), _np(full.row_start[d], np.uint64))


# ---- 5. host entry points --------------------------------------------------------------------------------------------------
def _host_vs_plain(cfg, data, offs, chunked=False, sparse=False, reuse_pair=None, want=None, pinned=False, flags=0, capacity=None,
                   slices=None):
    import halo2_regex_b200 as H
    from test_host_chunked import _equal, _res_tuple
    alloc = H.PinnedAllocator() if pinned else None
    n = len(offs) - 1
    kw2 = dict(max_records=8, compact_pitch=64)
    if want:
        kw2["want"] = want
    plain = cfg.match_batch_chunked_host if chunked else cfg.match_batch_host
    packed = cfg.match_batch_chunked_host_mult_packed if chunked else cfg.match_batch_host_mult_packed
    o1 = reuse_pair[0] if reuse_pair else cfg.new_host_outputs(n, fill=FILL, allocator=alloc, **kw2)
    o2 = reuse_pair[1] if reuse_pair else cfg.new_host_outputs(n, fill=FILL, allocator=alloc, **kw2)
    _, r1 = plain(data, offs, out=o1, check=False, sparse=sparse, reuse=bool(reuse_pair), flags=flags)
    b1 = cfg.last_host_bytes()
    pk = H.StringMultPacked(cfg, n, device="cpu", fill=FILL, pin=pinned, capacity=capacity)
    _, pk, r2 = packed(data, offs, out=o2, pk=pk, check=False, sparse=sparse, reuse=bool(reuse_pair), flags=flags)
    b2 = cfg.last_host_bytes()
    _equal(o1, o2)
    assert _res_tuple(r1) == _res_tuple(r2)
    # the device result on the same strings
    _, sm, dev, _ = _device_pair(cfg, data, offs)
    stored_bytes = 0
    for d in range(cfg.n_defs):
        rs = _np(pk.row_start[d], np.uint64)
        assert np.array_equal(rs, _np(dev.row_start[d], np.uint64)), d
        assert np.array_equal(_np(pk.endpoint_counts[d]), _np(dev.endpoint_counts[d])), d
        stored = rs[1:][rs[1:] <= pk.capacity]
        top = int(stored.max(initial=0))
        e = _np(pk.entries[d])
        assert np.array_equal(e[:top], _np(dev.entries[d])[:top]), d
        assert (e[top:] == FILL_WORD).all(), d
        stored_bytes += 8 * top + 8 * n + 8 * n * cfg.endpoint_num_rows[d]
    # nothing goes up for the counts; only the stored entries, row_start and the endpoint counts come back
    assert b2[0] == b1[0] and b2[1] == b1[1] + stored_bytes, (b1, b2, stored_bytes)
    return (o1, o2), pk


@pytest.mark.gpu
@pytest.mark.parametrize("chunked", [False, True])
def test_packed_host_entries(chunked):
    from halo2_regex_b200 import _abi
    M = 1025
    cfg = product_config("three", M)
    strings = _ragged("three", M, 200, 7)
    data, offs = _pack(strings, lead=5)
    few, foffs = _pack(strings[:9], lead=5)
    _host_vs_plain(cfg, few, foffs, chunked=chunked)                                   # small path
    _, pk = _host_vs_plain(cfg, few, foffs, chunked=chunked, capacity=300)               # small path, capacity cut
    cfg.set_option("slices", 3)                                                        # forced slices (chunked path)
    _, pk = _host_vs_plain(cfg, data, offs, chunked=chunked)
    rs = _np(pk.row_start[0], np.uint64).astype(np.int64)
    for cap in (int(rs[120]), int(rs[120]) - 1, int(rs[40]), 0):                        # capacity cuts in later slices
        _host_vs_plain(cfg, data, offs, chunked=chunked, capacity=cap)
    cfg.set_option("small_path", 0)
    _host_vs_plain(cfg, few, foffs, chunked=chunked, pinned=True)
    pair, _ = _host_vs_plain(cfg, data, offs, chunked=chunked, sparse=True, pinned=True)
    _host_vs_plain(cfg, data, offs, chunked=chunked, sparse=True, reuse_pair=pair)
    _host_vs_plain(cfg, data, offs, chunked=chunked, flags=_abi.B2R_OUT_ACCUMULATE_MULT, pinned=True)
    cfg.set_option("slices", 0)
    _host_vs_plain(cfg, data, offs, chunked=chunked, want={"substr_ids", "masked_chars", "mult"})   # no states, no status


@pytest.mark.gpu
def test_packed_host_entry_many_slices():
    """2^15 strings: b2r_match_batch_host cuts 8 slices by count; the slice bases cross every boundary."""
    cfg = product_config("regex1", 1025)
    data, offs = _config1_like(1 << 15, 3)
    _, pk = _host_vs_plain(cfg, data, offs, pinned=True)
    rs = _np(pk.row_start[0], np.uint64).astype(np.int64)
    _host_vs_plain(cfg, data, offs, capacity=int(rs[(1 << 15) * 5 // 8 + 3]), sparse=True,
                   want={"states", "substr_ids", "status", "mult", "endpoint_mult"})


# ---- 6. the device entry on a multi-device handle --------------------------------------------------------------------------
@pytest.mark.gpu
def test_packed_device_entry_rejects_a_multi_device_handle():
    import os
    import halo2_regex_b200 as H
    from halo2_regex_b200 import _abi
    from halo2_regex_b200._ffi import last_error, lib
    from conftest import DEFS
    a, ss = DEF_SETS["regex1"][0]
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(os.path.join(DEFS, a)), [H.SubstrRegexDef.read_from_text(os.path.join(DEFS, x)) for x in ss])]
    try:
        mcfg = H.RegexVerifyConfig.configure(1025, defs, devices=[0])
    except RuntimeError as e:
        pytest.skip(f"multi-device handle unavailable: {e}")
    rc = lib.b2r_string_mult_packed(mcfg._h, None, None, 0, 0, 0, C.byref(_dev_out(mcfg)), C.byref(_pk_struct(mcfg)), None)
    assert rc == _abi.B2R_ERR_INVALID_ARG
    assert "multi-device" in last_error()


# ---- 7. CUDA graph capture -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_packed_cuda_graph():
    import torch
    import halo2_regex_b200 as H
    M = 1025
    cfg = product_config("three", M)
    strings = _ragged("three", M, 150, 17)
    data, offs = _pack(strings)
    n = len(strings)
    cfg.set_option("chunked_max_maps", 400_000)                           # several passes inside the graph
    _, sm, ref, (d_bytes, d_offs) = _device_pair(cfg, data, offs)
    out = H.DeviceOutputs(cfg, n, want={"states", "status"})
    cfg.match_batch_device(d_bytes, d_offs, out)
    pk = H.StringMultPacked(cfg, n, fill=FILL)
    cfg.string_mult_packed_device(d_bytes, d_offs, out, pk)               # sizes the workspace
    torch.cuda.synchronize()
    for d in range(cfg.n_defs):                                           # what the replays must write again
        pk.row_start[d].view(torch.uint8).fill_(FILL)
        pk.entries[d].view(torch.uint8).fill_(FILL)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cfg.string_mult_packed_device(d_bytes, d_offs, out, pk)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        _vs_slot(pk, sm)
        for d in range(cfg.n_defs):
            assert np.array_equal(_np(pk.entries[d]), _np(ref.entries[d]))


# ---- 8. multi-device handle ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_dev", [2, 4])
@pytest.mark.parametrize("chunked", [False, True])
def test_packed_multi_device(n_dev, chunked):
    import os
    import torch
    import halo2_regex_b200 as H
    if torch.cuda.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    from conftest import DEFS
    M = 1025
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(os.path.join(DEFS, a)), [H.SubstrRegexDef.read_from_text(os.path.join(DEFS, s)) for s in ss])
            for a, ss in DEF_SETS["three"]]
    try:
        mcfg = H.RegexVerifyConfig.configure(M, defs, devices=list(range(n_dev)))
    except RuntimeError as e:
        pytest.skip(f"multi-device handle unavailable: {e}")
    cfg = product_config("three", M)
    strings = _ragged("three", M, 300, n_dev)
    data, offs = _pack(strings)
    _, pk, _ = (mcfg.match_batch_chunked_host_mult_packed if chunked else mcfg.match_batch_host_mult_packed)(data, offs, check=False)
    _, pk1, _ = (cfg.match_batch_chunked_host_mult_packed if chunked else cfg.match_batch_host_mult_packed)(data, offs, check=False)
    rs = _np(pk1.row_start[1], np.uint64).astype(np.int64)
    _, pkc, _ = (mcfg.match_batch_chunked_host_mult_packed if chunked else mcfg.match_batch_host_mult_packed)(
        data, offs, check=False, pk=H.StringMultPacked(mcfg, len(strings), device="cpu", fill=FILL, capacity=int(rs[200]) - 1))
    for d in range(cfg.n_defs):
        assert np.array_equal(_np(pk.row_start[d], np.uint64), _np(pk1.row_start[d], np.uint64)), d
        assert np.array_equal(_np(pk.entries[d]), _np(pk1.entries[d])), d
        assert np.array_equal(_np(pk.endpoint_counts[d]), _np(pk1.endpoint_counts[d])), d
        assert np.array_equal(_np(pkc.row_start[d], np.uint64), _np(pk1.row_start[d], np.uint64)), d
        r = _np(pk1.row_start[d], np.uint64).astype(np.int64)
        top = int(r[1:][r[1:] <= pkc.capacity].max(initial=0))
        e = _np(pkc.entries[d])
        assert np.array_equal(e[:top], _np(pk1.entries[d])[:top]) and (e[top:] == FILL_WORD).all(), d
