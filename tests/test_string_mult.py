"""Per-string lookup multiplicities: b2r_string_mult (device post-pass) and b2r_match_batch_host_mult /
b2r_match_batch_chunked_host_mult.  The contract (include/b2r.h): the counts of string j equal the mult / endpoint_mult of a
one-string batch of string j with the same M; flagged strings count nothing and keep their entry slots; the sum over the
strings of a call equals the batch counters of that call.  Expected per-string counts come from one-string oracle batches."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, product_config
from test_batch_chunked import ALPHA, _example, _strings, _to_device
from test_dfa_shapes import _oracle, _product, make_dfa
from test_gpu_parity import _pack
from test_oracle_golden import SNIPPETS

FILL = 0x5A
FILL_WORD = 0x5A5A5A5A
DEAD = (1 << 9) | (1 << 10)          # B2R_ST_INVALID_TRANSITION | B2R_ST_TOO_LONG


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_struct_layout():
    from halo2_regex_b200 import _abi
    assert C.sizeof(_abi.RowCount) == 8
    assert (_abi.RowCount.row.offset, _abi.RowCount.count.offset) == (0, 4)
    S = _abi.StringMultStruct
    assert C.sizeof(S) == 8 + 3 * 4 * 8
    assert (S.max_entries.offset, S.reserved.offset, S.entries.offset, S.n_entries.offset, S.endpoint_counts.offset) == (0, 4, 8, 40, 72)


def test_symbols_exported():
    import subprocess
    import halo2_regex_b200 as H
    out = subprocess.check_output(["nm", "-D", H.LIB_PATH]).decode()
    for name in ("b2r_string_mult", "b2r_match_batch_host_mult", "b2r_match_batch_chunked_host_mult"):
        assert f" T {name}\n" in out


def _sm_struct(cfg, entries=True, n_entries=True, ep=True, max_entries=4, base=0x10000):
    from halo2_regex_b200 import _abi
    s = _abi.StringMultStruct()
    s.max_entries = max_entries
    for d in range(cfg.n_defs):
        s.entries[d] = base + 0x1000 * d if entries else None
        s.n_entries[d] = base + 0x100000 + 0x1000 * d if n_entries else None
        s.endpoint_counts[d] = base + 0x200000 + 0x1000 * d if ep else None
    return s


def _calls(cfg, out, sm):
    from halo2_regex_b200._ffi import lib
    data = np.zeros(16, np.uint8)
    offs = np.array([0, 3], np.uint64)
    res = __import__("halo2_regex_b200")._abi.BatchStatus()
    return [lib.b2r_string_mult(cfg._h, 0x1000, 0x2000, 1, 3, 0, C.byref(out), C.byref(sm), None),
            lib.b2r_match_batch_host_mult(cfg._h, data.ctypes.data, offs.ctypes.data, 1, C.byref(out), C.byref(sm), C.byref(res)),
            lib.b2r_match_batch_chunked_host_mult(cfg._h, data.ctypes.data, offs.ctypes.data, 1, C.byref(out), C.byref(sm), C.byref(res))]


def _dev_out(cfg, states=True, status=True):
    from halo2_regex_b200 import _abi
    o = _abi.Outputs()
    o.row_pitch = 1056 if cfg.max_chars_size == 1025 else 64
    o.bitmap_pitch = 160
    for d in range(cfg.n_defs):
        o.states[d] = 0x400000 + 0x10000 * d if states else None
    o.status = 0x800000 if status else None
    return o


def test_deviceless_handle_and_argument_errors():
    from halo2_regex_b200 import _abi
    cfg = product_config("three", 1025, device=-1)
    ok = _sm_struct(cfg)
    assert _calls(cfg, _dev_out(cfg), ok) == [_abi.B2R_ERR_CUDA] * 3
    # entries without n_entries; entries with max_entries 0
    assert _calls(cfg, _dev_out(cfg), _sm_struct(cfg, n_entries=False)) == [_abi.B2R_ERR_INVALID_ARG] * 3
    assert _calls(cfg, _dev_out(cfg), _sm_struct(cfg, max_entries=0)) == [_abi.B2R_ERR_INVALID_ARG] * 3
    # max_entries 0 is fine without entries
    assert _calls(cfg, _dev_out(cfg), _sm_struct(cfg, entries=False, max_entries=0)) == [_abi.B2R_ERR_CUDA] * 3
    # the device entry reads the state columns and the status; the host entries use scratch ones
    assert _calls(cfg, _dev_out(cfg, states=False), ok) == [_abi.B2R_ERR_INVALID_ARG, _abi.B2R_ERR_CUDA, _abi.B2R_ERR_CUDA]
    assert _calls(cfg, _dev_out(cfg, status=False), ok) == [_abi.B2R_ERR_INVALID_ARG, _abi.B2R_ERR_CUDA, _abi.B2R_ERR_CUDA]
    # nothing asked for: no state column needed
    assert _calls(cfg, _dev_out(cfg, states=False, status=False), _sm_struct(cfg, False, False, False))[0] == _abi.B2R_ERR_CUDA
    # alignment
    for kw, off in ((dict(base=0x10004), 4), (dict(base=0x10002), 2)):
        assert _calls(cfg, _dev_out(cfg), _sm_struct(cfg, **kw)) == [_abi.B2R_ERR_ALIGNMENT] * 3, off
    s = _sm_struct(cfg)
    s.endpoint_counts[1] = 0x30002
    assert _calls(cfg, _dev_out(cfg), s) == [_abi.B2R_ERR_ALIGNMENT] * 3
    # null outputs
    from halo2_regex_b200._ffi import lib
    assert lib.b2r_string_mult(cfg._h, None, None, 0, 0, 0, None, C.byref(ok), None) == _abi.B2R_ERR_INVALID_ARG
    assert lib.b2r_string_mult(None, None, None, 0, 0, 0, None, None, None) == _abi.B2R_ERR_INVALID_ARG


def test_dense_and_holder_on_host():
    import halo2_regex_b200 as H
    cfg = product_config("regex1", 1025, device=-1)
    sm = H.StringMultOutputs(cfg, 2, device="cpu")
    assert sm.max_entries == min(1025, cfg.table_num_rows[0])
    sm.n_entries[0][0] = 3
    sm.entries[0][0, :3] = __import__("torch").tensor([[0, 1000], [5, 20], [7, 5]], dtype=__import__("torch").int32)
    v = sm.dense(0, 0)
    assert len(v) == cfg.table_num_rows[0] and v[0] == 1000 and v[5] == 20 and v[7] == 5 and v.sum() == 1025


# ---- helpers of the GPU cases ----------------------------------------------------------------------------------------------
def _expected(ocfg, data, offs):
    """Per string: (flagged, [mult per def], [endpoint_mult per def]) of a one-string oracle batch."""
    exp = []
    for j in range(len(offs) - 1):
        a, b = int(offs[j]), int(offs[j + 1])
        o, _ = ocfg.match_batch(np.ascontiguousarray(data[a:b]), np.array([0, b - a], np.uint64), want={"status", "mult", "endpoint_mult"})
        exp.append((bool(o.status["flags"][0] & DEAD), [m.copy() for m in o.mult], [e.copy() for e in o.endpoint_mult]))
    return exp


def _host(sm):
    h = sm.to_host()
    return ([None if t is None else t.numpy().view(np.uint32) for t in h.entries], [None if t is None else t.numpy().view(np.uint32) for t in h.n_entries],
            [None if t is None else t.numpy().view(np.uint32) for t in h.endpoint_counts], h.max_entries)


def _check(sm, exp, filled=True):
    ent, nent, epc, maxe = _host(sm)
    for j, (dead, mults, eps) in enumerate(exp):
        for d in range(len(mults)):
            if dead:
                assert nent[d][j] == 0, (j, d)
                assert not epc[d][j].any(), (j, d)
                if filled:
                    assert (ent[d][j] == FILL_WORD).all(), (j, d)
                continue
            rows = np.flatnonzero(mults[d])
            assert nent[d][j] == len(rows), (j, d, nent[d][j], len(rows))
            k = min(len(rows), maxe)
            got = ent[d][j, :k]
            assert np.array_equal(got[:, 0], rows[:k]), (j, d)
            assert np.array_equal(got[:, 1], mults[d][rows[:k]].astype(np.uint32)), (j, d)
            if filled:
                assert (ent[d][j, k:] == FILL_WORD).all(), (j, d)
            assert np.array_equal(epc[d][j], eps[d].astype(np.uint32)), (j, d)


def _sums(sm, d):
    """(sum over strings of the dense counts, sum over strings of the endpoint counts, per-string sums of the counts)"""
    ent, nent, epc, maxe = _host(sm)
    n = len(nent[d])
    k = np.arange(maxe)[None, :] < np.minimum(nent[d], maxe)[:, None]
    rows, cnt = ent[d][..., 0], ent[d][..., 1]
    tot = np.zeros(sm.cfg.table_num_rows[d], np.uint64)
    np.add.at(tot, rows[k].astype(np.int64), cnt[k].astype(np.uint64))
    per = np.where(k, cnt, 0).astype(np.uint64).sum(axis=1)
    assert len(per) == n
    return tot, epc[d].astype(np.uint64).sum(axis=0), per


def _device_run(cfg, data, offs, chunked=False, want=("states", "status"), **smkw):
    import halo2_regex_b200 as H
    d_bytes, d_offs = _to_device(data, offs)
    n = len(offs) - 1
    out = H.DeviceOutputs(cfg, n, want=set(want) | {"mult", "endpoint_mult"})
    (cfg.match_batch_chunked_device if chunked else cfg.match_batch_device)(d_bytes, d_offs, out)
    sm = H.StringMultOutputs(cfg, n, fill=FILL, **smkw)
    cfg.string_mult_device(d_bytes, d_offs, out, sm)
    __import__("torch").cuda.synchronize()
    return out, sm


def _ragged(set_name, M, n, seed):
    rng = random.Random(seed)
    lens = [0, 0, 1, M - 1, M - 1] + [rng.randrange(0, M) for _ in range(n - 5)]
    strings = [_example(L) for L in lens] if set_name == "example" else _strings(rng, M, lens)
    for k in range(0, len(strings), 23):                                 # invalid transitions
        s = bytearray(strings[k])
        if s:
            s[rng.randrange(len(s))] = 0xFF
        strings[k] = bytes(s)
    strings += [b"a" * M, b"ab" * M]                                     # too long
    rng.shuffle(strings)
    return strings


# ---- 2. oracle parity ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("set_name", list(DEF_SETS))
def test_oracle_parity(set_name):
    M = 1025
    cfg, ocfg = product_config(set_name, M), oracle_config(set_name, M)
    strings = _ragged(set_name, M, 300, zlib.crc32(set_name.encode()))
    data, offs = _pack(strings, lead=3)
    out, sm = _device_run(cfg, data, offs)
    exp = _expected(ocfg, data, offs)
    assert any(e[0] for e in exp)
    _check(sm, exp)
    assert cfg.last_launch_count() == 1


# ---- 3. batch consistency -------------------------------------------------------------------------------------------------
def _config1_like(n, seed):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(ALPHA, np.uint8)
    rows = alpha[rng.integers(0, len(alpha), size=(n, 1024))]
    for k in range(0, n, 3):
        sn = np.frombuffer(SNIPPETS[k % len(SNIPPETS)], np.uint8)
        at = int(rng.integers(0, 1024 - len(sn)))
        rows[k, at:at + len(sn)] = sn
    lens = rng.integers(0, 1025, size=n)
    lens[:8] = 1024
    data = rows.reshape(-1)
    offs = np.zeros(n + 1, np.uint64)
    offs[1:] = np.cumsum(lens)
    packed = np.concatenate([rows[j, :lens[j]] for j in range(n)]) if n else data[:0]
    return packed, offs


def _consistency(cfg, data, offs, chunked=False):
    out, sm = _device_run(cfg, data, offs, chunked=chunked)
    res = cfg.batch_result(check=False)
    assert res.code == 0
    M = cfg.max_chars_size
    for d in range(cfg.n_defs):
        tot, ep, per = _sums(sm, d)
        assert np.array_equal(tot, out.mult[d].cpu().numpy().astype(np.uint64)), d
        assert np.array_equal(ep, out.endpoint_mult[d].cpu().numpy().astype(np.uint64)), d
        assert (per == M).all(), d
        E = cfg.endpoint_num_rows[d]
        epc = sm.endpoint_counts[d].cpu().numpy().view(np.uint32).astype(np.uint64)
        assert (epc[:, :E].sum(axis=1) == M).all() and (epc[:, E:].sum(axis=1) == M).all()
    return out, sm


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["regex1", "three", "large_dfa", "mixed_widths"])
def test_batch_consistency_2_15_x_1k(which):
    import halo2_regex_b200 as H
    from halo2_regex_b200 import workloads as W
    n, M = 1 << 15, 1025
    if which in ("regex1", "three"):
        cfg = product_config(which, M)
        data, offs = _config1_like(n, 15)
    elif which == "large_dfa":
        allstr, substr, _ = W.large_dfa_texts()
        cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
        rows, _ = W.config4_numpy(n, 1024)
        data, offs = rows.reshape(-1), np.arange(n + 1, dtype=np.uint64) * 1024
    else:
        dfas = [make_dfa(300, 4, 0, 7, "perm", seed=3, alphabet=b"xyz."), make_dfa(40, 3, 1, 5, "collapse_2", seed=4, alphabet=b"xyz.")]
        cfg = _product(dfas, M)
        rng = np.random.default_rng(7)
        data = np.frombuffer(b"xyz.", np.uint8)[rng.integers(0, 4, size=n * 1024)]
        offs = np.arange(n + 1, dtype=np.uint64) * 1024
        assert cfg.state_widths == [2, 2] and cfg.dummy_states[1] <= 255
    _consistency(cfg, data, offs)


# ---- 4. truncation ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_truncation():
    M = 1025
    cfg, ocfg = product_config("three", M), oracle_config("three", M)
    strings = _ragged("three", M, 80, 44)
    data, offs = _pack(strings)
    _, full = _device_run(cfg, data, offs)
    _, cut = _device_run(cfg, data, offs, max_entries=4)
    ef, nf, pf, _ = _host(full)
    ec, nc, pc, _ = _host(cut)
    for d in range(cfg.n_defs):
        assert np.array_equal(nf[d], nc[d]) and np.array_equal(pf[d], pc[d])
        for j in range(len(nf[d])):
            k = min(int(nf[d][j]), 4)
            assert np.array_equal(ec[d][j, :k], ef[d][j, :k])
            assert (ec[d][j, k:] == FILL_WORD).all()
    _check(cut, _expected(ocfg, data, offs))


# ---- 5. the other device paths ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_after_chunked_batch_several_passes():
    M = 65537
    rng = random.Random(65537)
    lens = [0, 1, 4095, 4096, 4097, 8192, 8193, M - 1] + [rng.randrange(0, M) for _ in range(28)]
    strings = _strings(rng, M, lens)
    strings[5] = strings[5][:100] + b"\xff" + strings[5][101:]
    data, offs = _pack(strings, lead=7)
    cfg = product_config("three", M)
    _, a = _device_run(cfg, data, offs)
    cfg.set_option("chunked_max_maps", 300_000)       # several passes of the chunked walk and of the per-string counters
    _, b = _device_run(cfg, data, offs, chunked=True)
    assert cfg.last_launch_count() > 2
    for x, y in zip(_host(a)[:3], _host(b)[:3]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    _check(b, _expected(oracle_config("three", M), data, offs))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1, 1023, 1024, 1025, 4095, 4096, 4097, 65537, 262145, 16 << 20])
def test_after_long_string(L):
    import torch
    import halo2_regex_b200 as H
    cfg = product_config("regex1", 1025)
    rng = np.random.default_rng(L)
    s = np.frombuffer(ALPHA, np.uint8)[rng.integers(0, len(ALPHA), size=L)].copy()
    for k, at in enumerate(range(0, max(0, L - 64), max(64, L // 50))):
        sn = np.frombuffer(SNIPPETS[k % len(SNIPPETS)], np.uint8)
        s[at:at + len(sn)] = sn
    d_bytes = torch.from_numpy(s).cuda() if L else torch.zeros(0, dtype=torch.uint8, device="cuda")
    out = H.DeviceOutputs(cfg, 1, max_chars_size=L + 1, want={"states", "status", "mult", "endpoint_mult"})
    cfg.match_long_device(d_bytes, out)
    d_offs = torch.tensor([0, L], dtype=torch.int64, device="cuda")
    sm = cfg.string_mult_device(d_bytes, d_offs, out, max_chars_size=L + 1)
    torch.cuda.synchronize()
    assert cfg.batch_result(check=False).code == 0
    assert np.array_equal(sm.dense(0, 0), out.mult[0].cpu().numpy().astype(np.uint64))
    assert np.array_equal(sm.endpoint_counts[0][0].cpu().numpy().view(np.uint32), out.endpoint_mult[0].cpu().numpy().astype(np.uint32))


# ---- 6. host entries -------------------------------------------------------------------------------------------------------
def _host_vs_plain(cfg, data, offs, chunked=False, sparse=False, reuse_pair=None, want=None, pinned=False, **kw):
    import halo2_regex_b200 as H
    from test_host_chunked import _equal, _res_tuple
    alloc = H.PinnedAllocator() if pinned else None
    n = len(offs) - 1
    kw2 = dict(max_records=8, compact_pitch=64)
    if want:
        kw2["want"] = want
    plain = (cfg.match_batch_chunked_host if chunked else cfg.match_batch_host)
    mult = (cfg.match_batch_chunked_host_mult if chunked else cfg.match_batch_host_mult)
    o1 = reuse_pair[0] if reuse_pair else cfg.new_host_outputs(n, fill=FILL, allocator=alloc, **kw2)
    o2 = reuse_pair[1] if reuse_pair else cfg.new_host_outputs(n, fill=FILL, allocator=alloc, **kw2)
    _, r1 = plain(data, offs, out=o1, check=False, sparse=sparse, reuse=bool(reuse_pair))
    sm = H.StringMultOutputs(cfg, n, device="cpu", fill=FILL, pin=pinned)
    _, sm, r2 = mult(data, offs, out=o2, sm=sm, check=False, sparse=sparse, reuse=bool(reuse_pair))
    _equal(o1, o2)
    assert _res_tuple(r1) == _res_tuple(r2)
    _, dev = _device_run(cfg, data, offs)
    for x, y in zip(_host(sm)[:3], _host(dev)[:3]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    return (o1, o2), sm


@pytest.mark.gpu
@pytest.mark.parametrize("chunked", [False, True])
def test_host_entries(chunked):
    M = 1025
    cfg, ocfg = product_config("three", M), oracle_config("three", M)
    strings = _ragged("three", M, 200, 7)
    data, offs = _pack(strings, lead=5)
    few, foffs = _pack(strings[:9], lead=5)
    _, sm = _host_vs_plain(cfg, few, foffs, chunked=chunked)                     # small path
    _check(sm, _expected(ocfg, few, foffs))
    cfg.set_option("slices", 3)                                                   # forced slices (chunked path)
    _, sm = _host_vs_plain(cfg, data, offs, chunked=chunked)
    _check(sm, _expected(ocfg, data, offs))
    cfg.set_option("small_path", 0)
    _host_vs_plain(cfg, few, foffs, chunked=chunked, pinned=True)
    pair, _ = _host_vs_plain(cfg, data, offs, chunked=chunked, sparse=True, pinned=True)
    _host_vs_plain(cfg, data, offs, chunked=chunked, sparse=True, reuse_pair=pair)
    cfg.set_option("slices", 0)
    _host_vs_plain(cfg, data, offs, chunked=chunked, want={"substr_ids", "masked_chars", "mult"})   # no states, no status


@pytest.mark.gpu
def test_host_entry_many_slices():
    """2^15 strings: b2r_match_batch_host cuts 8 slices by count."""
    cfg = product_config("regex1", 1025)
    data, offs = _config1_like(1 << 15, 3)
    _host_vs_plain(cfg, data, offs, pinned=True)
    _host_vs_plain(cfg, data, offs, sparse=True, want={"states", "substr_ids", "status", "mult", "endpoint_mult"})


@pytest.mark.gpu
@pytest.mark.parametrize("n_dev", [2, 4])
@pytest.mark.parametrize("chunked", [False, True])
def test_multi_device(n_dev, chunked):
    import torch
    import halo2_regex_b200 as H
    if torch.cuda.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    import os
    from conftest import DEFS
    M = 1025
    spec = DEF_SETS["three"]
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(os.path.join(DEFS, a)), [H.SubstrRegexDef.read_from_text(os.path.join(DEFS, s)) for s in ss])
            for a, ss in spec]
    try:
        mcfg = H.RegexVerifyConfig.configure(M, defs, devices=list(range(n_dev)))
    except RuntimeError as e:
        pytest.skip(f"multi-device handle unavailable: {e}")
    strings = _ragged("three", M, 300, n_dev)
    data, offs = _pack(strings)
    _, sm, _ = (mcfg.match_batch_chunked_host_mult if chunked else mcfg.match_batch_host_mult)(data, offs, check=False)
    _check(sm, _expected(oracle_config("three", M), data, offs), filled=False)


# ---- 7. a post-pass given a smaller M than the match used ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which,L", [("regex1", 1500), ("regex1", 5000), ("regex1", 9000), ("large_dfa", 8192)])
def test_post_pass_m_below_the_match(which, L):
    """After b2r_match_long of a string longer than the handle's M - 1, a post-pass left at the handle's M (max_chars_size 0)
    counts nothing for it (n_entries 0, zero endpoint counts, slots untouched), like the match's own too-long rule; the same
    columns with M = len + 1 then give the counts of the call."""
    import torch
    import halo2_regex_b200 as H
    from halo2_regex_b200 import workloads as W
    if which == "large_dfa":
        allstr, substr, _ = W.large_dfa_texts()
        cfg = H.RegexVerifyConfig.configure(1025, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
        rows, _ = W.config4_numpy(1, L)
        s = np.ascontiguousarray(rows.reshape(-1)[:L])
    else:
        cfg = product_config(which, 1025)
        rng = np.random.default_rng(L)
        s = np.frombuffer(ALPHA, np.uint8)[rng.integers(0, len(ALPHA), size=L)].copy()
    d_bytes = torch.from_numpy(s).cuda()
    out = H.DeviceOutputs(cfg, 1, max_chars_size=L + 1, want={"states", "status", "mult", "endpoint_mult"})
    cfg.match_long_device(d_bytes, out)
    d_offs = torch.tensor([0, L], dtype=torch.int64, device="cuda")
    sm = H.StringMultOutputs(cfg, 1, fill=FILL, max_chars_size=L + 1)
    cfg.string_mult_device(d_bytes, d_offs, out, sm)                              # M = the handle's 1025
    torch.cuda.synchronize()
    assert cfg.batch_result(check=False).code == 0
    ent, nent, epc, _ = _host(sm)
    assert nent[0][0] == 0 and not epc[0][0].any() and (ent[0][0] == FILL_WORD).all()
    sm = cfg.string_mult_device(d_bytes, d_offs, out, max_chars_size=L + 1)
    torch.cuda.synchronize()
    assert np.array_equal(sm.dense(0, 0), out.mult[0].cpu().numpy().astype(np.uint64))


@pytest.mark.gpu
def test_post_pass_m_below_the_batch_m():
    """A batch matched at M = 4097, counted with max_chars_size 1025: the strings longer than 1024 count nothing, the others
    have the counts of a one-string batch at M = 1025."""
    rng = random.Random(4097)
    lens = [0, 1, 1023, 1024, 1025, 2000, 4095, 4096] + [rng.randrange(0, 4097) for _ in range(40)]
    strings = _strings(rng, 4097, lens)
    data, offs = _pack(strings, lead=2)
    cfg = product_config("three", 4097)
    import halo2_regex_b200 as H
    d_bytes, d_offs = _to_device(data, offs)
    out = H.DeviceOutputs(cfg, len(strings), want={"states", "status"})
    cfg.match_batch_device(d_bytes, d_offs, out)
    sm = H.StringMultOutputs(cfg, len(strings), fill=FILL, max_chars_size=1025, max_entries=1025)
    cfg.string_mult_device(d_bytes, d_offs, out, sm, max_chars_size=1025)
    __import__("torch").cuda.synchronize()
    exp = _expected(oracle_config("three", 1025), data, offs)
    assert sum(e[0] for e in exp) >= 3
    _check(sm, exp)


@pytest.mark.gpu
def test_device_entry_rejects_a_multi_device_handle():
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
    rc = lib.b2r_string_mult(mcfg._h, None, None, 0, 0, 0, C.byref(_dev_out(mcfg)), C.byref(_sm_struct(mcfg)), None)
    assert rc == _abi.B2R_ERR_INVALID_ARG
    assert "multi-device" in last_error()
