"""GPU (-m gpu): b2r_match_batch_chunked_host, the host-buffer entry point with the kernels of b2r_match_batch_chunked.  Its
contract is that it writes exactly what b2r_match_batch_host writes for the same call, so every case runs both on the same
handle and inputs, into host buffers pre-filled with the same pattern, and compares every column whole, the status, records,
compact bytes, both counter arrays and the b2r_batch_status fields.  Small cases are also compared with the CPU oracle.  Every
chunked call is checked against the launch count its slices imply (`_expected_launches`), which proves how the batch was cut."""
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, product_config
from test_batch_chunked import _chunked_launches, _example, _lengths, _strings
from test_dfa_shapes import _first_and_accepted, _max_smem, _oracle, _product, make_dfa
from test_gpu_parity import _pack

pytestmark = pytest.mark.gpu

MAX_SLICES = 16                                                       # b2r_config::MAX_SLICES (csrc/config.hpp)


# ---- helpers ------------------------------------------------------------------------------------------------------------------
def _cuts(offs, slices=0):
    """Slice boundaries of the chunked pipeline (csrc/host.cu, host_batch): balanced by bytes, multiples of 4 strings, no empty
    slice; by default at least 8 MiB and 32 strings per slice, at most 16 slices; `slices` = the forced count."""
    offs = np.asarray(offs, dtype=np.uint64)
    n = len(offs) - 1
    base, nbytes = int(offs[0]), int(offs[n]) - int(offs[0])
    k = slices if 1 <= slices <= MAX_SLICES else max(1, min(MAX_SLICES, nbytes >> 23, n // 32))
    cuts = [0]
    for i in range(1, k):
        target = base + nbytes // k * i + nbytes % k * i // k
        j = int(np.searchsorted(offs, np.uint64(target), side="left"))
        cuts.append(max(cuts[-1], min(n, (j + 2) & ~3)))
    cuts.append(n)
    cuts = sorted(set(cuts))
    return cuts if len(cuts) > 1 else [0, n]


def _n_sparse_cols(cfg, want):
    per_def = sum(1 for c in ("substr_ids", "start_enable", "end_enable") if c in want)
    return cfg.n_defs * per_def + sum(1 for c in ("masked_chars", "masked_substr_ids") if c in want)


def _small(cfg, offs, out):
    """The one-copy path of host_batch_small: n <= 32 within its byte limit."""
    n = len(offs) - 1
    nbytes = int(offs[-1]) - int(offs[0])
    D = cfg.n_defs
    return 1 <= n <= 32 and n * (out.row_pitch * (4 + 3 * D) + 2 * out.bitmap_pitch * D) + nbytes <= 8 << 20


def _expected_launches(cfg, offs, out, sparse=False, slices=0, small_path=True):
    """Kernel launches of one b2r_match_batch_chunked_host call: the chunked kernels of every slice (finalize always runs: it
    leaves the slice's counters in pinned memory), plus in sparse mode one compaction per non-empty slice and sparse column and
    one count publication per slice."""
    M, max_smem = cfg.max_chars_size, _max_smem()
    if small_path and _small(cfg, offs, out):
        return _chunked_launches(cfg, len(offs) - 1, M, max_smem)
    cuts = _cuts(offs, slices)
    total = sum(_chunked_launches(cfg, hi - lo, M, max_smem) for lo, hi in zip(cuts, cuts[1:]))
    n_sc = _n_sparse_cols(cfg, out.want)
    if sparse and len(offs) > 1 and n_sc:
        total += sum(n_sc for lo, hi in zip(cuts, cuts[1:]) if hi > lo) + (len(cuts) - 1)
    return total


def _res_tuple(r):
    return (r.code, r.string_idx, r.pos, r.state, r.byte, r.defidx, r.n_overlap_lo)


def _equal(a, b):
    for x, y in zip(a.all_arrays(), b.all_arrays()):
        xb, yb = x.reshape(-1).view(np.uint8), y.reshape(-1).view(np.uint8)
        if not np.array_equal(xb, yb):
            bad = np.flatnonzero(xb != yb)
            raise AssertionError(f"array of shape {x.shape} differs at bytes {bad[:4].tolist()} ({len(bad)} bytes)")


def _both(cfg, data, offs, outs=None, fill=0x5A, flags=0, sparse=False, reuse=False, slices=0, small_path=True, launches=True, **kw):
    """b2r_match_batch_host, then b2r_match_batch_chunked_host, same handle and inputs, into outputs pre-filled with one
    pattern (or into `outs`, a pair); everything equal.  Returns (chunked outputs, its result, host outputs)."""
    res, got = [], []
    for i, fn in enumerate((cfg.match_batch_host, cfg.match_batch_chunked_host)):
        out = outs[i] if outs else cfg.new_host_outputs(len(offs) - 1, fill=fill, **kw)
        o, r = fn(data, offs, out=out, flags=flags, check=False, sparse=sparse, reuse=reuse)
        got.append(o)
        res.append(r)
        if i == 0:
            h2d_host = cfg.last_host_bytes()[0]
    if launches:
        exp = _expected_launches(cfg, offs, got[1], sparse=sparse, slices=slices, small_path=small_path)
        assert cfg.last_launch_count() == exp, (cfg.last_launch_count(), exp)
    assert cfg.last_host_bytes()[0] == h2d_host                          # the same bytes went up
    cfg.last_plan()
    _equal(got[0], got[1])
    assert _res_tuple(res[0]) == _res_tuple(res[1])
    return got[1], res[1], got[0]


def _vs_oracle(out, res, ocfg, data, offs, **kw):
    import halo2_regex_b200 as H
    o, ores = ocfg.match_batch(data, offs, **kw)
    assert res.code == ores.code
    if ores.code != 0:
        assert (res.string_idx, res.pos, res.state, res.byte, res.defidx) == (ores.string_idx, ores.pos, ores.state, ores.byte, ores.defidx)
    assert res.n_overlap_lo == ores.n_overlap_lo
    errs = H.compare_outputs(out, o)
    assert errs == [], "\n".join(errs[:10])


def _forced(cfg, slices, small_path=1):
    cfg.set_option("slices", slices)
    cfg.set_option("small_path", small_path)


# ---- 1. every def set at slot-edge lengths, sliced, unaligned base ---------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 1025, 4097, 65537])
@pytest.mark.parametrize("set_name", list(DEF_SETS))
def test_def_sets_and_lengths(set_name, M):
    """Ragged lengths (0, M-1, around 1024 k, random), snippets across slot edges, a base offset that is not 16-byte aligned;
    37 strings in three forced slices, then the same strings through the one-copy small path."""
    rng = random.Random(zlib.crc32(f"host/{set_name}/{M}".encode()))
    cfg, ocfg = product_config(set_name, M), oracle_config(set_name, M)
    lens = _lengths(rng, M, n_random=0)
    lens += [min(M - 1, max(0, 1024 * k + d)) for k in (1, 2, 3) for d in (-1, 0, 1)]
    lens += [rng.randrange(0, M) for _ in range(37 - len(lens))]
    rng.shuffle(lens)
    if set_name == "example":
        strings = [_example(L) for L in lens]
    else:
        strings = _strings(rng, M, lens)
    data, offs = _pack(strings, lead=5)
    kw = dict(max_records=8, compact_pitch=64)
    _forced(cfg, 3)
    out, res, _ = _both(cfg, data, offs, slices=3, **kw)
    _vs_oracle(out, res, ocfg, data, offs, **kw)
    few, foffs = _pack(strings[:9], lead=5)
    _forced(cfg, 0)
    out, res, _ = _both(cfg, few, foffs, **kw)
    _vs_oracle(out, res, ocfg, few, foffs, **kw)


def test_default_slicing_by_bytes():
    """No forced count: 403 strings of 24 to 64 KiB (about 17 MiB) are cut into two slices by bytes."""
    from test_batch_chunked import ALPHA
    from test_oracle_golden import SNIPPETS
    M = 65537
    rng = np.random.default_rng(403)
    cfg = product_config("regex1", M)
    alpha = np.frombuffer(ALPHA, np.uint8)
    strings = []
    for L in rng.integers(24 << 10, M, 403):
        b = alpha[rng.integers(0, len(alpha), int(L))].tobytes()
        at, sn = int(rng.integers(0, L - 64)), SNIPPETS[int(rng.integers(0, len(SNIPPETS)))]
        strings.append(b[:at] + sn + b[at + len(sn):])
    data, offs = _pack(strings, lead=3)
    assert len(_cuts(offs)) - 1 == 2
    _forced(cfg, 0)
    for sparse in (False, True):
        _both(cfg, data, offs, sparse=sparse, max_records=4, compact_pitch=32)


# ---- 2. D2H modes, buffers, NULL columns, accumulate, u16 states ---------------------------------------------------------------
def _max_sectors(out, cuts):
    """The most non-zero 32-byte sectors of one sparse column in one slice."""
    cols = out.substr_ids + out.start_enable + out.end_enable + [out.masked_chars, out.masked_substr_ids]
    best = 0
    for col in (c for c in cols if c is not None):
        for lo, hi in zip(cuts, cuts[1:]):
            b = col[lo:hi].reshape(-1)
            b = np.concatenate([b, np.zeros(-len(b) % 32, np.uint8)]).reshape(-1, 32)
            best = max(best, int(b.any(axis=1).sum()))
    return best


def test_dense_sparse_and_reuse(capfd):
    """Dense D2H, B2R_OUT_SPARSE_D2H, then B2R_OUT_SPARSE_REUSE on the same buffers with different strings (other slice
    boundaries): the reuse call clears the sectors of the first call; a low sparse_cap forces dense fallbacks in between."""
    import halo2_regex_b200 as H
    M = 4097
    rng = random.Random(77)
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    kw = dict(max_records=4, compact_pitch=32)
    n = 90
    _forced(cfg, 5)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(n)])
    data, offs = _pack(strings, lead=1)
    out, res, _ = _both(cfg, data, offs, slices=5, **kw)
    _vs_oracle(out, res, ocfg, data, offs, **kw)
    # the reuse record of a handle is that of its last SPARSE call: the reference calls of b2r_match_batch_host are dense here, so
    # that every chunked call finds the record of the chunked call before it.  Step 2 changes sparse_cap (no reuse: the layout of
    # the record differs), steps 2-4 take dense fallbacks that the next step clears from the record, step 4 changes the slice
    # count (reuse all the same: the record carries its own slices).  The trace says whether a call reused.
    mine = cfg.new_host_outputs(n, fill=0xAB, **kw)
    cfg.set_option("trace_host", 1)
    for step, (cap, slices, reused) in enumerate(((0, 5, False), (0, 5, True), (8, 5, False), (8, 5, True), (8, 3, True))):
        strings = _strings(rng, M, [rng.randrange(0, 300) if step == 0 else rng.randrange(M // 2, M) for _ in range(n)])
        data, offs = _pack(strings, lead=step)
        cfg.set_option("sparse_cap", cap)
        _forced(cfg, slices)
        capfd.readouterr()
        g, r = cfg.match_batch_chunked_host(data, offs, out=mine, check=False, sparse=True, reuse=step > 0)
        assert ("reused buffers" in capfd.readouterr().err) == reused, step
        assert cfg.last_launch_count() == _expected_launches(cfg, offs, g, sparse=True, slices=slices)
        if cap == 0:                                                   # sparse D2H moved fewer bytes than the columns hold
            assert cfg.last_host_bytes()[1] < 0.6 * sum(a.nbytes for a in g.all_arrays())
        else:                                                          # some column slice has more non-zero sectors than the cap
            assert _max_sectors(g, _cuts(offs, slices)) > cap
        g_host, r_host = cfg.match_batch_host(data, offs, check=False, fill=0xCD, **kw)
        _equal(g_host, g)
        assert _res_tuple(r_host) == _res_tuple(r)
        _vs_oracle(g, r, ocfg, data, offs, **kw)
    cfg.set_option("trace_host", 0)
    _forced(cfg, 5)
    cfg.set_option("sparse_cap", 0)
    # pinned buffers from the library's allocator
    alloc = H.PinnedAllocator()
    try:
        pins = tuple(cfg.new_host_outputs(n, fill=0x33, allocator=alloc, **kw) for _ in range(2))
        for sparse in (False, True):
            _both(cfg, data, offs, outs=pins, sparse=sparse, slices=5)
    finally:
        alloc.free()


def test_null_columns_accumulate_and_u16_states():
    import halo2_regex_b200 as H
    M = 2500
    rng = random.Random(21)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(81)])
    data, offs = _pack(strings, lead=7)
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    _forced(cfg, 4)
    for want in ({"status", "masked_chars"}, {"states", "status", "mult"}, {"status", "records", "compact_bytes", "masked_substr_ids"},
                 {"start_enable", "end_enable", "status", "endpoint_mult"}):
        for sparse in (False, True):
            _both(cfg, data, offs, want=want, sparse=sparse, slices=4, max_records=8, compact_pitch=64)
    # B2R_OUT_ACCUMULATE_MULT: counters pre-filled with one call's counts, one accumulating call on top
    outs = (cfg.new_host_outputs(81, fill=0x11), cfg.new_host_outputs(81, fill=0x11))
    _both(cfg, data, offs, outs=outs, slices=4)
    out, _, _ = _both(cfg, data, offs, outs=outs, flags=H._abi.B2R_OUT_ACCUMULATE_MULT, slices=4)
    o, _ = ocfg.match_batch(data, offs)
    for d in range(2):
        assert np.array_equal(out.mult[d], 2 * o.mult[d]) and np.array_equal(out.endpoint_mult[d], 2 * o.endpoint_mult[d])
    # u16 state column: the 1023-state DFA
    dfa = make_dfa(1023, 6, *_first_and_accepted(1023, 3), "sink", seed=1023)
    M = 3073
    cfg, ocfg = _product([dfa], M), _oracle([dfa], M)
    assert cfg.state_widths == [2]
    alpha = bytes(b for b in dfa.alphabet if b != dfa.sink_byte)
    strings = _strings(rng, M, [0, 1, M - 1] + [rng.randrange(0, M) for _ in range(38)], alphabet=alpha, plant=False)
    data, offs = _pack(strings, lead=2)
    _forced(cfg, 3)
    for sparse in (False, True):
        out, res, _ = _both(cfg, data, offs, sparse=sparse, slices=3, max_records=16, compact_pitch=128)
        _vs_oracle(out, res, ocfg, data, offs, max_records=16, compact_pitch=128)


# ---- 3. forced slices, odd pitches -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,row_pitch,bitmap_pitch", [(90, 96, 12), (4097, 4112, 516)])
@pytest.mark.parametrize("compact_pitch", [8, 13])
def test_forced_slices_and_odd_pitches(M, row_pitch, bitmap_pitch, compact_pitch):
    """n not a multiple of 4 or 32, slice bases at every multiple of 4 strings: bitmap_pitch 12 / 516 puts column slices on
    16-byte (not 32-byte) boundaries, compact_pitch 8 and 13 the compact areas on 8-byte and odd ones."""
    rng = random.Random(M * 31 + compact_pitch)
    cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
    n = 203 if M < 1000 else 67
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(n)])
    data, offs = _pack(strings, lead=9)
    kw = dict(row_pitch=row_pitch, bitmap_pitch=bitmap_pitch, max_records=3, compact_pitch=compact_pitch)
    inner = []
    for slices in (2, 5, 16):
        _forced(cfg, slices)
        inner += _cuts(offs, slices)[1:-1]
        for sparse in (False, True):
            out, res, _ = _both(cfg, data, offs, sparse=sparse, slices=slices, **kw)
        _vs_oracle(out, res, ocfg, data, offs, **kw)
    assert any(c % 32 for c in inner) and any(c % 8 for c in inner)      # boundaries between those of the batch path


# ---- 4. failures in a later slice -------------------------------------------------------------------------------------------------
def test_failures_in_later_slices():
    """The partial `example` DFA: an invalid transition and a too-long string in later slices; the lowest global index wins,
    with the same code, string_idx, pos, state, byte and def as b2r_match_batch_host."""
    import halo2_regex_b200 as H
    M = 3500
    body = _example(M - 1)

    def bad_at(p):
        return body[:p] + b"X" + body[p + 1:]
    rng = random.Random(5)
    strings = [_example(rng.randrange(0, M)) for _ in range(43)]
    cfg, ocfg = product_config("example", M), oracle_config("example", M)
    _forced(cfg, 4)
    bad = list(strings)
    bad[30], bad[35] = bad_at(1500), body + b"e"
    data, offs = _pack(bad, lead=3)
    assert _cuts(offs, 4)[1] <= 30
    for sparse in (False, True):
        out, res, _ = _both(cfg, data, offs, sparse=sparse, slices=4)
        assert res.code == H._abi.B2R_ERR_INVALID_TRANSITION and res.string_idx == 30 and res.pos == 1500
    _vs_oracle(out, res, ocfg, data, offs)
    bad = list(strings)
    bad[25], bad[33] = body + b"email", bad_at(7)
    data, offs = _pack(bad)
    out, res, _ = _both(cfg, data, offs, slices=4)
    assert res.code == H._abi.B2R_ERR_TOO_LONG and res.string_idx == 25
    _vs_oracle(out, res, ocfg, data, offs)
    with pytest.raises(H.InvalidTransitionError) as e:
        cfg.match_batch_chunked_host(*_pack([_example(100), bad_at(9)]))
    assert (e.value.string_idx, e.value.pos) == (1, 9)


# ---- 5. the small path and the empty batch ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 5, 32])
def test_small_path_and_empty_batch(n):
    import halo2_regex_b200 as H
    M = 8193
    rng = random.Random(n)
    cfg, ocfg = product_config("three", M), oracle_config("three", M)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(n)])
    data, offs = _pack(strings, lead=11)
    out, res, _ = _both(cfg, data, offs)
    assert n == 0 or _small(cfg, offs, out)
    _vs_oracle(out, res, ocfg, data, offs)
    if n:
        outs = (cfg.new_host_outputs(n, fill=1), cfg.new_host_outputs(n, fill=1))
        _both(cfg, data, offs, outs=outs)
        out, _, _ = _both(cfg, data, offs, outs=outs, flags=H._abi.B2R_OUT_ACCUMULATE_MULT)
        o, _ = ocfg.match_batch(data, offs)
        for d in range(3):
            assert np.array_equal(out.mult[d], 2 * o.mult[d])
        _forced(cfg, 0, small_path=0)                                  # the same batch through the sliced pipeline
        _both(cfg, data, offs, small_path=False)
        _forced(cfg, 0)


# ---- 6. multi-device handle ------------------------------------------------------------------------------------------------------
def _device_ranges(offs, nd):
    """csrc/host.cu, multi_host_batch: ranges balanced by bytes, cut at multiples of 4 strings for the chunked variant."""
    offs = np.asarray(offs, dtype=np.uint64)
    n = len(offs) - 1
    b0, total = int(offs[0]), int(offs[n]) - int(offs[0])
    cuts = [0]
    for k in range(1, nd):
        target = b0 + total // nd * k + total % nd * k // nd
        j = int(np.searchsorted(offs, np.uint64(target), side="left"))
        cuts.append(max(cuts[-1], min(n, (j + 2) & ~3)))
    return cuts + [n]


@pytest.mark.parametrize("n_dev", [2, 4])
def test_multi_device_handle(n_dev):
    """Fewer than 32 strings per device still reach every device; the all-reduced counters equal those of a single-device call."""
    import os
    import torch
    import halo2_regex_b200 as H
    from conftest import DEFS
    if torch.cuda.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    M = 8193
    rng = random.Random(n_dev)
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(os.path.join(DEFS, a)), [H.SubstrRegexDef.read_from_text(os.path.join(DEFS, s)) for s in ss])
            for a, ss in DEF_SETS["test1"]]
    cfg = H.RegexVerifyConfig.configure(M, defs, devices=list(range(n_dev)))
    one, ocfg = product_config("test1", M), oracle_config("test1", M)
    for n in (6 * n_dev + 3, 150):
        strings = _strings(rng, M, [rng.randrange(M // 2, M) for _ in range(n)])
        data, offs = _pack(strings, lead=1)
        ranges = _device_ranges(offs, n_dev)
        assert all(hi > lo for lo, hi in zip(ranges, ranges[1:])), ranges
        for sparse in (False, True):
            out, res, _ = _both(cfg, data, offs, sparse=sparse, launches=False)
            # every device ran the chunked kernels over its range (one slice each: far less than 8 MiB per device)
            exp = sum(_chunked_launches(cfg, hi - lo, M, _max_smem()) for lo, hi in zip(ranges, ranges[1:]))
            if sparse:
                exp += sum(_n_sparse_cols(cfg, out.want) + 1 for lo, hi in zip(ranges, ranges[1:]))
            assert cfg.last_launch_count() == exp, (cfg.last_launch_count(), exp)
            single, sres = one.match_batch_chunked_host(data, offs, check=False, fill=0x5A, sparse=sparse)
            _equal(out, single)
            assert _res_tuple(res) == _res_tuple(sres)
        _vs_oracle(out, res, ocfg, data, offs)
