"""Every tuning knob of b2r_config_set_option on every entry point that plans a walk, against the CPU oracle.  include/b2r.h
promises bit-identical results under every setting (debug / host_debug aside); each case here compares every column, status,
record, compact byte and counter with the oracle, and asserts b2r_last_plan where a placement is forced.

  chunked batch    every forced table / bin placement on 1, 2, 3 and 4 u8 defs, a u16 def (S = 300, REPL16 still fits) and the
                   1023-state DFA; each call against b2r_match_batch under the same knob, tensor for tensor, and the oracle
  long string      the same configs and placements at lengths 0, 1, 1025 and 70 001, fused and general prefix pass, device and
                   host entry points in turn
  batch            the placements for 2 and 4 defs
  hist_cache_log2  bin caches of 2^8 .. 2^14 slots (and out-of-range values, which mean 2^12) in front of the global bins, on a
                   DFA whose keys all fit the smallest cache and on one with ~77 k keys; four defs whose 2^14-slot caches
                   cannot fit together (the planner shrinks them)
  spread_fill = 0  the walk's zero-fill issued in one burst, with the emit stage fused and separate
  host pipeline    slices (and out-of-range values), dense and sparse D2H, sparse_direct, B2R_OUT_SPARSE_REUSE across a change
                   of sparse_direct
  accumulate       B2R_OUT_ACCUMULATE_MULT on b2r_match_long and b2r_match_long_host

The oracle runs once per input, not once per knob setting."""
import random
import zlib

import numpy as np
import pytest

from conftest import oracle_config, product_config
from test_batch_chunked import _both, _to_device, _vs_oracle
from test_batch_chunked import _strings as _snippet_strings
from test_dfa_shapes import PLACEMENTS, Dfa, _compare, _long_body, _oracle, _placement_expected, _product, _run_long, _strings, make_dfa
from test_gpu_parity import FOUR_DEFS, _pack
from test_oracle_golden import SNIPPETS, _random_strings

pytestmark = pytest.mark.gpu

PRODUCT_SETS = {"regex1": "regex1", "test1": "test1", "three": "three", "four": FOUR_DEFS}
CONFIGS = ["regex1", "test1", "three", "four", "u16_S300", "dfa1023"]
LONG_LENGTHS = [0, 1, 1025, 70001]


@pytest.fixture(scope="module")
def max_smem():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


class _Defs:
    """One def config of the matrix: product and oracle handles at any max_chars_size, batch strings and long bodies."""

    def __init__(self, name):
        self.name = name
        self.spec = PRODUCT_SETS.get(name)
        if name == "u16_S300":          # P = 512 padded states, 3 byte classes: 16-bit replicated tables still fit
            self.dfas = [make_dfa(300, 2, 150, 17, "perm", seed=301, alphabet=b"ab")]
        elif name == "dfa1023":
            from halo2_regex_b200 import workloads as W
            allstr, substr, _ = W.large_dfa_texts()
            self.dfas = [Dfa(1023, None, None, allstr, [substr], None)]
        elif name.startswith("hist_"):  # the bin-cache DFAs of test_hist_cache_sizes
            S, C = {"hist_S3_C3": (3, 3), "hist_S300_C256": (300, 256)}[name]
            self.dfas = [make_dfa(S, C, 1, 2, "perm", seed=S, alphabet=b"xyz" if S == 3 else bytes(range(256)))]
        else:
            self.dfas = None

    def product(self, M):
        return product_config(self.spec, M) if self.spec else _product(self.dfas, M)

    def oracle(self, M):
        return oracle_config(self.spec, M) if self.spec else _oracle(self.dfas, M)

    def strings(self, rng, M, n=40):
        """n ragged strings: lengths 0, 1, 1024, 1025 and M-1 among random ones."""
        fixed = [0, 1, 1024, 1025, M - 1]
        lens = fixed + [rng.randrange(0, M) for _ in range(n - len(fixed))]
        if self.spec:
            return _snippet_strings(rng, M, lens)
        if self.name == "dfa1023":
            from halo2_regex_b200 import workloads as W
            rows, _ = W.config4_numpy(n, M - 1)
            return [bytes(rows[j][:L]) for j, L in enumerate(lens)]
        np_rng = np.random.default_rng(rng.randrange(1 << 30))
        return _strings(rng, self.dfas[0], n - 2, M, extra=[_long_body(np_rng, self.dfas[0], L).tobytes() for L in (1024, 1025)])

    def body(self, rng, length):
        if self.spec:
            return _snippet_strings(rng, length + 1, [length])[0]
        if self.name == "dfa1023":
            from halo2_regex_b200 import workloads as W
            rows, _ = W.config4_numpy(-(-length // 4096) or 1, 4096)
            return rows.reshape(-1)[:length].tobytes()
        return _long_body(np.random.default_rng(rng.randrange(1 << 30)), self.dfas[0], length).tobytes()


class _OracleOnce:
    """An oracle handle for one input batch: computed on the first call, then returned for every knob setting."""

    def __init__(self, ocfg):
        self.ocfg, self.out = ocfg, None

    def match_batch(self, data, offs, **kw):
        if self.out is None:
            self.out = self.ocfg.match_batch(data, offs, **kw)
        return self.out


def _check_plan(path, cfg, tm, hm, max_smem):
    """b2r_last_plan after a call with (tm, hm) forced: honoured where it fits with room to spare, never across a limit of the
    planner.  Prints one line of the (path, defs, state width, forced placement) -> plan table."""
    plan = cfg.last_plan()
    exp = _placement_expected(cfg.dummy_states, cfg.num_byte_classes, tm, hm, max_smem)
    print(f"plan | {path} | {cfg.n_defs} | u{8 * cfg.state_widths[0]} | S={cfg.dummy_states} C={cfg.num_byte_classes} | {tm}/{hm} | {plan[0]}/{plan[1]} | {exp}")
    if exp is True:
        assert plan == (tm, hm), (path, tm, hm, plan)
    elif isinstance(exp, tuple):
        if not exp[0]:
            assert plan[0] != tm, (path, tm, hm, plan)
        if not exp[1]:
            assert plan[1] != hm, (path, tm, hm, plan)
    return plan


def _force(cfg, tm, hm):
    cfg.set_option("table_mode", tm)
    cfg.set_option("hist_mode", hm)


# ---- a. chunked batch x placements ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CONFIGS)
def test_chunked_placements(name, max_smem):
    """Every forced placement on b2r_match_batch_chunked: 40 ragged strings of 2-3 slots plus a partial one (slots past a
    string's end hold dummy rows), behind an unaligned lead; equal to b2r_match_batch under the same knob and to the oracle."""
    defs = _Defs(name)
    M = 2049 if CONFIGS.index(name) % 2 == 0 else 3073
    cfg = defs.product(M)
    rng = random.Random(zlib.crc32(f"chunked/{name}".encode()))
    strings = defs.strings(rng, M)
    data, offs = _pack(strings, lead=5)
    d_bytes, d_offs = _to_device(data, offs)
    once = _OracleOnce(defs.oracle(M))
    for tm, hm in PLACEMENTS:
        _force(cfg, tm, hm)
        out, res = _both(cfg, d_bytes, d_offs, M, max_records=8, compact_pitch=64)
        try:
            _vs_oracle(out, res, once, data, offs, max_records=8, compact_pitch=64)
        except AssertionError as e:
            raise AssertionError(f"{name} {tm}/{hm}: {e}") from None
        _check_plan("chunked", cfg, tm, hm, max_smem)


# ---- b. long string x placements --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CONFIGS)
def test_long_placements(name, max_smem):
    """Every forced placement on b2r_match_long / b2r_match_long_host (alternating) at lengths 0, 1, 1025 and 70 001, with the
    fused and the general prefix pass where the fused one applies; b2r_last_plan reports the walk over the chunks."""
    defs = _Defs(name)
    cfg = defs.product(64)
    rng = random.Random(zlib.crc32(f"long/{name}".encode()))
    fuseds = (1, 0) if max(cfg.dummy_states) + 1 <= 33 else (1,)
    for j, length in enumerate(LONG_LENGTHS):
        s = defs.body(rng, length)
        assert len(s) == length
        data, offs = _pack([s])
        expected = defs.oracle(length + 1).match_batch(data, offs, max_records=64, compact_pitch=512)
        for k, (tm, hm) in enumerate(PLACEMENTS):
            _force(cfg, tm, hm)
            for fused in fuseds:
                try:
                    _run_long(cfg, None, s, device=(j + k + fused) % 2 == 0, fused=fused, max_smem=max_smem, expected=expected)
                except AssertionError as e:
                    raise AssertionError(f"{name} {tm}/{hm}: {e}") from None
                _check_plan("long", cfg, tm, hm, max_smem)


# ---- c. batch x placements, 2 and 4 defs ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["test1", "four"])
def test_batch_placements_multi_def(name, max_smem):
    """The rows of the batch placement matrix that test_gpu_parity / test_dfa_shapes leave out: two and four defs."""
    defs = _Defs(name)
    M = 261
    cfg = defs.product(M)
    rng = random.Random(zlib.crc32(f"batch/{name}".encode()))
    strings = _random_strings(rng, 300, M - 1, SNIPPETS) + [b"", b"q", b"x" * (M - 1)]
    data, offs = _pack(strings, lead=3)
    o, ores = defs.oracle(M).match_batch(data, offs, max_records=8, compact_pitch=64)
    for tm, hm in PLACEMENTS:
        _force(cfg, tm, hm)
        g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, max_records=8, compact_pitch=64)
        try:
            _compare(g, gres, o, ores)
        except AssertionError as e:
            raise AssertionError(f"{name} {tm}/{hm}: {e}") from None
        _check_plan("batch", cfg, tm, hm, max_smem)


# ---- d. hist_cache_log2 ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,values", [("hist_S3_C3", [8, 9, 13, 14, 0, 7, 15]), ("hist_S300_C256", [8, 9, 13, 14, 0, 7, 15]),
                                         ("four", [14])])
def test_hist_cache_sizes(name, values, max_smem):
    """Global bins behind shared-memory caches of every size on the batch, chunked and long paths.  A slot belongs to the first
    key that hashes to it; every other key of that slot is counted in the global bins.  S = 3 over 3 bytes: every key fits the
    smallest cache.  S = 300 over all 256 bytes: ~77 k keys, far more than 2^14 slots, so many keys take the global atomics.
    Four defs at 2^14: 4 x 128 KB of caches cannot fit, the planner shrinks them.  mult and endpoint_mult must stay exact."""
    defs = _Defs(name)
    M = 2049
    cfg = defs.product(M)
    rng = random.Random(zlib.crc32(f"hist/{name}".encode()))
    strings = defs.strings(rng, M)
    data, offs = _pack(strings, lead=1)
    d_bytes, d_offs = _to_device(data, offs)
    once = _OracleOnce(defs.oracle(M))
    body = defs.body(rng, 70001)
    bd, bo = _pack([body])
    long_expected = defs.oracle(len(body) + 1).match_batch(bd, bo, max_records=64, compact_pitch=512)
    cfg.set_option("hist_mode", "global")
    for k, v in enumerate(values):
        cfg.set_option("hist_cache_log2", v)
        try:
            out, res = _both(cfg, d_bytes, d_offs, M, max_records=8, compact_pitch=64)   # batch, then chunked: equal tensors
            assert cfg.last_plan()[1] == "global"
            _vs_oracle(out, res, once, data, offs, max_records=8, compact_pitch=64)
            _run_long(cfg, None, body, device=k % 2 == 0, fused=1, max_smem=max_smem, expected=long_expected)
            assert cfg.last_plan()[1] == "global"
        except AssertionError as e:
            raise AssertionError(f"{name} hist_cache_log2={v}: {e}") from None
    assert res.code == 0 and not (out.mult_all == 0).all()


# ---- e. spread_fill = 0 -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("set_name", ["regex1", "three"])
def test_spread_fill_off(set_name):
    """spread_fill = 0: the walk issues each tile's zero-fill ops at once instead of spreading them over the chunk loop (M = 513:
    17 chunks of 32 rows per tile), with the emit stage fused (fuse = 1) and as its own kernel (fuse = 2)."""
    M = 513
    cfg = product_config(set_name, M)
    rng = random.Random(zlib.crc32(f"spread/{set_name}".encode()))
    strings = _random_strings(rng, 400, M - 1, SNIPPETS) + [b"", b"x" * (M - 1)]
    data, offs = _pack(strings, lead=7)
    o, ores = oracle_config(set_name, M).match_batch(data, offs, max_records=8, compact_pitch=64)
    cfg.set_option("spread_fill", 0)
    for fuse in (1, 2):
        cfg.set_option("fuse", fuse)
        g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, max_records=8, compact_pitch=64)
        _compare(g, gres, o, ores)
        assert cfg.last_launch_count() == (2 if fuse == 1 else 3)


# ---- f. host pipeline knobs --------------------------------------------------------------------------------------------------
def test_host_slices_and_sparse_modes():
    """b2r_match_batch_host at n = 16 411 (>= 16 384: the sliced pipeline): slices 1, 3, 16 and the out-of-range 0 and 17 (the
    default then), each with dense D2H, sparse D2H compacted in device memory and sparse D2H stored straight into pinned memory."""
    M, n = 97, 16411
    cfg = product_config("test1", M)
    rng = random.Random(16411)
    strings = _random_strings(rng, n, M - 1, SNIPPETS)
    data, offs = _pack(strings, lead=3)
    kw = dict(max_records=4, compact_pitch=32)
    o, ores = oracle_config("test1", M).match_batch(data, offs, **kw)
    for slices in (1, 3, 16, 0, 17):
        cfg.set_option("slices", slices)
        for sparse, direct in ((False, 0), (True, 0), (True, 1)):
            cfg.set_option("sparse_direct", direct)
            g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xAB, sparse=sparse, **kw)
            try:
                _compare(g, gres, o, ores)
                assert gres.n_overlap_lo == ores.n_overlap_lo
            except AssertionError as e:
                raise AssertionError(f"slices={slices} sparse={sparse} sparse_direct={direct}: {e}") from None


def test_sparse_reuse_across_sparse_direct():
    """B2R_OUT_SPARSE_REUSE on the same host buffers: one sparse call, then three reuse calls with different strings; sparse_direct
    changes between the reuse calls (the reuse record of the previous call does not say which mode wrote it)."""
    M, n = 97, 16411
    cfg = product_config("three", M)
    kw = dict(max_records=4, compact_pitch=32)
    out = cfg.new_host_outputs(n, fill=0xAB, **kw)
    rng = random.Random(4)
    for step, direct in enumerate((0, 0, 1, 0)):
        strings = _random_strings(rng, n, M - 1, SNIPPETS)
        data, offs = _pack(strings, lead=step)
        o, ores = oracle_config("three", M).match_batch(data, offs, **kw)
        cfg.set_option("sparse_direct", direct)
        g, gres = cfg.match_batch_host(data, offs, out=out, check=False, sparse=True, reuse=step > 0)
        try:
            _compare(g, gres, o, ores)
        except AssertionError as e:
            raise AssertionError(f"step {step} sparse_direct={direct}: {e}") from None


# ---- g. long path with B2R_OUT_ACCUMULATE_MULT -------------------------------------------------------------------------------
@pytest.mark.parametrize("device", [True, False])
def test_long_accumulate_mult(device):
    """B2R_OUT_ACCUMULATE_MULT on the long path: counters pre-filled with the oracle's counters of another string, then two
    accumulating calls (fused, then general prefix pass); after call k the counters are the other string's plus k times this
    one's, and every other output is this string's."""
    import torch
    import halo2_regex_b200 as H
    from halo2_regex_b200.buffers import HostOutputs
    acc = H._abi.B2R_OUT_ACCUMULATE_MULT
    cfg = product_config("test1", 64)
    rng = random.Random(7)
    a, b = _snippet_strings(rng, 5001, [5000])[0], _snippet_strings(rng, 3001, [3000])[0]
    kw = dict(max_records=64, compact_pitch=512)
    o, ores = oracle_config("test1", 5001).match_batch(*_pack([a]), **kw)
    ob, _ = oracle_config("test1", 3001).match_batch(*_pack([b]), **kw)
    one = ([m.copy() for m in o.mult], [m.copy() for m in o.endpoint_mult])
    D = cfg.n_defs
    if device:
        buf = torch.zeros(len(a) + 16, dtype=torch.uint8, device="cuda")
        buf[:len(a)].copy_(torch.from_numpy(np.frombuffer(a, np.uint8).copy()))
        out = H.DeviceOutputs(cfg, 1, max_chars_size=len(a) + 1, **kw)
        for d in range(D):
            out.mult[d].copy_(torch.from_numpy(ob.mult[d].astype(np.int64)))
            out.endpoint_mult[d].copy_(torch.from_numpy(ob.endpoint_mult[d].astype(np.int64)))
    else:
        out = HostOutputs(1, len(a) + 1, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, fill=0xCD, **kw)
        for d in range(D):
            out.mult[d][:] = ob.mult[d]
            out.endpoint_mult[d][:] = ob.endpoint_mult[d]
    for k, fused in ((1, 1), (2, 0)):
        cfg.set_option("long_fused", fused)
        if device:
            cfg.match_long_device(buf[:len(a)], out, flags=acc)
            g, gres = out.to_host(), cfg.batch_result(check=False)
        else:
            g, gres = cfg.match_long_host(a, out=out, flags=acc, check=False)
        for d in range(D):
            o.mult[d] = ob.mult[d] + k * one[0][d]
            o.endpoint_mult[d] = ob.endpoint_mult[d] + k * one[1][d]
        try:
            _compare(g, gres, o, ores)
        except AssertionError as e:
            raise AssertionError(f"accumulating call {k} ({'device' if device else 'host'}): {e}") from None
