"""b2r_match_batch_chunked: the batch entry point that cuts every string into 1 KiB slots walked in parallel.  Its contract is
that it writes exactly what b2r_match_batch writes for the same call, so every GPU case runs both on the same device inputs and
handle, into outputs pre-filled with the same pattern, and compares every output tensor whole (torch.equal), the multiplicity
counters and the b2r_batch_result fields.  Cases small enough for it are also compared with the CPU oracle, and every case
asserts the launch count of `_chunked_launches`, which proves how many passes and which composition branch ran.

The largest cases carry `huge` in their names so that a slow run (a sanitizer) can skip them."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, product_config
from test_dfa_shapes import LONG_CHUNK, LONG_FANOUT, _first_and_accepted, _max_smem, _oracle, _product, make_dfa
from test_gpu_parity import _pack
from test_oracle_golden import SNIPPETS

ALPHA = b"abc xyz.@\r\n"


# ---- helpers ------------------------------------------------------------------------------------------------------------------
def _chunked_launches(cfg, n, M, max_smem, per_pass=None, finalize=True):
    """Kernel launches of one b2r_match_batch_chunked call (csrc/api.cu, match_batch_chunked_impl): per pass of whole strings and
    per def head / dedupe / tail / gather / reset, then the tree over the pass's slots (one scan per level + resolve when
    2 * 64 * (S+1) u16 fit shared memory, else compose + propagate per level + the root entry), then one walk per pass; emit once;
    finalize when a multiplicity column is wanted.  A pass holds at most 1 GiB of level-0 transition vectors (chunked_max_maps)."""
    if n == 0:
        return 1 if finalize else 0
    K = -(-M // LONG_CHUNK)
    S1s = [s + 1 for s in cfg.dummy_states]
    if per_pass is None:
        per_pass = max(1, (1 << 30) // (K * sum(S1s) * 2))
    per_pass = min(per_pass, n)
    total = 0
    for j0 in range(0, n, per_pass):
        levels, m = 1, min(per_pass, n - j0) * K
        while m > 1:
            m = -(-m // LONG_FANOUT)
            levels += 1
        scan = lambda s1: 2 * LONG_FANOUT * s1 * 2 <= max_smem and levels <= 12  # noqa: E731
        total += sum(5 + (levels if scan(s1) else 2 * (levels - 1) + 1) for s1 in S1s) + 1
    return total + 1 + (1 if finalize else 0)


def _strings(rng, M, lengths, alphabet=ALPHA, snippets=SNIPPETS, plant=True):
    """Strings of the given lengths; snippets planted at random places and across slot boundaries (at 1024c - 3)."""
    out = []
    for L in lengths:
        b = bytearray(rng.choice(alphabet) for _ in range(L))
        if plant and snippets:
            spots = [rng.randrange(L) for _ in range(min(3, L // 64))] + [c * LONG_CHUNK - 3 for c in range(1, L // LONG_CHUNK + 1)]
            for at in spots:
                sn = rng.choice(snippets)
                if 0 <= at and at + len(sn) <= L:
                    b[at:at + len(sn)] = sn
        out.append(bytes(b))
    return out


def _lengths(rng, M, n_random=6):
    fixed = [0, 1, 1023, 1024, 1025, 2048, M - 1]
    return sorted({L for L in fixed if 0 <= L <= M - 1}) + [rng.randrange(0, M) for _ in range(n_random)]


def _example(L):
    """A string of length L that the partial `example` DFA walks without an invalid transition: 'email was meant for @' + a
    name of L - 22 lowercase letters + '.' (shorter: a prefix of that)."""
    s = b"email was meant for @" + (b"vitalik" * (L // 7 + 1))[:max(0, L - 22)] + b"."
    return s[:L]


def _outputs(cfg, n, fill=0x5A, **kw):
    """DeviceOutputs with every column (not the counters) pre-filled with one pattern, so that whole tensors can be compared."""
    import halo2_regex_b200 as H
    out = H.DeviceOutputs(cfg, n, **kw)
    for t in _tensors(out):
        t.fill_(fill if t.dtype == __import__("torch").uint8 else fill * 257)
    return out


def _tensors(out):
    cols = list(out.states) + list(out.substr_ids) + list(out.start_enable) + list(out.end_enable)
    cols += [out.masked_chars, out.masked_substr_ids, out.status, out.records, out.compact_bytes]
    return [t for t in cols if t is not None]


def _res_tuple(r):
    return (r.code, r.string_idx, r.pos, r.state, r.byte, r.defidx, r.n_overlap_lo)


def _to_device(data, offs):
    import torch
    d_bytes = torch.from_numpy(data.copy()).cuda() if len(data) else torch.zeros(0, dtype=torch.uint8, device="cuda")
    d_offs = torch.from_numpy(offs.astype(np.int64)).cuda()
    return d_bytes, d_offs


def _both(cfg, d_bytes, d_offs, M, flags=0, launches=None, runs=1, stream=None, **kw):
    """b2r_match_batch, then b2r_match_batch_chunked (each `runs` times into its own outputs), same inputs and handle; every
    output tensor, counter and b2r_batch_result field equal.  Returns (chunked outputs, its batch result)."""
    import torch
    n = d_offs.numel() - 1
    res = []
    outs = []
    for chunked in (False, True):
        out = _outputs(cfg, n, **kw)
        for _ in range(runs):
            if chunked:
                cfg.match_batch_chunked_device(d_bytes, d_offs, out, flags=flags, stream=stream)
            else:
                cfg.match_batch_device(d_bytes, d_offs, out, flags=flags, stream=stream)
        if chunked and launches is not None:
            assert cfg.last_launch_count() == launches, (cfg.last_launch_count(), launches)
        res.append(cfg.batch_result(stream=stream, check=False))
        outs.append(out)
    a, b = outs
    for x, y in zip(_tensors(a) + [a.mult_all], _tensors(b) + [b.mult_all]):
        if not torch.equal(x, y):
            bad = torch.nonzero((x != y).reshape(x.shape[0], -1) if x.dim() > 1 else (x != y))
            raise AssertionError(f"tensor of shape {tuple(x.shape)} differs at {bad[:4].tolist()} ({len(bad)} cells)")
    assert _res_tuple(res[0]) == _res_tuple(res[1])
    return b, res[1]


def _vs_oracle(out, res, ocfg, data, offs, max_records=8, compact_pitch=64):
    import halo2_regex_b200 as H
    o, ores = ocfg.match_batch(data, offs, max_records=max_records, compact_pitch=compact_pitch)
    assert res.code == ores.code
    if ores.code != 0:
        assert (res.string_idx, res.pos, res.state, res.byte, res.defidx) == (ores.string_idx, ores.pos, ores.state, ores.byte, ores.defidx)
    assert res.n_overlap_lo == ores.n_overlap_lo
    errs = H.compare_outputs(out.to_host(), o)
    assert errs == [], "\n".join(errs)


def _case(cfg, ocfg, strings, M, lead=0, max_smem=None, oracle=True, **kw):
    data, offs = _pack(strings, lead)
    d_bytes, d_offs = _to_device(data, offs)
    kw.setdefault("max_records", 8)
    kw.setdefault("compact_pitch", 64)
    fin = kw.get("want") is None or bool({"mult", "endpoint_mult"} & set(kw["want"]))
    launches = _chunked_launches(cfg, len(strings), M, max_smem if max_smem else _max_smem(), finalize=fin)
    out, res = _both(cfg, d_bytes, d_offs, M, launches=launches, **kw)
    if oracle:
        _vs_oracle(out, res, ocfg, data, offs, kw["max_records"], kw["compact_pitch"])
    return out, res


# ---- CPU: argument errors -----------------------------------------------------------------------------------------------------
def test_null_config_and_deviceless_handle():
    from halo2_regex_b200 import _abi
    from halo2_regex_b200._ffi import last_error, lib
    o = _abi.Outputs()
    assert lib.b2r_match_batch_chunked(None, None, None, 0, 0, C.byref(o), None) == _abi.B2R_ERR_INVALID_ARG
    cfg = product_config("regex1", 64, device=-1)
    assert cfg.device == -1
    out = cfg.new_host_outputs(1)
    assert lib.b2r_match_batch_chunked(cfg._h, None, None, 0, 0, C.byref(out.struct(0)), None) == _abi.B2R_ERR_CUDA
    assert "no CPU fallback" in last_error()


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
MS = [1, 2, 1024, 1025, 1026, 2048, 2049, 4097, 65537]


@pytest.mark.gpu
@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("set_name", list(DEF_SETS))
def test_def_sets_and_lengths(set_name, M):
    """Every def set at every slot-edge M: lengths 0, 1, 1023, 1024, 1025, 2048, M-1 and random ones, snippets across slot edges."""
    rng = random.Random(zlib.crc32(f"{set_name}/{M}".encode()))
    cfg, ocfg = product_config(set_name, M), oracle_config(set_name, M)
    if set_name == "example":   # a partial DFA: its own sentence with a long name (valid), one string with a byte it has no transition for
        strings = [_example(L) for L in _lengths(rng, M)]
        if M > 40:
            strings.append(b"email was" + b"\x01" + b"x" * (M - 20))
    else:
        strings = _strings(rng, M, _lengths(rng, M))
    _case(cfg, ocfg, strings, M)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000])
def test_ragged_batch_sizes(n):
    M = 2049
    rng = random.Random(n)
    cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
    _case(cfg, ocfg, _strings(rng, M, [rng.randrange(0, M) for _ in range(n)]), M)


@pytest.mark.gpu
def test_empty_batch_and_empty_strings():
    M = 3000
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    _case(cfg, ocfg, [], M)
    _case(cfg, ocfg, [b""] * 40, M)


@pytest.mark.gpu
@pytest.mark.parametrize("lead", [1, 7, 16, 33])
def test_unaligned_offsets(lead):
    """String starts at every alignment, total bytes not a multiple of 16."""
    M = 4097
    rng = random.Random(lead)
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(40)] + [M - 1, 3])
    assert (lead + sum(map(len, strings))) % 16
    _case(cfg, ocfg, strings, M, lead=lead)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["regex1_sink", "first_state_nonzero"])
def test_previous_string_ends_away_from_first_state(which):
    """Consecutive strings whose previous final state is not first_state: the slot after a string's last slot must start in
    first_state (the constant-map reset), not where the previous string ended."""
    rng = random.Random(3)
    if which == "regex1_sink":
        M = 3073
        cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
        strings = _strings(rng, M, [rng.randrange(1, M) for _ in range(60)])
        # strings that end right after a match (regex1's accepting sink), followed by strings that must not inherit it
        strings = [s[:-30] + b"email was meant for @ab." + b"x" * 6 if len(s) > 40 else s for s in strings]
        first = 0
    else:
        M = 2100
        dfa = make_dfa(17, 5, 9, 3, "sink", seed=11)
        cfg, ocfg = _product([dfa], M), _oracle([dfa], M)
        strings = _strings(rng, M, [rng.randrange(1, M) for _ in range(60)], alphabet=dfa.alphabet, plant=False)
        first = 9
    out, res = _case(cfg, ocfg, strings, M)
    h = out.to_host()
    finals = [int(h.states[0][j, len(s)]) for j, s in enumerate(strings)]
    assert sum(f != first for f in finals) > 10            # the case really has strings that end away from first_state


@pytest.mark.gpu
def test_truncation_and_overlap_across_slots():
    M = 4097
    rng = random.Random(9)
    strings = _strings(rng, M, [M - 1, 3000, 2049, 1025, 100] + [rng.randrange(0, M) for _ in range(20)])
    cfg, ocfg = product_config("regex3", M), oracle_config("regex3", M)
    out, _ = _case(cfg, ocfg, strings, M, max_records=1, compact_pitch=3)
    st = out.to_host().status
    assert (st["n_records"] > 1).any() and (st["n_compact"] > 3).any()
    spec = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"])] * 2       # two defs flag the same rows: overlap
    cfg, ocfg = product_config(spec, M), oracle_config(spec, M)
    out, res = _case(cfg, ocfg, strings, M)
    assert res.n_overlap_lo > 0


@pytest.mark.gpu
def test_invalid_transitions_and_too_long_strings():
    """The partial `example` DFA: invalid bytes in slot 0, in a later slot and in the last partial slot; too-long strings (and
    offsets past the byte buffer) mixed in.  The lowest failing string index wins in b2r_batch_result."""
    import halo2_regex_b200 as H
    M = 3500
    body = _example(M - 1)

    def bad_at(p):
        return body[:p] + b"X" + body[p + 1:]
    strings = [_example(2000), bad_at(5), body, bad_at(1500), bad_at(M - 3), _example(1024), _example(1025)]
    cfg, ocfg = product_config("example", M), oracle_config("example", M)
    out, res = _case(cfg, ocfg, strings, M)
    assert res.code == H._abi.B2R_ERR_INVALID_TRANSITION and res.string_idx == 1 and res.pos == 5
    flags = out.to_host().status["flags"]
    assert [j for j in range(len(strings)) if flags[j] & H._abi.B2R_ST_INVALID_TRANSITION] == [1, 3, 4]
    # a too-long string in front of an invalid one, another one behind it
    long_first = [_example(10), body + b"e", strings[0], bad_at(40), body + b"email"]
    out, res = _case(cfg, ocfg, long_first, M)
    assert res.code == H._abi.B2R_ERR_TOO_LONG and res.string_idx == 1
    flags = out.to_host().status["flags"]
    assert flags[4] & H._abi.B2R_ST_TOO_LONG and flags[3] & H._abi.B2R_ST_INVALID_TRANSITION
    # offsets that leave the byte buffer
    data, offs = _pack([_example(100), _example(200)])
    offs[2] = offs[2] + 50
    d_bytes, d_offs = _to_device(data, offs)
    _, res = _both(cfg, d_bytes, d_offs, M)
    assert res.code == H._abi.B2R_ERR_TOO_LONG and res.string_idx == 1


@pytest.mark.gpu
def test_argument_errors_match_the_batch_path():
    import torch
    import halo2_regex_b200 as H
    from halo2_regex_b200._ffi import lib
    M = 2000
    cfg = product_config("regex1", M)
    d_bytes, d_offs = _to_device(*_pack([b"abc"] * 3))
    for make in (lambda o: setattr(o, "row_pitch", 2001), lambda o: setattr(o, "bitmap_pitch", 2)):
        out = H.DeviceOutputs(cfg, 3)
        st = out.struct(0)
        make(st)
        rcs = [f(cfg._h, d_bytes.data_ptr(), d_offs.data_ptr(), 3, 3, C.byref(st), None) for f in (lib.b2r_match_batch, lib.b2r_match_batch_chunked)]
        assert rcs[0] == rcs[1] == H._abi.B2R_ERR_ALIGNMENT
    out = H.DeviceOutputs(cfg, 3)
    st = out.struct(0)
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    rcs = [f(cfg._h, buf.data_ptr() + 1, d_offs.data_ptr(), 3, 3, C.byref(st), None) for f in (lib.b2r_match_batch, lib.b2r_match_batch_chunked)]
    assert rcs[0] == rcs[1] == H._abi.B2R_ERR_ALIGNMENT
    rcs = [f(cfg._h, d_bytes.data_ptr(), None, 3, 3, C.byref(st), None) for f in (lib.b2r_match_batch, lib.b2r_match_batch_chunked)]
    assert rcs[0] == rcs[1] == H._abi.B2R_ERR_INVALID_ARG


@pytest.mark.gpu
def test_null_columns_and_accumulate():
    M = 2500
    rng = random.Random(21)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(80)])
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    for want in ({"status", "masked_chars"}, {"states", "status", "mult"}, {"status", "records", "compact_bytes", "masked_substr_ids"},
                 {"start_enable", "end_enable", "status", "endpoint_mult"}):
        _case(cfg, ocfg, strings, M, want=want)
    # B2R_OUT_ACCUMULATE_MULT over two calls: twice the counts of one call
    import halo2_regex_b200 as H
    data, offs = _pack(strings)
    d_bytes, d_offs = _to_device(data, offs)
    out, _ = _both(cfg, d_bytes, d_offs, M, flags=H._abi.B2R_OUT_ACCUMULATE_MULT, runs=2)
    o, _ = ocfg.match_batch(data, offs)
    for d in range(2):
        assert np.array_equal(out.mult[d].cpu().numpy(), 2 * o.mult[d].astype(np.int64))
        assert np.array_equal(out.endpoint_mult[d].cpu().numpy(), 2 * o.endpoint_mult[d].astype(np.int64))


def _shape_dfa(shape, k, max_smem):
    if shape in ("S31", "S32"):
        S = int(shape[1:])
        return make_dfa(S, 6, *_first_and_accepted(S, k), "collapse_2", seed=S + k, n_substrs=2)
    if shape == "S300_C256":                                  # u16 state column, tables in global memory for the prefix pass
        return make_dfa(300, 256, *_first_and_accepted(300, k + 1), "perm", seed=300 + k, alphabet=bytes(range(256)))
    S = max_smem // (2 * LONG_FANOUT * 2) - (1 if shape == "scan_edge" else 0)   # the largest tree the shared-memory scan takes, and one more
    return make_dfa(S, 6, *_first_and_accepted(S, k), "sink", seed=S + k)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["S31", "S32", "S300_C256", "scan_edge", "compose_edge"])
def test_dfa_shapes(shape):
    max_smem = _max_smem()
    k = ["S31", "S32", "S300_C256", "scan_edge", "compose_edge"].index(shape)
    dfa = _shape_dfa(shape, k, max_smem)
    M = 66 * LONG_CHUNK + 5                                     # > 64 slots per string: two tree levels even for one string
    cfg, ocfg = _product([dfa], M), _oracle([dfa], M)
    if shape == "S300_C256":
        assert cfg.state_widths[0] == 2
    if shape in ("scan_edge", "compose_edge"):
        assert (2 * LONG_FANOUT * (dfa.S + 1) * 2 <= max_smem) == (shape == "scan_edge")
    rng = random.Random(k)
    alpha = bytes(b for b in dfa.alphabet if b != dfa.sink_byte)
    strings = _strings(rng, M, [0, 1, 1024, M - 1] + [rng.randrange(0, M) for _ in range(8)], alphabet=alpha, plant=False)
    _case(cfg, ocfg, strings, M, max_smem=max_smem, max_records=64, compact_pitch=512)


@pytest.mark.gpu
def test_large_dfa_1023_states():
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from halo2_regex_b200 import workloads as W
    allstr, substr, _ = W.large_dfa_texts()
    M = 8193
    cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
    ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], M)
    rows, _ = W.config4_numpy(24, 8192)
    rng = random.Random(4)
    strings = [bytes(r[:rng.randrange(0, M)]) for r in rows] + [bytes(rows[0])]
    _case(cfg, ocfg, strings, M, max_records=16, compact_pitch=256)


@pytest.mark.gpu
def test_several_passes():
    """chunked_max_maps small enough for three strings per pass: the passes split the batch at string boundaries."""
    M = 4097
    rng = random.Random(12)
    strings = _strings(rng, M, [rng.randrange(0, M) for _ in range(50)] + [M - 1])
    cfg, ocfg = product_config("three", M), oracle_config("three", M)
    K = -(-M // LONG_CHUNK)
    per_str = K * sum(s + 1 for s in cfg.dummy_states) * 2
    cfg.set_option("chunked_max_maps", 3 * per_str + 5)
    data, offs = _pack(strings)
    d_bytes, d_offs = _to_device(data, offs)
    out, res = _both(cfg, d_bytes, d_offs, M, launches=_chunked_launches(cfg, len(strings), M, _max_smem(), per_pass=3))
    _vs_oracle(out, res, ocfg, data, offs)


@pytest.mark.gpu
def test_passes_s65535_huge():
    """S = 65535: 72 strings of 128 KiB hold 1.2 GB of level-0 transition vectors, more than one pass takes."""
    M = 128 * LONG_CHUNK + 1
    dfa = make_dfa(65535, 3, 65535 // 2, 7, "collapse_2", seed=5, alphabet=b"xyz")
    cfg = _product([dfa], M)
    np_rng = np.random.default_rng(7)
    lens = np_rng.integers(M // 2, M, 72)
    lens[:3] = [M - 1, 0, LONG_CHUNK]
    strings = [np.frombuffer(b"xyz", np.uint8)[np_rng.integers(0, 3, int(L))].tobytes() for L in lens]
    K = -(-M // LONG_CHUNK)
    per_pass = (1 << 30) // (K * 65536 * 2)
    assert per_pass < len(strings)
    data, offs = _pack(strings)
    d_bytes, d_offs = _to_device(data, offs)
    want = {"states", "substr_ids", "status", "mult"}
    out, res = _both(cfg, d_bytes, d_offs, M, want=want, launches=_chunked_launches(cfg, len(strings), M, _max_smem(), per_pass=per_pass))
    assert res.code == 0
    # the oracle on a few of the strings (its own batch)
    sample = [0, 1, 2, 40]
    sd, so = _pack([strings[j] for j in sample])
    o, _ = _oracle([dfa], M).match_batch(sd, so)
    h = out.to_host()
    for i, j in enumerate(sample):
        assert np.array_equal(h.states[0][j, :M], o.states[0][i, :M])


@pytest.mark.gpu
def test_large_batch_2048_x_64k_huge():
    """2048 strings of 64 KiB (regex1 with planted substrings): equal to b2r_match_batch on the device, and to the oracle on a
    seeded sample of strings."""
    import halo2_regex_b200 as H
    from halo2_regex_b200 import workloads as W
    M, n, L = 65537, 2048, 65536
    cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
    d = W.config1_torch(n, L)
    d_bytes = d.reshape(-1)
    import torch
    d_offs = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
    out, res = _both(cfg, d_bytes, d_offs, M, launches=_chunked_launches(cfg, n, M, _max_smem()))
    assert res.code == 0
    sample = sorted(random.Random(1).sample(range(n), 6))
    host = d.cpu().numpy()
    sd, so = _pack([host[j].tobytes() for j in sample])
    o, _ = ocfg.match_batch(sd, so, max_records=8, compact_pitch=64)
    h = out.to_host()
    for i, j in enumerate(sample):
        assert np.array_equal(h.states[0][j, :M], o.states[0][i, :M])
        assert np.array_equal(h.masked_chars[j, :M], o.masked_chars[i, :M])
        assert np.array_equal(h.substr_ids[0][j, :M], o.substr_ids[0][i, :M])
        for f in ("flags", "n_records", "n_compact"):
            assert h.status[f][j] == o.status[f][i]
    assert (h.status["flags"] & H._abi.B2R_ST_ACCEPTED(0)).any()


@pytest.mark.gpu
def test_side_stream_and_cuda_graph():
    """On a side stream, then captured once in a CUDA graph (after a first call of the same shape sized the workspace) and
    replayed twice with new bytes in the captured input buffer; each replay against b2r_match_batch and the oracle."""
    import torch
    import halo2_regex_b200 as H
    M = 5000
    rng = random.Random(31)
    lens = [rng.randrange(0, M) for _ in range(100)]
    cfg, ocfg = product_config("test1", M), oracle_config("test1", M)
    data, offs = _pack(_strings(rng, M, lens))
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_bytes, d_offs = _to_device(data, offs)
        out, res = _both(cfg, d_bytes, d_offs, M, stream=stream, launches=_chunked_launches(cfg, len(lens), M, _max_smem()))
    stream.synchronize()
    _vs_oracle(out, res, ocfg, data, offs)
    g_out = _outputs(cfg, len(lens))
    cfg.match_batch_chunked_device(d_bytes, d_offs, g_out)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cfg.match_batch_chunked_device(d_bytes, d_offs, g_out)
    for seed in (2, 3):
        r = random.Random(seed)
        data, _ = _pack(_strings(r, M, lens))
        d_bytes.copy_(torch.from_numpy(data.copy()))
        graph.replay()
        torch.cuda.synchronize()
        o, ores = ocfg.match_batch(data, offs, max_records=8, compact_pitch=64)
        assert ores.code == 0
        errs = H.compare_outputs(g_out.to_host(), o)
        assert errs == [], (seed, errs)
