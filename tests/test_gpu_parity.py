"""GPU (-m gpu): parity of the CUDA path, called through the C ABI, against the CPU oracle on identical inputs —
bit-exact for every witness column, status record, substring record and multiplicity counter."""
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, product_config
from test_oracle_golden import SNIPPETS, _random_strings, expected_masked

pytestmark = pytest.mark.gpu


def _pack(strings, lead=0):
    data = np.frombuffer(b"\x00" * lead + b"".join(strings), dtype=np.uint8)
    offs = np.zeros(len(strings) + 1, dtype=np.uint64)
    offs[0] = lead
    offs[1:] = lead + np.cumsum([len(s) for s in strings])
    return data, offs


def _both(set_name, M, strings, lead=0, check=True, **kw):
    import halo2_regex_b200 as H
    cfg = product_config(set_name, M)
    ocfg = oracle_config(set_name, M)
    data, offs = _pack(strings, lead)
    kw.setdefault("max_records", 8)
    kw.setdefault("compact_pitch", 64)
    g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, **kw)
    o, ores = ocfg.match_batch(data, offs, **kw)
    assert gres.code == ores.code
    if ores.code != 0:
        assert (gres.string_idx, gres.pos, gres.state, gres.byte, gres.defidx) == (ores.string_idx, ores.pos, ores.state, ores.byte, ores.defidx)
    assert gres.n_overlap_lo == ores.n_overlap_lo
    errs = H.compare_outputs(g, o)
    assert errs == [], "\n".join(errs)
    return cfg, g, o


def test_golden_vectors_on_gpu(golden_vectors):
    """G1-G9 straight through the product API (the reference tests' own expectations)."""
    import halo2_regex_b200 as H
    for v in golden_vectors:
        cfg = product_config(v["defs"], v["M"])
        r = cfg.match_substrs(v["input"].encode())
        assert all(r.accepted) == v["verify_ok"], v["name"]
        if v["substrs"] is not None:
            mc, ms = expected_masked(v)
            assert np.array_equal(r.masked_characters, mc), v["name"]       # src/lib.rs:1052-1059
            assert np.array_equal(r.all_substr_ids, ms), v["name"]
            assert r.substr_bytes == "".join(s for _, s in v["substrs"]).encode()
        assert len(r.all_enable_flags) == v["M"] and int(r.all_enable_flags.sum()) == len(v["input"])
        _both(v["defs"], v["M"], [v["input"].encode()])


def test_derive_helpers_match_reference_shapes():
    cfg = product_config("example", 128)
    s = b"email was meant for @vitalik."
    st = cfg.derive_states(s)
    assert len(st) == 1 and len(st[0]) == len(s) + 1 and st[0][0] == 0 and st[0][-1] == 2
    ids = cfg.derive_substr_ids(s)
    assert ids[0] == [0] * 21 + [1] * 7 + [0]
    is_starts, is_ends = cfg.derive_is_start_end(s)
    assert len(is_starts[0]) == len(s) + 1 and len(is_ends[0]) == len(s) + 1
    assert [i for i, x in enumerate(is_starts[0]) if x] == [21]
    assert is_ends[0][0] is False


@pytest.mark.parametrize("set_name", ["regex1", "regex2", "regex3", "test1", "regex3_k3", "three"])
def test_random_ragged_batches(set_name):
    rng = random.Random(zlib.crc32(set_name.encode()) + 1)
    strings = _random_strings(rng, 700, 200, SNIPPETS) + [b"", b"", b"x"]
    _both(set_name, 201, strings)


@pytest.mark.parametrize("lead", [0, 1, 7, 16, 33])
def test_unaligned_offsets(lead):
    rng = random.Random(lead)
    strings = _random_strings(rng, 100, 130, SNIPPETS)
    _both("test1", 131, strings, lead=lead)


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 63, 65, 1000])
def test_batch_sizes(n):
    rng = random.Random(n)
    _both("regex1", 100, _random_strings(rng, n, 99, SNIPPETS))


def test_empty_batch_and_empty_strings():
    _both("regex1", 64, [])
    _both("regex1", 64, [b""] * 40)
    _both("regex3", 1, [b""] * 3)          # M = 1: only the final-state row exists


@pytest.mark.parametrize("M", [16, 17, 63, 64, 65, 128, 129, 1024, 1025])
def test_max_length_strings(M):
    """len = M-1 is the longest legal string: the final state lands in the last row (src/lib.rs:404-418)."""
    rng = random.Random(M)
    strings = [bytes(rng.choice(b"abc @.\r\n") for _ in range(M - 1)) for _ in range(5)]
    strings += [b"email was meant for @ab." + b"z" * (M - 25) if M >= 25 else b"q" * (M - 1)]
    _both("test1", M, strings)


def test_config1_shape_fixed_length():
    """BASELINE config 1 at reduced N: 1 KiB strings, M = 1025, regex1+substr1."""
    from halo2_regex_b200 import workloads as W
    data, _ = W.config1_numpy(2048, 1024)
    strings = [bytes(r) for r in data]
    cfg, g, o = _both("regex1", 1025, strings, compact_pitch=8)
    acc = (g.status["flags"] & 1).astype(bool)
    assert 0.9 < acc.mean() < 0.97          # 15 in 16 strings carry a match
    assert int(g.mult[0].sum()) == 2048 * 1025


def test_config1_ragged():
    from halo2_regex_b200 import workloads as W
    data, _ = W.config1_numpy(1024, 1024)
    flat, offs = W.ragged_from_fixed(data, 99)
    strings = [bytes(flat[int(offs[i]):int(offs[i + 1])]) for i in range(1024)]
    _both("regex1", 1025, strings)


def test_invalid_transition_reports_reference_panic():
    import halo2_regex_b200 as H
    good = b"email was meant for @vitalik."
    strings = [good, good[:10] + b"X" + good[11:], good, b"\xff"]
    cfg, g, o = _both("example", 64, strings)
    assert g.status["flags"][1] & H._abi.B2R_ST_INVALID_TRANSITION
    with pytest.raises(H.InvalidTransitionError, match=r"The transition from \d+ by 88 is invalid!"):
        cfg.match_strings(strings)
    # lowest def wins even when a later def fails earlier in the string (derive_states walks def 0 first)
    spec = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"]), ("ex_allstr.txt", ["ex_substr_id1.txt"])]
    _both(spec, 64, [b"zz\x01", b"email was \x01", b"email was meant for @vitalik."])
    spec.reverse()
    _both(spec, 64, [b"zz\x01", b"email was \x01", b"email was meant for @vitalik."])


def test_too_long_string():
    import halo2_regex_b200 as H
    cfg, g, o = _both("regex1", 16, [b"a" * 15, b"a" * 16, b"b" * 3])
    assert g.status["flags"][1] & H._abi.B2R_ST_TOO_LONG
    with pytest.raises(H.StringTooLongError):
        cfg.match_strings([b"a" * 16])


def test_long_substrings_and_multi_run_segments():
    """Dense substring coverage (long masked stretches, vector fill path) and hand-made defs whose id sum changes
    inside a masked segment without a flag (the re-walk path)."""
    import halo2_regex_b200 as H
    from oracle import oracle as O
    allstr = b"0\n3\n3\n" + b"".join(f"{s} {t} {c}\n".encode() for s, t, c in [
        (0, 0, 120), (0, 1, 97), (1, 1, 97), (1, 2, 98), (2, 2, 98), (2, 3, 99), (3, 3, 120), (3, 1, 97), (2, 1, 97), (1, 3, 99),
        (0, 0, 98), (0, 0, 99), (1, 0, 120), (2, 0, 120), (3, 3, 98), (3, 3, 99)])
    # substr A covers a-runs, substr B covers b-runs; start only at 0->1 / 3->1, end only at ->3: A,B alternate unflagged
    sub_a = b"9\n0\n9\n0 3\n3\n0 1\n1 1\n3 1\n1 3\n2 1\n"
    sub_b = b"9\n0\n9\n\n3\n1 2\n2 2\n2 3\n"
    rng = random.Random(5)
    strings = [bytes(rng.choice(b"xaabbc") for _ in range(rng.randrange(0, 300))) for _ in range(300)]
    strings += [b"x" + b"a" * 250 + b"c", b"a" * 100 + b"b" * 100 + b"c" + b"x" * 20, b"aabbaabbc", b"aabb"]
    M = 301
    pa = H.AllstrRegexDef.read_from_reader(allstr)
    cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(pa, [H.SubstrRegexDef.read_from_reader(sub_a), H.SubstrRegexDef.read_from_reader(sub_b)])])
    ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(sub_a), O.OracleSubstr(sub_b)])], M)
    data, offs = _pack(strings)
    g, gres = cfg.match_batch_host(data, offs, max_records=16, compact_pitch=512, fill=0xCD)
    o, ores = ocfg.match_batch(data, offs, max_records=16, compact_pitch=512)
    assert H.compare_outputs(g, o) == []
    assert (g.status["n_records"] > 1).any() and (g.status["n_compact"] > 200).any()


def test_overlapping_defs_are_flagged():
    """Two defs flagging the same row: out of the reference's boolean domain (SURVEY 8(a) out-of-domain ii)."""
    import halo2_regex_b200 as H
    spec = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"]), ("regex1_test_lookup.txt", ["substr1_test_lookup.txt"])]
    cfg, g, o = _both(spec, 64, [b"email was meant for @ab.", b"nothing here", b" email was meant for @q. "])
    assert g.status["flags"][0] & H._abi.B2R_ST_OVERLAP and not g.status["flags"][1] & H._abi.B2R_ST_OVERLAP


def test_null_columns_and_truncation():
    rng = random.Random(21)
    strings = _random_strings(rng, 200, 150, SNIPPETS)
    for want in ({"status", "masked_chars"}, {"states", "status", "mult"}, {"status", "records", "compact_bytes", "masked_substr_ids"},
                 {"start_enable", "end_enable", "status", "endpoint_mult"}):
        _both("test1", 151, strings, want=want)
    _both("regex3", 151, strings, max_records=1, compact_pitch=3)      # truncation flags and exact counts


def test_accumulate_multiplicities():
    import halo2_regex_b200 as H
    rng = random.Random(8)
    a, b = _random_strings(rng, 150, 90, SNIPPETS), _random_strings(rng, 170, 90, SNIPPETS)
    cfg, ocfg = product_config("test1", 91), oracle_config("test1", 91)
    g, _ = cfg.match_strings(a)
    g, _ = cfg.match_strings(b, out=cfg.new_host_outputs(len(b)), flags=0)
    da, oa = _pack(a)
    db, ob = _pack(b)
    out = cfg.new_host_outputs(len(b))
    first, _ = cfg.match_batch_host(da, oa)
    for d in range(2):
        out.mult[d][:] = first.mult[d]
        out.endpoint_mult[d][:] = first.endpoint_mult[d]
    cfg.match_batch_host(db, ob, out=out, flags=H._abi.B2R_OUT_ACCUMULATE_MULT)
    o, _ = ocfg.match_strings(a + b)
    for d in range(2):
        assert np.array_equal(out.mult[d], o.mult[d])
        assert np.array_equal(out.endpoint_mult[d], o.endpoint_mult[d])
        assert int(out.mult[d].sum()) == (len(a) + len(b)) * 91


def test_device_pointer_entry_point():
    """b2r_match_batch with device tensors on a non-default stream; outputs copied back and compared."""
    import torch
    import halo2_regex_b200 as H
    rng = random.Random(77)
    strings = _random_strings(rng, 3000, 120, SNIPPETS)
    cfg, ocfg = product_config("three", 121), oracle_config("three", 121)
    data, offs = _pack(strings)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_bytes = torch.from_numpy(data.copy()).cuda()
        d_offs = torch.from_numpy(offs.astype(np.int64)).cuda()
        out = H.DeviceOutputs(cfg, len(strings), max_records=8, compact_pitch=64)
        cfg.match_batch_device(d_bytes, d_offs, out, stream=stream)
        res = cfg.batch_result(stream=stream)
    assert res.code == 0 and cfg.last_launch_count() == 3      # three defs: walk (+ zero-fill), emit, finalize
    o, _ = ocfg.match_batch(data, offs, max_records=8, compact_pitch=64)
    assert H.compare_outputs(out.to_host(), o) == []


@pytest.mark.parametrize("table_mode,hist_mode", [("repl", "smem"), ("plain", "smem"), ("plain16", "smem"), ("repl", "global"), ("plain16", "global"), ("global", "global"),
                                                  ("repl16", "smem"), ("repl16", "global")])
@pytest.mark.parametrize("set_name", ["regex1", "three"])
def test_table_and_bin_placements(monkeypatch, set_name, table_mode, hist_mode):
    """Every placement of the walk tables (bank-replicated / single copy in shared memory, global) and of the
    multiplicity bins gives the same bits (the library picks by shared-memory budget; here they are forced)."""
    monkeypatch.setenv("B2R_TABLE_MODE", table_mode)
    monkeypatch.setenv("B2R_HIST_MODE", hist_mode)
    rng = random.Random(zlib.crc32((set_name + table_mode + hist_mode).encode()))
    strings = _random_strings(rng, 300, 260, SNIPPETS) + [b"", b"q"]
    cfg, g, o = _both(set_name, 261, strings)
    if not (set_name == "three" and table_mode == "repl"):      # three replicated tables exceed shared memory: the launcher says so
        assert cfg.last_plan()[0] == table_mode


@pytest.mark.parametrize("set_name,fuse", [("regex1", 0), ("test1", 0), ("regex3_k3", 0), ("three", 0), ("three", 1), ("regex1", 1), ("three", 2), ("regex1", 2), ("test1", 2)])
def test_emit_stage_fused_and_separate(monkeypatch, set_name, fuse):
    """B2R_FUSE=1: the emit stage inside walk_kernel, tile by tile (the default for one or two defs); 2: the walk zero-fills, the emit
    stage scans as its own kernel (the default for three or more); 0: the emit kernel does both."""
    monkeypatch.setenv("B2R_FUSE", str(fuse))
    rng = random.Random(zlib.crc32(set_name.encode()) + 7)
    strings = _random_strings(rng, 500, 300, SNIPPETS) + [b"", b"zz"]
    cfg, g, o = _both(set_name, 301, strings)
    assert cfg.last_launch_count() == (2 if fuse == 1 else 3)


def test_offset_warp_starts(monkeypatch):
    """B2R_STAGGER_NS: the warps of a walk CTA start at different times (the default only does this on large batches)."""
    monkeypatch.setenv("B2R_STAGGER_NS", "2000")
    rng = random.Random(5)
    strings = _random_strings(rng, 700, 200, SNIPPETS)
    _both("regex1", 201, strings)
    _both("three", 201, strings)


FOUR_DEFS = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"]), ("regex2_test_lookup.txt", ["substr2_test_lookup.txt"]),
             ("regex3_test_lookup.txt", ["substr3_test_lookup.txt"]), ("regex3_test_lookup.txt", ["substr1_test_lookup.txt", "substr2_test_lookup.txt"])]


@pytest.mark.parametrize("fuse", [1, 2, 0])
def test_four_defs(monkeypatch, fuse):
    """B2R_MAX_DEFS defs in one config (the emit kernel's per-thread scratch is at its largest)."""
    monkeypatch.setenv("B2R_FUSE", str(fuse))
    rng = random.Random(404 + fuse)
    strings = _random_strings(rng, 400, 260, SNIPPETS) + [b"", b"x"]
    _both(FOUR_DEFS, 261, strings)


def test_default_emit_placement():
    rng = random.Random(11)
    strings = _random_strings(rng, 200, 120, SNIPPETS)
    for set_name, launches in (("regex1", 2), ("test1", 3), ("three", 3)):
        cfg, g, o = _both(set_name, 121, strings)
        assert cfg.last_launch_count() == launches, set_name


def test_wide_state_column():
    """> 255 states: the state column becomes u16 (SURVEY 8(d) w_s = 2)."""
    import halo2_regex_b200 as H
    from oracle import oracle as O
    S = 300
    lines = [f"0\n{S - 1}\n{S - 1}\n"]
    for s in range(S):
        for c in (97, 98, 99):
            nxt = (s + 1) % S if c == 97 else (s * 7 + 3) % S if c == 98 else s
            lines.append(f"{s} {nxt} {c}\n")
    allstr = "".join(lines).encode()
    sub = b"5\n0\n9\n10 20\n11 21 30\n10 11\n20 21\n11 12\n21 22\n12 13\n29 30\n28 29\n"
    rng = random.Random(4)
    strings = [bytes(rng.choice(b"aaaabc") for _ in range(rng.randrange(0, 400))) for _ in range(200)] + [b"a" * 399]
    M = 400
    cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(sub)])])
    assert cfg.state_widths == [2]
    ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(sub)])], M)
    data, offs = _pack(strings)
    g, _ = cfg.match_batch_host(data, offs, fill=0xCD)
    o, _ = ocfg.match_batch(data, offs)
    assert H.compare_outputs(g, o) == []
    assert int(g.states[0].max()) > 255


def _wide_allstr(S=300):
    lines = [f"0\n{S - 1}\n{S - 1}\n"]
    for s in range(S):
        for c in range(32, 127):
            nxt = (s + 1) % S if c == 97 else (s * 7 + c) % S if c % 5 == 0 else s
            lines.append(f"{s} {nxt} {c}\n")
    return "".join(lines).encode()


@pytest.mark.parametrize("order", ["narrow_first", "wide_first"])
def test_mixed_state_widths_share_one_width(order):
    """A def with <= 255 states next to one with more: every state column of the config is stored as u16."""
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from conftest import read
    wide = (_wide_allstr(), [b"5\n0\n63\n10 \n13 \n10 11\n11 12\n12 13\n"])
    narrow = (read("regex1_test_lookup.txt"), [read("substr1_test_lookup.txt")])
    spec = [narrow, wide] if order == "narrow_first" else [wide, narrow]
    M = 200
    cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(a), [H.SubstrRegexDef.read_from_reader(x) for x in ss])
                                            for a, ss in spec])
    assert cfg.state_widths == [2, 2]
    ocfg = O.OracleConfig([(O.OracleAllstr(a), [O.OracleSubstr(x) for x in ss]) for a, ss in spec], M)
    assert ocfg.state_widths == [2, 2]
    rng = random.Random(9)
    strings = [bytes(rng.choice(b"aaaa bcdexyz@.") for _ in range(rng.randrange(0, M))) for _ in range(300)]
    strings += [b"x" * 5 + s + b"a" * rng.randrange(0, 40) for s in SNIPPETS[:4]]
    data, offs = _pack(strings)
    g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, max_records=8, compact_pitch=16)
    o, ores = ocfg.match_batch(data, offs, max_records=8, compact_pitch=16)
    assert gres.code == ores.code
    assert H.compare_outputs(g, o) == []
    assert int(g.states[0 if order == "wide_first" else 1].max()) > 255


def test_multiplicity_invariant_full_size_property():
    """Size-independent property at a larger N (oracle too slow to be the checker): sum(mult) = N*M, row 0 = padded
    rows, accepted fraction as planted, masked bytes equal the planted names."""
    import torch
    import halo2_regex_b200 as H
    from halo2_regex_b200 import workloads as W
    N, L, M = 1 << 15, 1024, 1025
    cfg = product_config("regex1", M)
    d_bytes = W.config1_torch(N, L, device="cuda").reshape(-1)
    d_offs = torch.arange(N + 1, dtype=torch.int64, device="cuda") * L
    out = H.DeviceOutputs(cfg, N, compact_pitch=8, max_records=2)
    cfg.match_batch_device(d_bytes, d_offs, out)
    assert cfg.batch_result().code == 0
    mult = out.mult[0].cpu().numpy().astype(np.uint64)
    assert int(mult.sum()) == N * M and int(mult[0]) == N * (M - L)
    h_data, plan = W.config1_numpy(N, L)
    status = out.status.cpu().numpy().view(H._abi.STATUS_DTYPE).reshape(-1)
    acc = (status["flags"] & 1).astype(bool)
    assert np.array_equal(acc | ~plan["has_match"], np.ones(N, bool))
    mc = out.masked_chars.cpu().numpy()
    j = int(np.nonzero(plan["has_match"])[0][5])
    o, nl = int(plan["offset"][j]) + 21, int(plan["name_len"][j])
    assert bytes(mc[j, o:o + nl]) == bytes(h_data[j, o:o + nl])


@pytest.mark.parametrize("set_name,length", [("regex2", 0), ("regex2", 1), ("regex2", 1023), ("regex2", 1024), ("regex2", 1025), ("regex2", 70000),
                                             ("regex1", 5000), ("test1", 40000), ("regex3_k3", 3333)])
def test_long_string_path(set_name, length):
    """b2r_match_long (BASELINE config 3 at reduced size): one string cut into 1 KiB chunks, transition vectors composed by
    parallel prefix, chunk walks from the resolved entry states, ordered emit - against the oracle on the same single string
    with max_chars_size = len + 1."""
    import torch
    import halo2_regex_b200 as H
    rng = random.Random(length * 7 + len(set_name))
    alphabet = bytes([9, 10, 13] + list(range(32, 127)))
    body = bytearray(rng.choice(alphabet) for _ in range(length))
    for snip in SNIPPETS:                                   # plant matches, some of them across chunk boundaries
        for _ in range(3):
            if length > len(snip) + 2:
                at = rng.choice([rng.randrange(0, length - len(snip)), max(0, min(length - len(snip), 1024 * rng.randrange(0, length // 1024 + 1) - rng.randrange(0, len(snip))))])
                body[at:at + len(snip)] = snip
    s = bytes(body)
    M = length + 1
    cfg, ocfg = product_config(set_name, 64), oracle_config(set_name, M)      # the handle's own max_chars_size is ignored
    d = torch.from_numpy(np.frombuffer(s + b"\0" * 16, dtype=np.uint8).copy()).cuda()[:length]
    out = H.DeviceOutputs(cfg, 1, max_records=64, compact_pitch=256, max_chars_size=M)
    cfg.match_long_device(d, out)
    res = cfg.batch_result(check=False)
    data, offs = _pack([s])
    o, ores = ocfg.match_batch(data, offs, max_records=64, compact_pitch=256)
    assert res.code == ores.code
    assert H.compare_outputs(out.to_host(), o) == []


@pytest.mark.parametrize("set_name,length", [("regex1", 0), ("regex1", 5000), ("test1", 70001), ("regex3", 1024)])
def test_long_string_host_entry_point(set_name, length):
    """b2r_match_long_host: host bytes in, host columns out, same answer as the oracle with max_chars_size = len + 1."""
    rng = random.Random(length + 5)
    body = bytearray(rng.choice(b"abc xyz.@\r\n") for _ in range(length))
    for snip in SNIPPETS[:5]:
        if length > 200:
            at = rng.randrange(0, length - len(snip))
            body[at:at + len(snip)] = snip
    s = bytes(body)
    M = length + 1
    cfg = product_config(set_name, 64)
    ocfg = oracle_config(set_name, M)
    g, gres = cfg.match_long_host(s, check=False, max_records=8, compact_pitch=64, fill=0xCD)
    data, offs = _pack([s])
    o, ores = ocfg.match_batch(data, offs, max_records=8, compact_pitch=64)
    assert (gres.code, gres.pos, gres.state, gres.byte) == (ores.code, ores.pos, ores.state, ores.byte)
    import halo2_regex_b200 as H
    assert H.compare_outputs(g, o) == []


def test_long_string_16_mib_bit_exact():
    """A quarter of BASELINE config 3 (one 16 MiB string, 16 385 chunks, three tree levels) against the oracle, every column."""
    import halo2_regex_b200 as H
    rng = np.random.default_rng(0xB2000003)
    length = 1 << 24
    alphabet = np.array([9, 10, 13] + list(range(32, 127)), dtype=np.uint8)
    body = alphabet[rng.integers(0, len(alphabet), length)]
    plant = np.frombuffer(b" Also for xyzzy.", dtype=np.uint8)
    for at in [0, 1013, 1020, 65530, (1 << 22) - 7, length - len(plant)] + list(rng.integers(0, length - 64, 200)):
        body[at:at + len(plant)] = plant                       # some straddle chunk and tree-node boundaries
    s = body.tobytes()
    M = length + 1
    cfg = product_config("regex2", 64)
    ocfg = oracle_config("regex2", M)
    g, gres = cfg.match_long_host(s, check=False, max_records=8, compact_pitch=64)
    data, offs = _pack([s])
    o, ores = ocfg.match_batch(data, offs, max_records=8, compact_pitch=64)
    assert gres.code == ores.code == 0
    assert H.compare_outputs(g, o) == []
    assert int(g.mult[0].sum()) == M


def test_long_string_64_mib_bit_exact():
    """BASELINE config 3 at its full size (one 64 MiB string through regex2, 65 536 chunks, 256 groups, 8 super groups) against the
    oracle, every column; the planted match and a few more straddle chunk, group and super-group boundaries."""
    import halo2_regex_b200 as H
    import workloads as W
    length = 1 << 26
    body, at = W.config3_numpy(length)
    plant = np.frombuffer(b" Also for xyzzy.", dtype=np.uint8)
    for pos in [0, 1013, (1 << 18) - 5, (1 << 23) - 9, (1 << 25) + 1020, length - len(plant)]:
        body[pos:pos + len(plant)] = plant
    M = length + 1
    cfg = product_config("regex2", 64)
    g, gres = cfg.match_long_host(body, check=False, max_records=16, compact_pitch=128)
    o, ores = oracle_config("regex2", M).match_batch(body, np.array([0, length], dtype=np.uint64), max_records=16, compact_pitch=128)
    assert gres.code == ores.code == 0
    assert H.compare_outputs(g, o) == []
    assert int(g.mult[0].sum()) == M and int(g.status["n_records"][0]) >= 1


@pytest.mark.parametrize("fused", [0, 1])
@pytest.mark.parametrize("length", [1, 4097, 300000])
def test_long_string_counter_dfa_never_collapses(length, fused):
    """A DFA whose states never merge (x: s -> s+1 mod 7, y: s -> s): every chunk keeps 7 distinct images, so the fused prefix pass
    stays on its all-states rounds and the general pass on its wide-chunk path; both against the oracle.  Also the shipped DFAs
    through the general (multi-kernel) pass, which the fused one replaces by default."""
    import torch
    import halo2_regex_b200 as H
    from oracle import oracle as O
    S = 7
    allstr = f"0\n3\n{S - 1}\n" + "".join(f"{s} {(s + 1) % S} {ord('x')}\n{s} {s} {ord('y')}\n" for s in range(S))
    substr = "64\n0\n64\n2\n5\n2 3\n3 4\n4 5\n3 3\n4 4\n"
    rng = random.Random(length)
    s = bytes(rng.choice(b"xyyy") for _ in range(length))
    M = length + 1
    cfg = H.RegexVerifyConfig.configure(64, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr.encode()), [H.SubstrRegexDef.read_from_reader(substr.encode())])])
    cfg.set_option("long_fused", fused)
    ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], M)
    g, gres = cfg.match_long_host(s, check=False, max_records=16, compact_pitch=128)
    data, offs = _pack([s])
    o, ores = ocfg.match_batch(data, offs, max_records=16, compact_pitch=128)
    assert gres.code == ores.code == 0
    assert H.compare_outputs(g, o) == []
    # the shipped DFAs through the other pass
    for set_name in ("regex2", "test1"):
        body = bytearray(rng.choice(b"abc xyz.@\r\n") for _ in range(length))
        for snip in SNIPPETS[:6]:
            if length > 200:
                at = rng.randrange(0, length - len(snip))
                body[at:at + len(snip)] = snip
        c2 = product_config(set_name, 64)
        c2.set_option("long_fused", fused)
        g2, r2 = c2.match_long_host(bytes(body), check=False, max_records=16, compact_pitch=128)
        d2, f2 = _pack([bytes(body)])
        o2, or2 = oracle_config(set_name, M).match_batch(d2, f2, max_records=16, compact_pitch=128)
        assert r2.code == or2.code and H.compare_outputs(g2, o2) == []


def test_long_string_invalid_transition():
    import torch
    import halo2_regex_b200 as H
    s = b"email was meant for @vitalik." * 3 + b"\x01" + b"abc" * 2000
    M = len(s) + 1
    cfg, ocfg = product_config("regex1", 64), oracle_config("regex1", M)
    d = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda()
    out = H.DeviceOutputs(cfg, 1, max_chars_size=M)
    cfg.match_long_device(d, out)
    res = cfg.batch_result(check=False)
    data, offs = _pack([s])
    o, ores = ocfg.match_batch(data, offs)
    assert res.code == ores.code == H._abi.B2R_ERR_INVALID_TRANSITION
    assert (res.pos, res.state, res.byte) == (ores.pos, ores.state, ores.byte)


@pytest.mark.parametrize("set_name", ["regex3", "regex3_k3", "three"])
def test_config2_shape(set_name):
    """BASELINE config 2 at reduced N: from: header lines through regex3 — reading (i) regex3 + substr1..3 in one RegexDefs,
    reading (ii) three RegexDefs (SURVEY 8(d))."""
    from halo2_regex_b200 import workloads as W
    data, plan = W.config2_numpy(768, 1024)
    strings = [bytes(r) for r in data]
    cfg, g, o = _both(set_name, 1025, strings, compact_pitch=32)
    d = len(DEF_SETS[set_name]) - 1
    assert ((g.status["flags"] >> d) & 1).all()                      # every string ends in a well-formed from: line
    j = 5
    a0 = int(plan["addr_start"][j])
    addr = bytes(plan["addr"][j]).rstrip(b"\0")
    assert bytes(g.masked_chars[j, a0:a0 + len(addr)]) == addr


def test_config4_large_dfa():
    """BASELINE config 4 at reduced N: a synthetic DFA with 1023 states in the reference's text format (2-byte state column,
    tables beyond the replicated shared-memory layout), 4 KiB strings."""
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from halo2_regex_b200 import workloads as W
    allstr, substr, info = W.large_dfa_texts()
    assert info["states"] >= 512
    M = 4097
    cfg = H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
    assert cfg.state_widths == [2]
    ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], M)
    data, plan = W.config4_numpy(96, 4096)
    flat, offs = data.reshape(-1), np.arange(97, dtype=np.uint64) * 4096
    g, gres = cfg.match_batch_host(flat, offs, max_records=4, compact_pitch=64, fill=0xCD)
    o, ores = ocfg.match_batch(flat, offs, max_records=4, compact_pitch=64)
    assert gres.code == ores.code == 0
    assert H.compare_outputs(g, o) == []
    assert np.array_equal((g.status["flags"] & 1).astype(bool), plan["has_from"])


@pytest.mark.parametrize("which,log2n", [("regex1", 20), ("three", 17), ("regex3_k3", 17), ("large_dfa", 15)])
def test_large_batches_against_tiled_oracle(which, log2n):
    """Sizes the oracle cannot walk in seconds: the batch is `base` distinct strings tiled N/base times, so every
    multiplicity counter must be exactly N/base times the oracle's over the base strings (a checksum over all N*M rows),
    and every column of a sample of rows (first, last and a few tiles in between) must equal the oracle's."""
    import torch
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from halo2_regex_b200 import workloads as W
    base, N = 256, 1 << log2n
    if which == "large_dfa":
        L = 4096
        allstr, substr, _ = W.large_dfa_texts()
        cfg = H.RegexVerifyConfig.configure(L + 1, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
        ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], L + 1)
        data, _ = W.config4_numpy(base, L)
    else:
        L = 1024
        cfg, ocfg = product_config(which, L + 1), oracle_config(which, L + 1)
        data, _ = W.config1_numpy(base, L) if which == "regex1" else W.config2_numpy(base, L)      # regex1, 2^20: BASELINE config 1 in full
    M = L + 1
    d_bytes = torch.from_numpy(data).cuda().repeat(N // base, 1).reshape(-1).contiguous()
    d_offs = torch.arange(N + 1, dtype=torch.int64, device="cuda") * L
    out = H.DeviceOutputs(cfg, N, compact_pitch=32, max_records=4)
    cfg.match_batch_device(d_bytes, d_offs, out)
    assert cfg.batch_result().code == 0
    o, ores = ocfg.match_batch(data.reshape(-1), np.arange(base + 1, dtype=np.uint64) * L, max_records=4, compact_pitch=32)
    assert ores.code == 0
    for d in range(cfg.n_defs):
        mult = out.mult[d].cpu().numpy().astype(np.uint64)
        assert int(mult.sum()) == N * M
        assert np.array_equal(mult, o.mult[d].astype(np.uint64) * np.uint64(N // base)), d
        em = out.endpoint_mult[d].cpu().numpy().astype(np.uint64)
        assert np.array_equal(em, o.endpoint_mult[d].astype(np.uint64) * np.uint64(N // base)), d
    for t in (0, 1, N // base // 2, N // base - 1):          # tile t of the batch == the base strings again
        lo = t * base
        for d in range(cfg.n_defs):
            assert np.array_equal(out.states[d][lo:lo + base, :M].cpu().numpy().view(o.states[d].dtype), o.states[d][:, :M]), (t, d)
            assert np.array_equal(out.substr_ids[d][lo:lo + base, :M].cpu().numpy(), o.substr_ids[d][:, :M]), (t, d)
            assert np.array_equal(out.start_enable[d][lo:lo + base].cpu().numpy()[:, :(M + 7) // 8], o.start_enable[d][:, :(M + 7) // 8]), (t, d)
            assert np.array_equal(out.end_enable[d][lo:lo + base].cpu().numpy()[:, :(M + 7) // 8], o.end_enable[d][:, :(M + 7) // 8]), (t, d)
        assert np.array_equal(out.masked_chars[lo:lo + base, :M].cpu().numpy(), o.masked_chars[:, :M]), t
        assert np.array_equal(out.masked_substr_ids[lo:lo + base, :M].cpu().numpy(), o.masked_substr_ids[:, :M]), t
        st = out.status[lo:lo + base].cpu().numpy().view(H._abi.STATUS_DTYPE).reshape(-1)
        assert np.array_equal(st["flags"], o.status["flags"]), t


def test_host_entry_point_slices():
    """b2r_match_batch_host cuts large batches into slices (H2D / kernels / D2H overlap on three streams): same bits, the
    multiplicities of the slices add up, and the batch result is the lowest failing string over all slices."""
    rng = random.Random(99)
    strings = _random_strings(rng, 20000, 60, SNIPPETS)
    _both("test1", 61, strings)
    bad = list(strings)
    bad[17000] = b"email \x01"
    bad[9000] = b"\x02"
    cfg, g, o = _both("test1", 61, bad)
    import halo2_regex_b200 as H
    assert g.status["flags"][9000] & H._abi.B2R_ST_INVALID_TRANSITION and g.status["flags"][17000] & H._abi.B2R_ST_INVALID_TRANSITION


@pytest.mark.parametrize("set_name,M", [("regex1", 257), ("test1", 130), ("regex3_k3", 513), ("three", 100), ("example", 64)])
def test_fuzz_many_strings(set_name, M):
    """Differential fuzz at a larger count: 30 000 random ragged strings (snippets of the regexes spliced into alphabet noise,
    some with bytes outside the alphabet) per definition set, every column against the oracle."""
    rng = random.Random(zlib.crc32(f"{set_name}/{M}".encode()))
    strings = _random_strings(rng, 30000, M - 1, SNIPPETS)
    if set_name != "example":            # a few invalid bytes: the batch fails like the reference, per-string statuses must still agree
        for k in range(0, 30000, 7919):
            s = bytearray(strings[k] or b"x")
            s[rng.randrange(len(s))] = rng.choice([0, 1, 127, 200, 255])
            strings[k] = bytes(s)
    _both(set_name, M, strings)
