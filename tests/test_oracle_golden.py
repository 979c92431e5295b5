"""CPU: pins the oracle (oracle/oracle.c) against the reference's own known-answer vectors and against the second,
independently written Python restatement (oracle/pyref.py).  No GPU, no product code."""
import random
import zlib

import numpy as np
import pytest

from conftest import DEF_SETS, oracle_config, pyref_defs, read
from oracle import pyref as P

from halo2_regex_b200 import _abi
from halo2_regex_b200.workloads import ALPHABET


def expected_masked(v):
    M = v["M"]
    mc, ms = np.zeros(M, np.uint8), np.zeros(M, np.uint8)
    for k, (start, s) in enumerate(v["substrs"] or []):
        mc[start:start + len(s)] = np.frombuffer(s.encode(), np.uint8)      # src/lib.rs:1046-1051
        ms[start:start + len(s)] = k + 1
    return mc, ms


def test_golden_vectors(golden_vectors):
    """G1-G9: masked_characters / all_substr_ids literal expectations and verify() pass/fail of the reference tests."""
    for v in golden_vectors:
        cfg = oracle_config(v["defs"], v["M"])
        out, res = cfg.match_strings([v["input"].encode()])
        assert res.code == 0, v["name"]
        accepted = all(out.status["flags"][0] & _abi.B2R_ST_ACCEPTED(d) for d in range(cfg.n_defs))
        # every reference test satisfies all lookups/gates except (in the fail tests) the accept rule
        w = P.match_substrs(pyref_defs(v["defs"]), v["M"], v["input"].encode())
        cons_ok, _ = P.check_constraints(pyref_defs(v["defs"]), v["M"], w)
        assert cons_ok, v["name"]
        assert accepted == v["verify_ok"], v["name"]
        if v["substrs"] is not None:
            mc, ms = expected_masked(v)
            assert np.array_equal(out.masked_chars[0, :v["M"]], mc), v["name"]
            assert np.array_equal(out.masked_substr_ids[0, :v["M"]], ms), v["name"]
        assert not (out.status["flags"][0] & _abi.B2R_ST_OVERLAP)


def test_golden_states_survey():
    """Facts derived in SURVEY.md section 4 (final states; G9 state list)."""
    cfg = oracle_config("example", 128)
    s = b"email was meant for @vitalik."
    out, _ = cfg.match_strings([s])
    states = list(out.states[0][0, :len(s) + 1])
    assert states[0] == 0 and states[1:3] == [3, 4] and states[21] == 23 and states[22:29] == [1] * 7 and states[29] == 2
    assert list(out.states[0][0, len(s) + 1:128]) == [24] * (127 - len(s))    # dummy = largest_state_val + 1
    cfg = oracle_config("test1", 1024)
    for text, finals in ((b"email was meant for @y. Also for x.", (24, 12)), (b"email was meant for @@", (0, 0))):
        out, _ = cfg.match_strings([text])
        assert (int(out.states[0][0, len(text)]), int(out.states[1][0, len(text)])) == finals
    cfg = oracle_config("regex3", 1024)
    for text, final in ((b"from:alice@gmail.com\r\n", 5), (b"from:alice<alicegmail.com>\r\n", 9), (b"from:alice<alice@gmail.com>", 19),
                        (b"fromalice<alice@gmail.com>\r\n", 9)):
        out, _ = cfg.match_strings([text])
        assert int(out.states[0][0, len(text)]) == final


def _compare_with_pyref(set_name, M, strings, cfg=None, pdefs=None):
    """set_name: a DEF_SETS entry, or None with `cfg` (an OracleConfig) and `pdefs` (the same defs for pyref) given."""
    cfg = cfg if cfg is not None else oracle_config(set_name, M)
    pdefs = pdefs if pdefs is not None else pyref_defs(set_name)
    out, res = cfg.match_strings(strings, max_records=16, compact_pitch=M)
    for j, s in enumerate(strings):
        try:
            w = P.match_substrs(pdefs, M, s)
        except P.InvalidTransition as e:
            assert out.status["flags"][j] & _abi.B2R_ST_INVALID_TRANSITION
            _, d, pos, state, c = e.args
            assert (out.status["err_def"][j], out.status["err_pos"][j], out.status["err_state"][j], out.status["err_byte"][j]) == (d, pos, state, c)
            continue
        fl = int(out.status["flags"][j])
        assert not fl & _abi.B2R_ST_INVALID_TRANSITION
        assert bool(fl & _abi.B2R_ST_OVERLAP) == w["overlap"]
        for d in range(cfg.n_defs):
            assert list(out.states[d][j, :M]) == w["states"][d]
            assert list(out.substr_ids[d][j, :M]) == w["substr_ids"][d]
            assert list(out.bits(out.start_enable[d])[j].astype(int)) == w["start_enable"][d]
            assert list(out.bits(out.end_enable[d])[j].astype(int)) == w["end_enable"][d]
            assert bool(fl & _abi.B2R_ST_ACCEPTED(d)) == w["accepted"][d]
        if not w["overlap"]:
            assert list(out.masked_chars[j, :M]) == w["masked_chars"]
            assert list(out.masked_substr_ids[j, :M]) == w["masked_substr_ids"]
            assert bytes(out.compact_bytes[j, :out.status["n_compact"][j]]) == bytes(c for c, m in zip(w["chars"], w["mask"]) if m)
            cons_ok, _ = P.check_constraints(pdefs, M, w)
            assert cons_ok
    return out


def _random_strings(rng, n, max_len, snippets, alphabet=ALPHABET):
    out = []
    for _ in range(n):
        L = rng.randrange(0, max_len + 1)
        b = bytearray(rng.choice(alphabet) for _ in range(L))
        for _ in range(rng.randrange(0, 4)):
            sn = rng.choice(snippets)
            if len(sn) <= L:
                o = rng.randrange(0, L - len(sn) + 1)
                b[o:o + len(sn)] = sn
        out.append(bytes(b))
    return out


SNIPPETS = [b"email was meant for @ab.", b"email was meant for @z and xy.", b" Also for swq.", b"from:alice@gmail.com\r\n",
            b"\r\nfrom:bob<bob@x.org>\r\n", b"from:", b"@", b"\r\n", b"email was meant for @"]


@pytest.mark.parametrize("set_name", ["regex1", "regex2", "regex3", "test1", "regex3_k3", "three"])
def test_oracle_vs_pyref_random(set_name):
    rng = random.Random(zlib.crc32(set_name.encode()))
    strings = _random_strings(rng, 60, 95, SNIPPETS) + [b"", b"e", b"email was meant for @y. Also for x."]
    _compare_with_pyref(set_name, 96, strings)


def test_oracle_vs_pyref_partial_dfa():
    """ex_allstr.txt is a partial DFA: most random strings hit an invalid transition (src/lib.rs:817)."""
    rng = random.Random(7)
    alpha = b"email wsntfor@vitalik.abc"
    strings = _random_strings(rng, 40, 40, [b"email was meant for @vitalik.", b"email was meant for @a."], alphabet=alpha)
    strings += [b"email was meant for @vitalik.", b"email was meant for @vitalik.x", b"\xff"]
    out = _compare_with_pyref("example", 64, strings)
    assert (out.status["flags"] & _abi.B2R_ST_INVALID_TRANSITION).any()


def test_multiplicity_invariants():
    """sum_r mult[d][r] = N*M; both endpoint halves sum to N*M; row 0 = number of padded rows (SURVEY 8(a) row 12)."""
    rng = random.Random(3)
    strings = _random_strings(rng, 50, 100, SNIPPETS)
    M = 101
    cfg = oracle_config("three", M)
    out, res = cfg.match_strings(strings)
    assert res.code == 0
    pad = sum(M - len(s) for s in strings)
    for d in range(3):
        assert int(out.mult[d].sum()) == len(strings) * M
        assert int(out.mult[d][0]) == pad
        E = cfg.endpoint_num_rows[d]
        assert int(out.endpoint_mult[d][:E].sum()) == len(strings) * M
        assert int(out.endpoint_mult[d][E:].sum()) == len(strings) * M
        # recount from the dense columns: rows (char, cur) of the table
        rows = cfg.table_rows(d)
        key = {(int(r[0]), int(r[1])): i for i, r in enumerate(rows) if i > 0}
        cnt = np.zeros(len(rows), np.uint64)
        for j, s in enumerate(strings):
            for i, c in enumerate(s):
                cnt[key[(c, int(out.states[d][j, i]))]] += 1
        cnt[0] = pad
        assert np.array_equal(cnt, out.mult[d])


def test_too_long_and_threads():
    cfg = oracle_config("regex1", 16)
    out, res = cfg.match_strings([b"a" * 15, b"a" * 16, b"b" * 3])
    assert res.code == _abi.B2R_ERR_TOO_LONG and res.string_idx == 1
    assert out.status["flags"][1] & _abi.B2R_ST_TOO_LONG
    rng = random.Random(11)
    strings = _random_strings(rng, 64, 60, SNIPPETS)
    cfg = oracle_config("test1", 64)
    a, _ = cfg.match_strings(strings, nthreads=1)
    b, _ = cfg.match_strings(strings, nthreads=4)
    from halo2_regex_b200.buffers import compare_outputs
    assert compare_outputs(a, b) == []
