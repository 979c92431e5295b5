"""Parity across DFA shapes: synthetic definitions whose state count S (= largest_state_val + 1), number of byte classes C and
number of defs D sit on both sides of every branch the kernels take on them, with a first state other than 0 in about half
the cases.  Every column, status, record and multiplicity is compared bit-exactly with the oracle, and every case asserts the
plan (b2r_last_plan) or the launch count that proves which branch ran.

  batch path   S+1 on both sides of each power-of-two padding of the walk tables, of the u8/u16 state column (S = 255 / 256)
               and of the REPL / REPL16 entry-width limits; every forced table / bin placement; every emit placement
  long path    S+1 = 16 / 17 (SP of the fused pass), 32 / 33 (fused vs general pass), C * (S+1) > 65535 (tables in global
               memory), S+1 on both sides of the scan / compose limit of the composition tree, the 1023-state DFA, S = 65535;
               DFAs that never collapse, that collapse to k = 1..5 images (the dedupe's n = 1, 2, 3, 4 and wide chunks) and that
               fall into an absorbing sink
  graphs       the long path captured in a CUDA graph on each of its three prefix branches

The largest cases (8 MiB string, S = 65535) carry `huge` in their names so that a slow run (a sanitizer) can skip them."""
import random
import zlib

import numpy as np
import pytest

from test_gpu_parity import _pack
from test_oracle_golden import _compare_with_pyref

KINDS = ["perm"] + [f"collapse_{k}" for k in range(1, 6)] + ["sink"]
LONG_CHUNK, LONG_FANOUT = 1024, 64              # csrc/long.cuh


# ---- synthetic definitions ---------------------------------------------------------------------------------------------
class Dfa:
    """allstr / substr texts in the reference's format, the bytes that have transitions, and the header values."""

    def __init__(self, S, first, accepted, allstr, substrs, alphabet, sink_byte=None):
        self.S, self.first, self.accepted = S, first, accepted
        self.allstr, self.substrs, self.alphabet, self.sink_byte = allstr, substrs, alphabet, sink_byte


def make_dfa(S, n_classes, first, accepted, kind, seed, missing=0.0, alphabet=None, n_substrs=1, inside=0.995):
    """A DFA with S states (0 .. S-1), `n_classes` byte classes over `alphabet` (default: n_classes random bytes; every other
    byte is an invalid transition from every state), first / accepted state as given (accepted >= S: never accepted).
      perm        every class permutes the states: the walks of a chunk never merge
      collapse_k  class c maps state s to T[c][s mod k], T[c] hitting k different residues: after one byte exactly k distinct
                  images remain (plus the trap state of an invalid transition)
      sink        class 0 sends every state to one absorbing state (the accepted one when it exists), the others permute the rest
    `missing` drops that fraction of the (byte, state) transitions.  Substring defs: substr 1 is every transition between two
    states of a random set Q (a fraction `inside` of the states), so that substrings are hundreds of rows long with short gaps;
    substr 2 (n_substrs = 2) is every transition out of Q, a one-row substring behind each of them."""
    rng = random.Random(seed)
    if alphabet is None:
        alphabet = bytes(sorted(rng.sample(range(256), n_classes)))
    n_classes = min(n_classes, len(alphabet))
    nxt, seen = [], set()
    for c in range(n_classes):
        for _attempt in range(1000):                    # distinct classes where the state count allows it
            if kind == "perm":
                col = list(range(S))
                rng.shuffle(col)
            elif kind.startswith("collapse_"):
                k = min(int(kind[len("collapse_"):]), S)
                lanes = list(range(k))
                rng.shuffle(lanes)
                T = [lanes[j] + k * rng.randrange((S - 1 - lanes[j]) // k + 1) for j in range(k)]
                col = [T[s % k] for s in range(S)]
            elif kind == "sink":
                z = accepted if accepted < S else S - 1
                if c == 0:
                    col = [z] * S
                else:
                    rest = [s for s in range(S) if s != z]
                    perm = rest[:]
                    rng.shuffle(perm)
                    m = dict(zip(rest, perm))
                    col = [z if s == z else m[s] for s in range(S)]
            else:
                raise ValueError(kind)
            if tuple(col) not in seen:
                break
        seen.add(tuple(col))
        nxt.append(col)
    lines = [f"{first}\n{accepted}\n{S - 1}\n"]
    trans = []
    for s in range(S):
        for i, b in enumerate(alphabet):
            if missing and rng.random() < missing:
                continue
            t = nxt[i % n_classes][s]
            trans.append((s, t))
            lines.append(f"{s} {t} {b}\n")
    allstr = "".join(lines).encode()
    q = [rng.random() < inside for _ in range(S)]
    inner = sorted({(s, t) for s, t in trans if q[s] and q[t]})
    exits = sorted({(s, t) for s, t in trans if q[s] and not q[t]})
    # start / end states: every state of Q for small DFAs; for large ones (the loaders' endpoint tables are quadratic in these
    # lists) the states the walks visit most: the targets of the collapsing classes, or a sample of Q
    qs = [s for s in range(S) if q[s]]
    if len(qs) > 256:
        hot = sorted({t for col in nxt for t in col[:64]} & set(qs)) if kind.startswith("collapse_") else []
        qs = sorted(set(hot[:128]) | set(rng.sample(qs, 128)))
    ends = " ".join(map(str, qs))

    def substr(pairs):
        return (f"1000000\n0\n1000000\n{ends}\n{ends}\n" + "".join(f"{s} {t}\n" for s, t in pairs)).encode()

    substrs = [substr(inner)] + ([substr(exits)] if n_substrs > 1 else [])
    return Dfa(S, first, accepted, allstr, substrs, alphabet, sink_byte=alphabet[0] if kind == "sink" else None)


def _first_and_accepted(S, i):
    """Non-zero first state in about half the cases; every third case has accepted = S (never reached)."""
    first = 0 if i % 2 == 0 else (S - 1 if i % 4 == 1 else S // 2)
    accepted = S if i % 3 == 0 else (S - 1 - i) % S
    return first, accepted


def _oracle(dfas, M):
    from oracle import oracle as O
    return O.OracleConfig([(O.OracleAllstr(d.allstr), [O.OracleSubstr(x) for x in d.substrs]) for d in dfas], M)


def _product(dfas, M):
    import halo2_regex_b200 as H
    return H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(d.allstr),
                                                         [H.SubstrRegexDef.read_from_reader(x) for x in d.substrs]) for d in dfas])


def _strings(rng, dfa, n, M, extra=()):
    """Ragged strings over the DFA's alphabet: lengths 0, 1 and M-1 among random ones; sink bytes kept rare."""
    alpha = bytes(b for b in dfa.alphabet if b != dfa.sink_byte) or dfa.alphabet
    lens = [0, 1, M - 1, M - 1] + [rng.randrange(0, M) for _ in range(n - 4)]
    out = []
    for L in lens:
        s = bytearray(rng.choice(alpha) for _ in range(L))
        if dfa.sink_byte is not None and L > 8 and rng.random() < 0.5:
            s[rng.randrange(L)] = dfa.sink_byte
        out.append(bytes(s))
    return out + list(extra)


def _long_body(np_rng, dfa, length):
    """One long string over the DFA's alphabet; with a sink: a few sink bytes, one of them in the last quarter."""
    alpha = np.frombuffer(bytes(b for b in dfa.alphabet if b != dfa.sink_byte) or dfa.alphabet, dtype=np.uint8)
    body = alpha[np_rng.integers(0, len(alpha), length)] if length else np.zeros(0, np.uint8)
    if dfa.sink_byte is not None and length > 4:
        body[int(length * 0.8)] = dfa.sink_byte
    return body


def _compare(g, gres, o, ores):
    import halo2_regex_b200 as H
    assert gres.code == ores.code
    if ores.code != 0:
        assert (gres.string_idx, gres.pos, gres.state, gres.byte, gres.defidx) == (ores.string_idx, ores.pos, ores.state, ores.byte, ores.defidx)
    errs = H.compare_outputs(g, o)
    assert errs == [], "\n".join(errs)


# ---- CPU: the two references agree on the new shapes ------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("S", [1, 2, 17, 33, 256])
def test_generated_dfas_oracle_vs_pyref(S, kind):
    """oracle.c against the independent Python restatement on every synthetic shape the GPU tests use, including invalid
    transitions (`missing`), a non-zero first state and an accepted state >= S."""
    from oracle import pyref as P
    i = KINDS.index(kind)
    first, accepted = _first_and_accepted(S, i + S)
    dfa = make_dfa(S, 5, first, accepted, kind, seed=S * 31 + i, missing=0.02 if i % 2 else 0.0, n_substrs=1 + i % 2)
    M = 130
    rng = random.Random(S * 7 + i)
    bad = next(b for b in range(256) if b not in dfa.alphabet)
    strings = _strings(rng, dfa, 30, M, extra=[bytes([dfa.alphabet[0]]) * 129, bytes([dfa.alphabet[-1], bad])])
    pdefs = [(P.PyAllstr(dfa.allstr), [P.PySubstr(x) for x in dfa.substrs])]
    out = _compare_with_pyref(None, M, strings, cfg=_oracle([dfa], M), pdefs=pdefs)
    from halo2_regex_b200 import _abi
    if not out.status["flags"][2] & _abi.B2R_ST_INVALID_TRANSITION:
        assert int(out.states[0][2, 0]) == first                     # the walk starts in first_state (row 0 of a non-empty string)


def test_generated_substrings_are_long_and_many():
    """The substring defs of the generator do what the GPU tests rely on: masked segments hundreds of rows long, and strings with
    more than EMIT_NSEG = 4 segments (the emit stage's patch pass)."""
    dfa = make_dfa(40, 6, 3, 7, "perm", seed=5, n_substrs=2)
    M = 2049
    rng = random.Random(1)
    strings = _strings(rng, dfa, 40, M)
    o, res = _oracle([dfa], M).match_strings(strings, max_records=64, compact_pitch=M)
    assert res.code == 0
    assert int(o.status["n_records"].max()) > 4
    rec = o.records.view(np.uint32).reshape(len(strings), 64, 4)
    assert int(rec[..., 1].max()) >= 200                             # b2r_substr_record: start, len, substr_id, compact_off


def test_state_count_limit():
    """largest_state_val 65534 (S = 65535, the dummy state 65535 still fits the u16 column) configures; 65535 is refused with
    B2R_ERR_UNSUPPORTED."""
    import halo2_regex_b200 as H
    sub = b"1\n0\n1\n0\n1\n0 1\n"
    for largest, ok in ((65534, True), (65535, False)):
        allstr = f"0\n1\n{largest}\n0 1 97\n1 0 98\n".encode()
        defs = [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(sub)])]
        if ok:
            cfg = H.RegexVerifyConfig.configure(64, defs, device=-1)
            assert cfg.state_widths == [2] and cfg.dummy_states == [65535]
        else:
            with pytest.raises(RuntimeError, match=rf"\({H._abi.B2R_ERR_UNSUPPORTED}\)"):
                H.RegexVerifyConfig.configure(64, defs, device=-1)


# ---- batch path ---------------------------------------------------------------------------------------------------------
BATCH_S = [1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 255, 256, 257, 511, 512, 513, 1023, 1024, 4095, 65535]
PLACEMENTS = [("repl", "smem"), ("plain", "smem"), ("plain16", "smem"), ("repl", "global"), ("plain16", "global"), ("global", "global"),
              ("repl16", "smem"), ("repl16", "global")]
STRIDE = {"repl": 128, "repl16": 64, "plain": 4, "plain16": 2, "global": 0}     # csrc/walk.cuh walk_stride


def _padded(S):
    P = 1
    while P < S + 1:
        P <<= 1
    return P


def _placement_expected(S, C, tm, hm, max_smem):
    """Placement (tm, hm) forced on defs with S states and C byte classes (ints for one def, lists for several): a tuple
    (table_ok, hist_ok) with a False = the planner cannot honour that half (csrc/kernels.cu fits_k: every def's table entry holds
    next * stride in 16 bits, REPL16 only up to 512 padded states, the tables of all defs and their shared-memory bins must fit,
    shared bins only when no def needs a u16 state column, which then every def uses); True = it fits with room to spare and must
    be honoured; None = too close to call from here."""
    Ss, Cs = ([S], [C]) if isinstance(S, int) else (list(S), list(C))
    Ps, st = [_padded(s) for s in Ss], STRIDE[tm]
    tables = sum(c * P * st for c, P in zip(Cs, Ps))
    table_ok = tm == "global" or (all(P * st <= 65536 and (tm != "repl16" or P <= 512) for P in Ps) and tables <= max_smem)
    bins = sum((s + 1) * 256 * 4 for s in Ss)
    # two or three defs on 16-bit entries may keep compact bins (fewer columns than 256): only their width rule is certain
    compact = tm in ("plain16", "repl16") and 2 <= len(Ss) <= 3
    hist_ok = hm == "global" or (max(Ss) <= 255 and (bins <= max_smem or compact))
    if not table_ok or not hist_ok:
        return (table_ok, hist_ok)
    if hm == "smem" and bins > max_smem:
        return None
    used = (tables + len(Ps) * max(Ps) * st + 256 * 128 if tm != "global" else 0) + (bins if hm == "smem" else 2048 * len(Ss)) + 64 * 1024
    return True if used <= max_smem else None


@pytest.mark.gpu
@pytest.mark.parametrize("S", [pytest.param(s, id=f"S{s}" + ("_huge" if s > 4095 else "")) for s in BATCH_S])
def test_batch_state_counts(S):
    """One def with S states through the batch path: the default plan, then (S <= 1024) every forced table / bin placement and
    every emit placement, all against the oracle; lengths 0, 1 and M-1 at a 16-byte granule edge."""
    import torch
    import halo2_regex_b200 as H
    i = BATCH_S.index(S)
    kind = ("perm", "collapse_3", "sink", "collapse_1")[i % 4]
    first, accepted = _first_and_accepted(S, i)
    n_classes = 2 if S >= 256 else 5                     # few classes: the 512-state tables of REPL16 fit shared memory
    dfa = make_dfa(S, n_classes, first, accepted, kind, seed=1000 + S, n_substrs=1 + i % 2, alphabet=b"ab\x00\xffcz" if S >= 256 else None)
    M = (96, 97, 112, 113, 128, 129)[i % 6]
    rng = random.Random(S)
    strings = _strings(rng, dfa, 72 if S <= 4095 else 40, M)
    data, offs = _pack(strings)
    o, ores = _oracle([dfa], M).match_batch(data, offs, max_records=8, compact_pitch=64)
    cfg = _product([dfa], M)
    assert cfg.state_widths == [1 if S <= 255 else 2]      # csrc/defs.cpp: u8 up to 255 states
    assert cfg.dummy_states == [S]
    C = cfg.num_byte_classes[0]
    max_smem = torch.cuda.get_device_properties(0).shared_memory_per_block_optin

    def run(label):
        g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, max_records=8, compact_pitch=64)
        try:
            _compare(g, gres, o, ores)
        except AssertionError as e:
            raise AssertionError(f"S={S} {label}: {e}") from None
        return g

    g = run("default")
    if first and len(strings[2]):
        assert int(g.states[0][2, 0]) == first
    if S > 1024:
        return
    honoured = {}
    for tm, hm in PLACEMENTS:
        cfg.set_option("table_mode", tm)
        cfg.set_option("hist_mode", hm)
        run(f"{tm}/{hm}")
        plan = cfg.last_plan()
        exp = _placement_expected(S, C, tm, hm, max_smem)
        if exp is True:
            assert plan == (tm, hm), (S, tm, hm, plan)
        elif isinstance(exp, tuple):                         # the side of the limit the planner must not cross
            if not exp[0]:
                assert plan[0] != tm, (S, tm, hm, plan)
            if not exp[1]:
                assert plan[1] != hm, (S, tm, hm, plan)
        honoured[(tm, hm)] = plan == (tm, hm)
    # the boundaries themselves: 16-bit replicated entries up to 511 states (512 padded states), never 32-bit replicated ones
    # beyond that (512 * 128 B > 16 bits), shared-memory bins only for u8 columns
    if S == 511:
        assert honoured[("repl16", "global")]
    if S in (512, 513, 1023, 1024):
        assert not any(honoured[(t, h)] for t, h in PLACEMENTS if t in ("repl", "repl16"))
    if S in (255, 256, 257):
        assert not any(honoured[(t, h)] for t, h in PLACEMENTS if h == "smem")
    if S <= 127:
        assert honoured[("plain16", "smem")]
    cfg.set_option("table_mode", "auto")
    cfg.set_option("hist_mode", "auto")
    for fuse in (0, 1, 2):
        cfg.set_option("fuse", fuse)
        run(f"fuse={fuse}")
        assert cfg.last_launch_count() == (2 if fuse == 1 else 3)   # walk (+ emit) + finalize


@pytest.mark.gpu
@pytest.mark.parametrize("n_defs", [3, 4])
def test_batch_mixed_widths(n_defs):
    """Defs with 255 and 256 states side by side (every column of the config becomes u16), one of them never accepting, one of
    them starting in a non-zero state; default plan and every emit placement."""
    spec = [(255, "perm", 7, 3), (256, "collapse_2", 0, 256), (255, "sink", 254, 254), (256, "perm", 128, 17)][:n_defs]
    dfas = [make_dfa(S, 3, first, acc, kind, seed=77 + k, alphabet=b"abcd", n_substrs=1 + k % 2) for k, (S, kind, first, acc) in enumerate(spec)]
    M = 161
    rng = random.Random(n_defs)
    strings = _strings(rng, dfas[0], 90, M)
    data, offs = _pack(strings)
    o, ores = _oracle(dfas, M).match_batch(data, offs, max_records=8, compact_pitch=32)
    cfg = _product(dfas, M)
    assert cfg.state_widths == [2] * n_defs
    for fuse in (-1, 0, 1, 2):
        cfg.set_option("fuse", fuse)
        g, gres = cfg.match_batch_host(data, offs, check=False, fill=0xCD, max_records=8, compact_pitch=32)
        _compare(g, gres, o, ores)
        if fuse >= 0:
            assert cfg.last_launch_count() == (2 if fuse == 1 else 3)
    import halo2_regex_b200 as H
    assert not (g.status["flags"] & H._abi.B2R_ST_ACCEPTED(1)).any()          # def 1 (accepted = S) never accepts


# ---- long-string path ------------------------------------------------------------------------------------------------------
LONG_LENGTHS = [0, 1, 511, 512, 513, 1024, 1025, 262143, 262144, 262145]


def _max_smem():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _long_launches(cfg, length, fused_opt, max_smem):
    """Kernel launches of one b2r_match_long call, from launch_long_prepare (csrc/long.cu): the fused pass is 2 per def; the
    general pass is the offsets kernel, then per def head / dedupe / tail / gather, and the tree: one scan per level + resolve
    when 2 * 64 * (S+1) u16 fit shared memory, else compose + propagate per level + the root entry.  Then walk, emit, finalize."""
    n_chunks = max(1, -(-length // LONG_CHUNK))
    levels, n = 1, n_chunks
    while n > 1:
        n = -(-n // LONG_FANOUT)
        levels += 1
    S1s = [s + 1 for s in cfg.dummy_states]
    C = cfg.num_byte_classes

    def fused_smem(s1, c):                                   # long_fused_smem
        sp, P = (16 if s1 <= 16 else 32), 1
        while P < s1:
            P <<= 1
        return 256 * 128 + c * P * 128 + 512 * sp + 16 * 32 * 80

    fused = bool(fused_opt) and all(s1 <= 32 and fused_smem(s1, C[d]) <= max_smem for d, s1 in enumerate(S1s))
    if fused:
        prep = 2 * len(S1s)
    else:
        prep = 1 + sum(4 + ((levels - 1) + 1 if 2 * LONG_FANOUT * s1 * 2 <= max_smem and levels <= 12 else 2 * (levels - 1) + 1) for s1 in S1s)
    return prep + 3, fused


def _run_long(cfg, ocfg_for, s, device, fused, max_smem, max_records=64, compact_pitch=512, want=None, expected=None):
    """One long string through match_long_device or match_long_host, against the oracle with M = len + 1; returns the
    product's outputs."""
    import torch
    import halo2_regex_b200 as H
    length = len(s)
    M = length + 1
    cfg.set_option("long_fused", fused)
    if device:
        buf = torch.zeros(length + 16, dtype=torch.uint8, device="cuda")
        if length:
            buf[:length].copy_(torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()))
        out = H.DeviceOutputs(cfg, 1, max_records=max_records, compact_pitch=compact_pitch, max_chars_size=M, want=want)
        cfg.match_long_device(buf[:length], out)
        gres = cfg.batch_result(check=False)
        g = out.to_host()
    else:
        g, gres = cfg.match_long_host(s, check=False, max_records=max_records, compact_pitch=compact_pitch, fill=0xCD, want=want)
    if expected is None:
        data, offs = _pack([s])
        expected = ocfg_for(M).match_batch(data, offs, max_records=max_records, compact_pitch=compact_pitch)
    o, ores = expected
    launches, is_fused = _long_launches(cfg, length, fused, max_smem)
    try:
        _compare(g, gres, o, ores)
        assert cfg.last_launch_count() == launches, (cfg.last_launch_count(), launches)
    except AssertionError as e:
        raise AssertionError(f"len={length} {'device' if device else 'host'} long_fused={fused} (fused pass: {is_fused}): {e}") from None
    return g, o


def _long_shape(shape, kind, max_smem):
    """-> (dfa, lengths)"""
    k = KINDS.index(kind)
    if shape.startswith("S") and shape[1:].isdigit() and int(shape[1:]) <= 32:
        S = int(shape[1:])
        return make_dfa(S, 6, *_first_and_accepted(S, k), kind, seed=S * 13 + k, n_substrs=1 + k % 2), LONG_LENGTHS
    if shape == "S300_C256":                                  # C * (S+1) > 65535: the head / tail / gather kernels on global tables
        return make_dfa(300, 256, *_first_and_accepted(300, k + 1), kind, seed=300 + k, alphabet=bytes(range(256))), LONG_LENGTHS
    if shape in ("scan_edge", "compose_edge"):                # S+1 = the largest tree that the shared-memory scan takes, and one more
        S = max_smem // (2 * LONG_FANOUT * 2) - (1 if shape == "scan_edge" else 0)
        return make_dfa(S, 6, *_first_and_accepted(S, k), kind, seed=S + k), LONG_LENGTHS
    if shape == "S65535_huge":
        return make_dfa(65535, 3, *_first_and_accepted(65535, k), kind, seed=65535 + k, alphabet=b"xyz"), [0, 1, 1025, 128 * LONG_CHUNK + 1]
    raise ValueError(shape)


LONG_CASES = [(sh, kd) for sh in ("S15", "S16", "S31", "S32", "S300_C256", "scan_edge", "compose_edge") for kd in KINDS] + \
             [("S65535_huge", f"collapse_{k}") for k in range(1, 6)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,kind", LONG_CASES)
def test_long_shapes(shape, kind):
    """One string per length (0 .. 256 KiB + 1, at chunk edges) through b2r_match_long, device and host entry points in turn,
    against the oracle; the launch count proves the prefix branch (fused / general with scan / general with compose)."""
    max_smem = _max_smem()
    dfa, lengths = _long_shape(shape, kind, max_smem)
    cfg = _product([dfa], 64)
    if shape == "S300_C256":
        assert cfg.num_byte_classes[0] * 301 > 65535
    if shape in ("scan_edge", "compose_edge"):
        fits = 2 * LONG_FANOUT * (dfa.S + 1) * 2 <= max_smem
        assert fits == (shape == "scan_edge")
    np_rng = np.random.default_rng(zlib.crc32(f"{shape}/{kind}".encode()))
    both = dfa.S + 1 <= 33
    for j, length in enumerate(lengths):
        s = _long_body(np_rng, dfa, length).tobytes()
        data, offs = _pack([s])
        expected = _oracle([dfa], length + 1).match_batch(data, offs, max_records=64, compact_pitch=512)
        for fused in ((1, 0) if both else (1,)):
            _run_long(cfg, None, s, device=(j + fused) % 2 == 0, fused=fused, max_smem=max_smem, expected=expected)


@pytest.mark.gpu
def test_long_config4_dfa():
    """The 1023-state DFA of BASELINE config 4 (S+1 = 1024: the compose / propagate tree) on one long string of mail headers."""
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from halo2_regex_b200 import workloads as W
    allstr, substr, _ = W.large_dfa_texts()
    cfg = H.RegexVerifyConfig.configure(64, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
    assert cfg.dummy_states == [1023]
    rows, _ = W.config4_numpy(80, 4096)
    body = rows.reshape(-1)
    max_smem = _max_smem()

    def ocfg_for(M):
        return O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], M)

    for j, length in enumerate(LONG_LENGTHS[:-3] + [262143, 262145]):
        _run_long(cfg, ocfg_for, body[:length].tobytes(), device=j % 2 == 0, fused=1, max_smem=max_smem)


@pytest.mark.gpu
def test_long_dedupe_fourth_image_from_a_real_state():
    """A chunk whose fourth distinct image (of four: the general pass's dedupe keeps up to four) first appears at a real state that
    is also the chunk's entry state: state 0 dies (every transition out of it is invalid), so the trap is image 0 and states 1, 2, 3
    bring the three lanes; byte 'r' resets every state to 3, and it ends every chunk."""
    S, k = 40, 3
    rng = random.Random(40)
    lines = [f"5\n{S - 1}\n{S - 1}\n"]
    classes = b"abcdefg"
    for c in classes:
        lanes = list(range(k))
        rng.shuffle(lanes)
        T = [lanes[j] + k * rng.randrange(1, (S - 1 - lanes[j]) // k + 1) for j in range(k)]    # never state 0
        lines += [f"{s} {T[s % k]} {c}\n" for s in range(1, S)]
    lines += [f"{s} 3 {ord('r')}\n" for s in range(1, S)]
    allstr = "".join(lines).encode()
    sub = (f"100\n0\n100\n{' '.join(map(str, range(1, S, 2)))}\n{' '.join(map(str, range(2, S, 2)))}\n" +
           "".join(f"{s} {t}\n" for s in range(1, S) for t in range(1, S) if (s + t) % 5)).encode()
    dfa = Dfa(S, 5, S - 1, allstr, [sub], classes + b"r")
    cfg = _product([dfa], 64)
    max_smem = _max_smem()
    np_rng = np.random.default_rng(4)
    for length in (1024 * 5 + 100, 262144):
        body = np.frombuffer(classes, np.uint8)[np_rng.integers(0, len(classes), length)]
        body[LONG_CHUNK - 1::LONG_CHUNK] = ord("r")
        for fused in (0, 1):
            _run_long(cfg, lambda M: _oracle([dfa], M), body.tobytes(), device=fused == 0, fused=fused, max_smem=max_smem)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [20, 300])
def test_long_invalid_transitions(S):
    """An invalid byte in the head of a chunk after the first (every state of that chunk maps to the trap: one image), in the
    middle of a later chunk, and in the last partial chunk; fused and general pass."""
    dfa = make_dfa(S, 4, 3, 5, "collapse_2" if S == 20 else "perm", seed=S, alphabet=b"abcd")
    cfg = _product([dfa], 64)
    max_smem = _max_smem()
    np_rng = np.random.default_rng(S)
    length = 40 * LONG_CHUNK + 300
    for at in (3 * LONG_CHUNK + 10, 17 * LONG_CHUNK + 600, length - 5, 0):
        body = np.frombuffer(b"abcd", np.uint8)[np_rng.integers(0, 4, length)]
        body[at] = ord("q")
        for fused in (1, 0):
            g, o = _run_long(cfg, lambda M: _oracle([dfa], M), body.tobytes(), device=fused == 1, fused=fused, max_smem=max_smem)
            assert o.status["err_pos"][0] == at


@pytest.mark.gpu
@pytest.mark.parametrize("n_defs", [3, 4])
def test_long_multi_def(n_defs):
    """3 and 4 defs with u8 and u16 columns mixed (20, 300, 255, 256 states): every column; then a later def failing before def 0
    does (the reference walks def 0 over the whole string first: def 0's failure is the one reported)."""
    spec = [(20, "perm", 4, 19), (300, "collapse_3", 0, 300), (255, "collapse_4", 200, 17), (256, "sink", 9, 255)][:n_defs]
    dfas = [make_dfa(S, 4, first, acc, kind, seed=900 + k, alphabet=b"abcd", n_substrs=1 + k % 2) for k, (S, kind, first, acc) in enumerate(spec)]
    cfg = _product(dfas, 64)
    assert cfg.state_widths == [2] * n_defs
    max_smem = _max_smem()
    np_rng = np.random.default_rng(n_defs)
    for length in (1, 1025, 70001):
        body = np.frombuffer(b"bcd", np.uint8)[np_rng.integers(0, 3, length)]
        if length > 100:
            body[length // 2] = ord("a")                          # the sink byte of def 3 (class 0 of its alphabet)
        for fused in (1, 0):
            _run_long(cfg, lambda M: _oracle(dfas, M), body.tobytes(), device=fused == 1, fused=fused, max_smem=max_smem)
    # 'f' is invalid for the last def only and comes first; 'e' is invalid for every def
    late = [make_dfa(S, 4, first, acc, kind, seed=900 + k, alphabet=b"abcd" + (b"" if k == n_defs - 1 else b"f"), n_substrs=1)
            for k, (S, kind, first, acc) in enumerate(spec)]
    cfg = _product(late, 64)
    body = np.frombuffer(b"abcd", np.uint8)[np_rng.integers(0, 4, 9000)]
    body[2500] = ord("f")
    body[7000] = ord("e")
    for fused in (1, 0):
        g, o = _run_long(cfg, lambda M: _oracle(late, M), body.tobytes(), device=fused == 0, fused=fused, max_smem=max_smem)
        assert (o.status["err_def"][0], o.status["err_pos"][0]) == (0, 7000)


@pytest.mark.gpu
def test_long_overlap_across_chunk_boundary():
    """Two copies of one def: every substring row is flagged twice (B2R_ST_OVERLAP), with substrings crossing chunk edges."""
    import halo2_regex_b200 as H
    dfa = make_dfa(24, 5, 2, 9, "perm", seed=24)
    cfg = _product([dfa, dfa], 64)
    max_smem = _max_smem()
    np_rng = np.random.default_rng(24)
    body = _long_body(np_rng, dfa, 5 * LONG_CHUNK + 7).tobytes()
    for fused in (1, 0):
        g, o = _run_long(cfg, lambda M: _oracle([dfa, dfa], M), body, device=fused == 1, fused=fused, max_smem=max_smem)
        assert g.status["flags"][0] & H._abi.B2R_ST_OVERLAP


@pytest.mark.gpu
def test_long_dense_segments_truncation_and_missing_states():
    """Masked segments hundreds of rows long and more than four of them (the patch pass), crossing chunk edges; then the same
    string with max_records = 1 and compact_pitch = 3 (truncation flags, exact counts), and without the state columns (the
    long path walks into a workspace column instead)."""
    import halo2_regex_b200 as H
    dfa = make_dfa(40, 6, 3, 7, "perm", seed=5, n_substrs=2)
    cfg = _product([dfa], 64)
    max_smem = _max_smem()
    np_rng = np.random.default_rng(40)
    body = _long_body(np_rng, dfa, 20 * LONG_CHUNK + 33).tobytes()
    for fused in (1, 0):
        g, o = _run_long(cfg, lambda M: _oracle([dfa], M), body, device=fused == 1, fused=fused, max_smem=max_smem, max_records=256, compact_pitch=1 << 15)
        assert int(o.status["n_records"][0]) > 4
        rec = o.records.view(np.uint32).reshape(1, 256, 4)[0, :int(o.status["n_records"][0])]
        assert any(int(r[0]) // LONG_CHUNK != (int(r[0]) + int(r[1]) - 1) // LONG_CHUNK for r in rec)     # a segment crosses a chunk edge
        g, o = _run_long(cfg, lambda M: _oracle([dfa], M), body, device=fused == 0, fused=fused, max_smem=max_smem, max_records=1, compact_pitch=3)
        assert g.status["flags"][0] & H._abi.B2R_ST_RECORDS_TRUNCATED and g.status["flags"][0] & H._abi.B2R_ST_COMPACT_TRUNCATED
        want = {"substr_ids", "start_enable", "end_enable", "masked_chars", "masked_substr_ids", "status", "records", "compact_bytes", "mult", "endpoint_mult"}
        _run_long(cfg, lambda M: _oracle([dfa], M), body, device=True, fused=fused, max_smem=max_smem, want=want)
        _run_long(cfg, lambda M: _oracle([dfa], M), body, device=False, fused=fused, max_smem=max_smem, want=want)


@pytest.mark.gpu
def test_long_huge_8_mib_plus_one_fused():
    """8 MiB + 1 bytes on the fused pass (a DFA that never collapses: every sub-chunk walks all states): the string crosses a
    super-group boundary (32 groups x 256 chunks x 1 KiB)."""
    dfa = make_dfa(29, 6, 11, 4, "perm", seed=8)
    cfg = _product([dfa], 64)
    np_rng = np.random.default_rng(8)
    body = _long_body(np_rng, dfa, (8 << 20) + 1).tobytes()
    _run_long(cfg, lambda M: _oracle([dfa], M), body, device=True, fused=1, max_smem=_max_smem(), max_records=16, compact_pitch=256)


@pytest.mark.gpu
# ---- CUDA graph capture of the long path ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("branch", ["fused", "scan", "compose"])
def test_long_path_cuda_graph(branch):
    """match_long_device captured once in a CUDA graph (after a first call of the same length has sized the workspace), replayed
    twice with different bytes written into the captured input buffer; each replay against the oracle."""
    import torch
    import halo2_regex_b200 as H
    from oracle import oracle as O
    from conftest import oracle_config, product_config
    from halo2_regex_b200 import workloads as W
    length = 70 * LONG_CHUNK + 11                               # three tree levels
    M = length + 1
    if branch == "fused":
        cfg, ocfg = product_config("regex2", 64), oracle_config("regex2", M)
        rng = random.Random(2)

        def body(seed):
            rng.seed(seed)
            b = bytearray(rng.choice(b"abc xyz.@\r\n") for _ in range(length))
            for at in range(seed, length - 20, 997):
                b[at:at + 16] = b" Also for xyzzy."
            return bytes(b)
    elif branch == "scan":
        dfa = make_dfa(300, 256, 17, 3, "perm", seed=3, alphabet=bytes(range(256)))
        cfg, ocfg = _product([dfa], 64), _oracle([dfa], M)

        def body(seed):
            return _long_body(np.random.default_rng(seed), dfa, length).tobytes()
    else:
        allstr, substr, _ = W.large_dfa_texts()
        cfg = H.RegexVerifyConfig.configure(64, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
        ocfg = O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], M)
        rows, _ = W.config4_numpy(40, 4096)

        def body(seed):
            return np.roll(rows.reshape(-1), seed * 4096)[:length].tobytes()
    max_smem = _max_smem()
    launches, fused = _long_launches(cfg, length, 1, max_smem)
    assert fused == (branch == "fused")
    if branch != "fused":
        assert (2 * LONG_FANOUT * (cfg.dummy_states[0] + 1) * 2 <= max_smem) == (branch == "scan")
    buf = torch.zeros(length + 16, dtype=torch.uint8, device="cuda")
    d = buf[:length]
    out = H.DeviceOutputs(cfg, 1, max_records=16, compact_pitch=256, max_chars_size=M)
    d.copy_(torch.from_numpy(np.frombuffer(body(1), np.uint8).copy()))
    cfg.match_long_device(d, out)
    assert cfg.batch_result().code == 0
    assert cfg.last_launch_count() == launches
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cfg.match_long_device(d, out)
    for seed in (2, 3):
        s = body(seed)
        d.copy_(torch.from_numpy(np.frombuffer(s, np.uint8).copy()))
        graph.replay()
        torch.cuda.synchronize()
        data, offs = _pack([s])
        o, ores = ocfg.match_batch(data, offs, max_records=16, compact_pitch=256)
        assert ores.code == 0
        errs = H.compare_outputs(out.to_host(), o)
        assert errs == [], (seed, errs)
