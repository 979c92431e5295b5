"""For one def the emit stage writes records and compact areas as whole 32-byte sectors, and the fused kernel writes bitmap
sectors whole too (emit.cuh, DESIGN 4.2): a bitmap row's 256-row span in one store (word stores when the row's sectors are not
32-byte aligned, and in the stand-alone emit kernel), zeros after a string's last record up to the end of its sector, compact
areas of at most 8 bytes stored by the whole warp at once and longer ones padded with zeros.  Several defs keep the plain
stores.  Every case compares every column, status, record, compact byte and counter with the CPU oracle, with the output
columns pre-filled with a pattern, on the fused and the stand-alone emit stage (launch counts asserted):

  M                 1, 33, 257, 1025 and 4097 (the last bitmap sector of a row is partial)
  bitmap_pitch      132 and 136 (not a multiple of 32: word stores), 160; bitmap columns 16- but not 32-byte aligned
  spans             start and end bits of a match in one 256-row span and on both sides of a span boundary; more than 8 set
                    words in one row (and more masked segments than the registers hold)
  records           max_records 1, 2, 3 and 8, records pointer 16- but not 32-byte aligned
  compact bytes     compact_pitch 1, 7, 8, 32 and 64, with truncation
  strings           invalid, too long, overlapping (two defs flag one row), empty; partial tiles
  defs              one, two and three defs, and the 1023-state DFA"""
import random

import numpy as np
import pytest

from conftest import oracle_config, product_config
from test_gpu_parity import _pack
from test_oracle_golden import SNIPPETS, _random_strings

pytestmark = pytest.mark.gpu

MATCH = b"email was meant for @ab."
DUP = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"]), ("regex1_test_lookup.txt", ["substr1_test_lookup.txt"])]


def _planted(L, at_list, snippet=MATCH, fill=b"x"):
    b = bytearray(fill * L)
    for at in at_list:
        if 0 <= at and at + len(snippet) <= L:
            b[at:at + len(snippet)] = snippet
    return bytes(b)


def _strings(rng, M, n_random=70, invalid=False):
    """Valid strings of every shape up to M - 1 bytes (plus one too long one); invalid=True adds strings with bytes the DFAs
    have no transition for."""
    Lmax = M - 1
    out = [b"", b"x" * min(Lmax, 3)]
    if Lmax >= len(MATCH):
        out.append(MATCH)
        out.append(_planted(Lmax, [Lmax - len(MATCH)]))                           # a match that ends at the last row
        out.append(_planted(Lmax, list(range(0, Lmax, len(MATCH)))))               # back to back: every word of the row set
        out.append(_planted(Lmax, list(range(3, Lmax, 40))))                       # many segments, more than 8 set words
        out.append(_planted(Lmax, [5, Lmax // 2, Lmax - len(MATCH) - 1]))          # three segments in registers
        out.append((b"email was meant for @" + b"q" * 100 + b".")[:Lmax])           # more masked bytes than any compact area
        for span in range(256, Lmax, 256):
            out.append(_planted(Lmax, [span - 12]))                                # start and end bits on both sides of a span
            out.append(_planted(Lmax, [span - 40, span + 3]))
    out.append(b"y" * (M + 5))                                                     # too long
    out += _random_strings(rng, n_random, Lmax, SNIPPETS)
    if invalid:
        out += [bytes([0xFF]) * min(Lmax, 7), MATCH[:10] + b"\x01\x02" if Lmax >= 12 else b"\x01"]
    out = [s if len(s) <= M + 5 else s[:Lmax] for s in out]
    rng.shuffle(out)
    return out


def _offset16(t):
    """A view of a fresh tensor like t whose data pointer is 16 but not 32 bytes aligned."""
    import torch
    flat = torch.empty(t.numel() + 48, dtype=torch.uint8, device=t.device)
    base = flat.data_ptr() % 32
    start = (16 - base) % 32
    return flat[start:start + t.numel()].view(t.dtype).view(t.shape)


def _run(cfg, ocfg, strings, M, fuse, bitmap_pitch=None, max_records=8, compact_pitch=64, misalign=(), lead=0):
    import halo2_regex_b200 as H
    import torch
    data, offs = _pack(strings, lead)
    d_bytes = torch.from_numpy(data.copy()).cuda() if len(data) else torch.zeros(0, dtype=torch.uint8, device="cuda")
    d_offs = torch.from_numpy(offs.astype(np.int64)).cuda()
    out = H.DeviceOutputs(cfg, len(strings), bitmap_pitch=bitmap_pitch, max_records=max_records, compact_pitch=compact_pitch)
    if "records" in misalign:
        out.records = _offset16(out.records)
    if "bitmaps" in misalign:
        out.start_enable = [_offset16(t) for t in out.start_enable]
        out.end_enable = [_offset16(t) for t in out.end_enable]
    cols = list(out.states) + list(out.substr_ids) + list(out.start_enable) + list(out.end_enable)
    cols += [out.masked_chars, out.masked_substr_ids, out.status, out.records, out.compact_bytes]
    for t in cols:
        t.view(torch.uint8).fill_(0xA5)
    cfg.set_option("fuse", fuse)
    cfg.match_batch_device(d_bytes, d_offs, out)
    res = cfg.batch_result(check=False)
    assert cfg.last_launch_count() == (2 if fuse == 1 else 3)                     # walk (+ emit) + finalize
    o, ores = ocfg.match_batch(data, offs, bitmap_pitch=out.bitmap_pitch, max_records=max_records, compact_pitch=compact_pitch)
    assert res.code == ores.code
    if ores.code != 0:
        assert (res.string_idx, res.pos, res.state, res.byte, res.defidx) == (ores.string_idx, ores.pos, ores.state, ores.byte, ores.defidx)
    assert res.n_overlap_lo == ores.n_overlap_lo
    g = out.to_host()
    errs = H.compare_outputs(g, o)
    assert errs == [], f"fuse={fuse} bitmap_pitch={out.bitmap_pitch} misalign={misalign}: " + "\n".join(errs)
    return g, o


@pytest.mark.parametrize("M", [1, 33, 257, 1025, 4097])
def test_lengths_and_bitmap_pitch(M):
    """One def (fused and stand-alone emit): every M, with the bitmap pitches that keep rows 32-byte aligned and those that do
    not, and bitmap columns that are only 16-byte aligned."""
    rng = random.Random(M)
    cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
    strings = _strings(rng, M)
    bm = (M + 7) // 8
    pitches = [None, (bm + 3) // 4 * 4 + 4] + ([132, 136, 160] if M == 1025 else [])
    for fuse in (1, 2):
        for bp in pitches:
            _run(cfg, ocfg, strings, M, fuse, bitmap_pitch=bp)
        _run(cfg, ocfg, strings, M, fuse, misalign=("bitmaps",), lead=3)
    cfg.set_option("fuse", -1)


@pytest.mark.parametrize("max_records", [1, 2, 3, 8])
def test_records(max_records):
    """Records padded to the end of their sector, with the records pointer 32- and only 16-byte aligned; truncation.  One def
    with three substrings, whose strings have up to four records."""
    rng = random.Random(max_records)
    M = 1025
    cfg, ocfg = product_config("regex3_k3", M), oracle_config("regex3_k3", M)
    strings = _strings(rng, M, n_random=300)
    for fuse in (1, 2):
        for mis in ((), ("records",)):
            g, o = _run(cfg, ocfg, strings, M, fuse, max_records=max_records, compact_pitch=64, misalign=mis)
    n = g.status["n_records"]
    assert (n % 2 == 1).any() and ((n > 0) & (n % 2 == 0)).any()
    if max_records < 4:
        assert (n > max_records).any()                                          # some strings' records are truncated
    cfg.set_option("fuse", -1)


@pytest.mark.parametrize("compact_pitch", [1, 7, 8, 32, 64])
def test_compact_bytes(compact_pitch):
    """Compact areas of 1..8 bytes stored by the warp at once, longer ones padded with zeros; truncation; ragged offsets."""
    rng = random.Random(compact_pitch)
    M = 1025
    cfg, ocfg = product_config("regex1", M), oracle_config("regex1", M)
    strings = _strings(rng, M)
    for fuse in (1, 0):
        g, o = _run(cfg, ocfg, strings, M, fuse, max_records=2, compact_pitch=compact_pitch, lead=5)
    n = g.status["n_compact"]
    assert (n > compact_pitch).any() and ((n > 0) & (n < compact_pitch)).any() if compact_pitch > 1 else (n > 1).any()
    cfg.set_option("fuse", -1)


@pytest.mark.parametrize("set_name", ["regex1", "test1", "three", "dup"])
def test_defs_and_bad_strings(set_name):
    """One, two and three defs and two defs flagging the same rows (overlap), fused and stand-alone emit, with invalid and too
    long strings and a partial last tile."""
    rng = random.Random(len(set_name))
    M = 1025
    spec = DUP if set_name == "dup" else set_name
    cfg, ocfg = product_config(spec, M), oracle_config(spec, M)
    for invalid in (False, True):
        strings = _strings(rng, M, invalid=invalid)
        assert len(strings) % 32 != 0
        for fuse in (1, 2, 0):
            for max_records, compact_pitch in ((2, 8), (3, 7), (4, 32)):
                g, o = _run(cfg, ocfg, strings, M, fuse, max_records=max_records, compact_pitch=compact_pitch, misalign=("records",) if max_records == 4 else ())
    if set_name == "dup":
        assert (g.status["flags"] & __import__("halo2_regex_b200")._abi.B2R_ST_OVERLAP).any()
    cfg.set_option("fuse", -1)


def test_dfa1023():
    """The 1023-state DFA (2-byte state column, stand-alone emit by default) on config-4 header blocks, emit fused and not."""
    from halo2_regex_b200 import workloads as W
    from test_dfa_shapes import Dfa, _oracle, _product
    allstr, substr, _ = W.large_dfa_texts()
    dfa = Dfa(1023, None, None, allstr, [substr], None)
    M = 4097
    cfg, ocfg = _product([dfa], M), _oracle([dfa], M)
    data, _ = W.config4_numpy(96, 4096)
    strings = [bytes(r[:len(r) - k % 300]) for k, r in enumerate(data)] + [b"", b"from:ab@example.org\r\n"]
    for fuse in (1, 2):
        for max_records, compact_pitch in ((2, 64), (3, 8), (8, 7)):
            _run(cfg, ocfg, strings, M, fuse, max_records=max_records, compact_pitch=compact_pitch)
    cfg.set_option("fuse", -1)
