#!/usr/bin/env python3
"""Per-string lookup multiplicities: the match call and the b2r_string_mult post-pass after it, timed apart with CUDA events
(medians) on device-resident seeded inputs, plus the host entry end to end against b2r_match_batch_host.  For every shape it
reports the post-pass's bytes read (bytes + state columns + status + offsets) and written (entries, n_entries, endpoint counts),
its share of 6555 GB/s, and the mean distinct rows per string.  Prints the card and its power limit; with --out DIR also writes
string_mult_bench.json there."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import halo2_regex_b200 as H  # noqa: E402
from conftest import product_config  # noqa: E402
from halo2_regex_b200 import workloads as W  # noqa: E402

PEAK_GBS = 6555.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"card": name, "power_limit": power, "clocks_max_sm": clock}


def large_dfa(M):
    allstr, substr, _ = W.large_dfa_texts()
    return H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])


def events(fn, iters):
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def traffic(cfg, sm, offs_host, wide):
    lens = np.diff(offs_host.astype(np.int64))
    n = len(lens)
    rd = int(lens.sum()) * (1 + cfg.n_defs * (2 if wide else 1)) + n * 32 + (n + 1) * 8
    wr, distinct = 0, []
    for d in range(cfg.n_defs):
        ne = sm.n_entries[d].cpu().numpy().view(np.uint32).astype(np.int64)
        distinct.append(float(ne.mean()))
        wr += int(np.minimum(ne, sm.max_entries).sum()) * 8 + n * 4 + n * 2 * cfg.endpoint_num_rows[d] * 4
    return rd, wr, distinct


def device_shape(name, cfg, d_bytes, offs_host, iters, chunked=False, long=False, variants=False):
    n = len(offs_host) - 1
    M = int(offs_host[-1]) + 1 if long else cfg.max_chars_size
    out = H.DeviceOutputs(cfg, n, want={"states", "status", "mult", "endpoint_mult"}, max_chars_size=M if long else None)
    d_offs = torch.from_numpy(offs_host.astype(np.int64)).cuda()
    sm = H.StringMultOutputs(cfg, n, max_chars_size=M)
    if long:
        match = lambda: cfg.match_long_device(d_bytes, out)  # noqa: E731
    elif chunked:
        match = lambda: cfg.match_batch_chunked_device(d_bytes, d_offs, out)  # noqa: E731
    else:
        match = lambda: cfg.match_batch_device(d_bytes, d_offs, out)  # noqa: E731
    post = lambda: cfg.string_mult_device(d_bytes, d_offs, out, sm, max_chars_size=M if long else 0)  # noqa: E731
    match(); post(); torch.cuda.synchronize()                              # warm-up
    assert cfg.batch_result(check=False).code == 0
    launches = cfg.last_launch_count()
    match_ms, post_ms = events(match, iters), events(post, iters)
    # the sums of the per-string counts are the batch counters of the same call
    for d in range(cfg.n_defs):
        ne = sm.n_entries[d].cpu().numpy().view(np.uint32)
        assert (ne <= sm.max_entries).all()
        e = sm.entries[d].cpu().numpy().view(np.uint32)
        k = np.arange(sm.max_entries)[None, :] < ne[:, None]
        tot = np.zeros(cfg.table_num_rows[d], np.uint64)
        np.add.at(tot, e[..., 0][k].astype(np.int64), e[..., 1][k].astype(np.uint64))
        assert np.array_equal(tot, out.mult[d].cpu().numpy().astype(np.uint64)), name
    rd, wr, distinct = traffic(cfg, sm, offs_host, cfg.state_widths[0] == 2)
    parts = {}
    if variants:   # where the time goes: the same post-pass asked for fewer outputs (each drops one phase of string_mult_kernel)
        for label, want in (("n_entries only: count + rows + sort, no entry stores, no endpoint rows", ("n_entries",)),
                            ("entries: + entry stores, no endpoint rows", ("entries", "n_entries")),
                            ("endpoint counts only: count + rows + endpoint rows, no sort", ("endpoint_counts",))):
            smv = H.StringMultOutputs(cfg, n, max_chars_size=M, want=want)
            fn = lambda: cfg.string_mult_device(d_bytes, d_offs, out, smv, max_chars_size=M if long else 0)  # noqa: E731
            fn()
            parts[label] = round(events(fn, iters), 3)
    r = {"shape": name, "match_ms": round(match_ms, 4), "post_ms": round(post_ms, 4), "post_launches": launches,
         "post_read_gb": round(rd / 1e9, 4), "post_written_gb": round(wr / 1e9, 4),
         "post_gbs": round((rd + wr) / post_ms / 1e6, 1), "post_frac_of_6555": round((rd + wr) / post_ms / 1e6 / PEAK_GBS, 4),
         "mean_distinct_rows": [round(x, 1) for x in distinct]}
    if parts:
        r["post_ms_by_outputs"] = parts
    print(json.dumps(r), flush=True)
    return r


def host_shape(iters):
    n = 1 << 18
    cfg = product_config("regex1", 1025)
    data = W.config1_torch(n).cpu().numpy().reshape(-1)
    offs = np.arange(n + 1, dtype=np.uint64) * 1024
    alloc = H.PinnedAllocator()
    want = {"states", "substr_ids", "start_enable", "end_enable", "masked_chars", "masked_substr_ids", "status", "mult", "endpoint_mult"}
    o1 = cfg.new_host_outputs(n, allocator=alloc, want=want)
    o2 = cfg.new_host_outputs(n, allocator=alloc, want=want)
    sm = H.StringMultOutputs(cfg, n, device="cpu", pin=True)
    plain = lambda: cfg.match_batch_host(data, offs, out=o1)  # noqa: E731
    mult = lambda: cfg.match_batch_host_mult(data, offs, out=o2, sm=sm)  # noqa: E731
    plain()
    pcie_plain = cfg.last_host_bytes()
    mult()
    pcie_mult = cfg.last_host_bytes()
    t = {"plain": [], "mult": []}
    for _ in range(iters):                                                # alternating
        for k, fn in (("plain", plain), ("mult", mult)):
            t0 = time.perf_counter()
            fn()
            t[k].append((time.perf_counter() - t0) * 1e3)
    for d in range(cfg.n_defs):
        assert np.array_equal(o1.mult[d], o2.mult[d])
    r = {"shape": "host regex1 2^18 x 1 KiB, pinned", "host_ms": round(float(np.median(t["plain"])), 3),
         "host_mult_ms": round(float(np.median(t["mult"])), 3), "max_entries": sm.max_entries,
         "h2d_d2h_bytes_plain": list(pcie_plain), "h2d_d2h_bytes_mult": list(pcie_mult)}
    print(json.dumps(r), flush=True)
    alloc.free()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    res = []
    n1 = 1 << 20
    offs1 = np.arange(n1 + 1, dtype=np.uint64) * 1024
    cfg = product_config("regex1", 1025)
    res.append(device_shape("regex1 2^20 x 1 KiB", cfg, W.config1_torch(n1).reshape(-1), offs1, args.iters, variants=True))
    del cfg
    cfg = product_config("three", 1025)
    res.append(device_shape("three 2^20 x 1 KiB", cfg, W.config2_torch(n1).reshape(-1), offs1, args.iters))
    del cfg
    n4 = 1 << 17
    cfg = large_dfa(4097)
    res.append(device_shape("1023-state DFA 2^17 x 4 KiB", cfg, W.config4_torch(n4).reshape(-1), np.arange(n4 + 1, dtype=np.uint64) * 4096, args.iters))
    del cfg
    cfg = product_config("regex1", 65537)
    res.append(device_shape("regex1 2048 x 64 KiB, chunked", cfg, W.config1_torch(2048, 65536).reshape(-1), np.arange(2049, dtype=np.uint64) * 65536,
                            args.iters, chunked=True))
    del cfg
    cfg = product_config("regex2", 1025)
    d3, _ = W.config3_torch(1 << 26)
    res.append(device_shape("regex2 one 64 MiB string", cfg, d3, np.array([0, 1 << 26], np.uint64), max(3, args.iters // 3), long=True))
    del cfg, d3
    torch.cuda.empty_cache()
    res.append(host_shape(max(3, args.iters // 2)))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "string_mult_bench.json"), "w") as f:
            json.dump({"gpu": info, "results": res}, f, indent=1)


if __name__ == "__main__":
    main()
