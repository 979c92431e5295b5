#!/usr/bin/env python3
"""Per-string lookup multiplicities, packed layout against slots.  Device: the b2r_string_mult post-pass (slots, max_entries =
max_d min(M, T_d)) against b2r_string_mult_packed (the same counting kernels, then scan and pack) on device-resident seeded
inputs, CUDA-event medians, alternating.  Host, end to end from pinned buffers with every column: b2r_match_batch_host_mult
against b2r_match_batch_host_mult_packed (and b2r_match_batch_host for reference), wall time and b2r_last_host_bytes.  The lists
of the two layouts are checked equal on every shape.  Prints the card and its power limit; --out DIR writes
string_mult_packed_bench.json there."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import halo2_regex_b200 as H  # noqa: E402
from conftest import product_config  # noqa: E402
from halo2_regex_b200 import workloads as W  # noqa: E402
from string_mult_bench import gpu_info, large_dfa  # noqa: E402


def same_lists(cfg, sm, pk):
    for d in range(cfg.n_defs):
        ne = sm.n_entries[d].cpu().numpy().view(np.uint32).astype(np.int64)
        rs = pk.row_start[d].cpu().numpy().view(np.uint64).astype(np.int64)
        assert rs[0] == 0 and np.array_equal(np.diff(rs), ne), d
        e = sm.entries[d].cpu().numpy().view(np.uint32)
        k = np.arange(sm.max_entries)[None, :] < ne[:, None]
        assert np.array_equal(e[k], pk.entries[d][:rs[-1]].cpu().numpy().view(np.uint32)), d
        if sm.endpoint_counts[d] is not None:
            assert torch.equal(sm.endpoint_counts[d].cpu(), pk.endpoint_counts[d].cpu()), d
    return [int(pk.row_start[d][-1]) for d in range(cfg.n_defs)]


def device_shape(name, cfg, d_bytes, offs_host, iters, chunked=False):
    n = len(offs_host) - 1
    out = H.DeviceOutputs(cfg, n, want={"states", "status"})
    d_offs = torch.from_numpy(offs_host.astype(np.int64)).cuda()
    (cfg.match_batch_chunked_device if chunked else cfg.match_batch_device)(d_bytes, d_offs, out)
    sm = H.StringMultOutputs(cfg, n)
    pk = H.StringMultPacked(cfg, n)
    slot = lambda: cfg.string_mult_device(d_bytes, d_offs, out, sm)  # noqa: E731
    packed = lambda: cfg.string_mult_packed_device(d_bytes, d_offs, out, pk)  # noqa: E731
    slot(); packed(); torch.cuda.synchronize()                           # warm-up, workspaces sized
    assert cfg.batch_result(check=False).code == 0
    t = {"slot": [], "packed": []}
    for _ in range(iters):                                                # alternating
        for k, fn in (("slot", slot), ("packed", packed)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            t[k].append(a.elapsed_time(b))
    launches = cfg.last_launch_count()
    totals = same_lists(cfg, sm, pk)
    r = {"shape": name, "slot_ms": round(float(np.median(t["slot"])), 3), "packed_ms": round(float(np.median(t["packed"])), 3),
         "packed_launches": launches, "slot_area_gb": round(sum(n * sm.max_entries * 8 for _ in range(cfg.n_defs)) / 1e9, 3),
         "packed_entries_gb": round(sum(totals) * 8 / 1e9, 3)}
    print(json.dumps(r), flush=True)
    return r


def host_shape(name, cfg, data, offs, iters):
    n = len(offs) - 1
    alloc = H.PinnedAllocator()
    want = {"states", "substr_ids", "start_enable", "end_enable", "masked_chars", "masked_substr_ids", "status", "mult", "endpoint_mult"}
    o = [cfg.new_host_outputs(n, allocator=alloc, want=want) for _ in range(3)]
    sm = H.StringMultOutputs(cfg, n, device="cpu", pin=True)
    pk = H.StringMultPacked(cfg, n, device="cpu", pin=True)
    calls = {"plain": lambda: cfg.match_batch_host(data, offs, out=o[0]),
             "mult": lambda: cfg.match_batch_host_mult(data, offs, out=o[1], sm=sm),
             "mult_packed": lambda: cfg.match_batch_host_mult_packed(data, offs, out=o[2], pk=pk)}
    pcie, t = {}, {k: [] for k in calls}
    for k, fn in calls.items():
        fn()
        pcie[k] = [round(x / 1e9, 3) for x in cfg.last_host_bytes()]
    for _ in range(iters):                                                # alternating
        for k, fn in calls.items():
            t0 = time.perf_counter()
            fn()
            t[k].append((time.perf_counter() - t0) * 1e3)
    for d in range(cfg.n_defs):
        assert np.array_equal(o[1].mult[d], o[2].mult[d]) and np.array_equal(o[0].mult[d], o[2].mult[d])
    totals = same_lists(cfg, sm, pk)
    r = {"shape": name, **{f"{k}_ms": round(float(np.median(v)), 2) for k, v in t.items()}, **{f"{k}_h2d_d2h_gb": v for k, v in pcie.items()},
         "mean_rows_per_string": [round(x / n, 1) for x in totals]}
    print(json.dumps(r), flush=True)
    del o, sm, pk
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
    res.append(device_shape("regex1 2^20 x 1 KiB", cfg, W.config1_torch(n1).reshape(-1), offs1, args.iters))
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
    torch.cuda.empty_cache()
    n = 1 << 18
    offs = np.arange(n + 1, dtype=np.uint64) * 1024
    hi = max(3, args.iters // 2)
    res.append(host_shape("host regex1 2^18 x 1 KiB, pinned", product_config("regex1", 1025), W.config1_torch(n).cpu().numpy().reshape(-1), offs, hi))
    res.append(host_shape("host three 2^18 x 1 KiB, pinned", product_config("three", 1025), W.config2_torch(n).cpu().numpy().reshape(-1), offs, hi))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "string_mult_packed_bench.json"), "w") as f:
            json.dump({"gpu": info, "results": res}, f, indent=1)


if __name__ == "__main__":
    main()
