#!/usr/bin/env python3
"""b2r_match_batch_host against b2r_match_batch_chunked_host, end to end from host memory: the same seeded inputs; input bytes,
offsets and outputs in page-locked host memory (b2r_host_alloc); the two calls alternating in one process (one handle each, so
that B2R_OUT_SPARSE_REUSE finds the record of its own previous call).  Two rows per shape: `SPARSE_D2H | SPARSE_REUSE`, then
dense D2H.  The outputs of the two calls are checked equal on every row.  Prints one JSON line per row and the card (name, power
limit, max SM clock); --out DIR writes them to one file.  Development aid: it measures what slicing long strings by bytes gains
over the batch path's pipeline."""
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
from conftest import DEF_SETS, DEFS  # noqa: E402
from halo2_regex_b200 import _abi  # noqa: E402
from halo2_regex_b200 import workloads as W  # noqa: E402
from chunked_bench import gpu_info  # noqa: E402

# (n strings, M, devices): the regex1 shapes of tools/chunked_bench.py, then 2048 x 64 KiB on 2 and 4 GPUs
SHAPES = [(2048, 65537, 1), (256, 262145, 1), (16384, 8193, 1), (1 << 17, 1025, 1), (2048, 65537, 2), (2048, 65537, 4)]


def handle(M, n_dev):
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(os.path.join(DEFS, a)), [H.SubstrRegexDef.read_from_text(os.path.join(DEFS, s)) for s in ss])
            for a, ss in DEF_SETS["regex1"]]
    return H.RegexVerifyConfig.configure(M, defs, devices=list(range(n_dev)) if n_dev > 1 else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5, help="timed calls per entry point and row (after one warm-up call)")
    ap.add_argument("--out", default=None, help="directory for chunked_host_bench.json")
    ap.add_argument("--only", default=None, help="comma-separated shape indices")
    args = ap.parse_args()
    assert args.iters >= 5, "the median of at least 5 calls"
    shapes = [SHAPES[int(i)] for i in args.only.split(",")] if args.only else SHAPES
    info = gpu_info()
    print(json.dumps({"gpu": info, "device_count": torch.cuda.device_count()}), flush=True)
    rows = []
    for n, M, n_dev in shapes:
        if torch.cuda.device_count() < n_dev:
            print(json.dumps({"n": n, "M": M, "devices": n_dev, "skipped": "not enough GPUs"}), flush=True)
            continue
        L = M - 1
        cfgs = {"host": handle(M, n_dev), "chunked_host": handle(M, n_dev)}
        calls = {"host": cfgs["host"].match_batch_host, "chunked_host": cfgs["chunked_host"].match_batch_chunked_host}
        alloc = H.PinnedAllocator()
        try:
            # inputs in page-locked memory too: a pageable source is staged by the driver, which blocks the calling thread per copy
            data = alloc(n * L)
            data[:] = W.config1_numpy(n, L)[0].reshape(-1)
            offs = alloc(8 * (n + 1)).view(np.uint64)
            offs[:] = np.arange(n + 1, dtype=np.uint64) * L
            outs = {k: cfgs[k].new_host_outputs(n, fill=0, allocator=alloc, max_records=8, compact_pitch=64) for k in calls}
            for mode, sparse in (("sparse_reuse", True), ("dense", False)):
                times = {k: [] for k in calls}
                stats = {}
                for it in range(args.iters + 1):               # the first round warms up (workspaces, pinned arenas, modules)
                    for k in calls:
                        t0 = time.perf_counter()
                        _, res = calls[k](data, offs, out=outs[k], check=False, sparse=sparse, reuse=sparse and it > 0)
                        ms = (time.perf_counter() - t0) * 1e3      # the call synchronises before it returns
                        if it:
                            times[k].append(ms)
                        h2d, d2h = cfgs[k].last_host_bytes()
                        stats[k] = {"code": res.code, "launches": cfgs[k].last_launch_count(), "h2d_bytes": h2d, "d2h_bytes": d2h}
                equal = all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(outs["host"].all_arrays(), outs["chunked_host"].all_arrays()))
                row = {"n": n, "M": M, "devices": n_dev, "d2h": mode, "input_bytes": n * L, "outputs_equal": equal}
                for k in calls:
                    med = sorted(times[k])[len(times[k]) // 2]
                    row[k] = dict(stats[k], ms_median=round(med, 3), ms_all=[round(t, 3) for t in times[k]], input_GBps=round(n * L / med / 1e6, 2))
                row["speedup_chunked_host"] = round(row["host"]["ms_median"] / row["chunked_host"]["ms_median"], 3)
                print(json.dumps(row), flush=True)
                rows.append(row)
        finally:
            outs = data = offs = None                          # the arrays live in the pinned blocks freed here
            alloc.free()
        del cfgs, calls
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "chunked_host_bench.json"), "w") as f:
            json.dump({"gpu": info, "iters": args.iters, "flags": {"sparse_reuse": _abi.B2R_OUT_SPARSE_D2H | _abi.B2R_OUT_SPARSE_REUSE, "dense": 0},
                       "rows": rows}, f, indent=1)
    assert all(r["outputs_equal"] for r in rows), "b2r_match_batch_chunked_host outputs differ from b2r_match_batch_host"


if __name__ == "__main__":
    main()
