#!/usr/bin/env python3
"""b2r_match_batch against b2r_match_batch_chunked on the same device-resident seeded inputs, the two calls alternating in one
process; the outputs of the two are checked equal on every shape.  Writes one JSON file to --out DIR (ms per call, input GB/s,
launches, the card and its power limit / max SM clock).  Development aid: it measures where the chunked path starts to pay off."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import torch  # noqa: E402

import halo2_regex_b200 as H  # noqa: E402
from conftest import product_config  # noqa: E402
from halo2_regex_b200 import workloads as W  # noqa: E402

SHAPES = [("regex1", 2048, 65537), ("regex1", 256, 262145), ("regex1", 16384, 8193), ("regex1", 1 << 17, 1025), ("large_dfa", 512, 65537)]


def handle(which, M):
    if which == "large_dfa":
        allstr, substr, _ = W.large_dfa_texts()
        return H.RegexVerifyConfig.configure(M, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])])
    return product_config(which, M)


def tensors(out):
    cols = list(out.states) + list(out.substr_ids) + list(out.start_enable) + list(out.end_enable)
    cols += [out.masked_chars, out.masked_substr_ids, out.status, out.records, out.compact_bytes, out.mult_all]
    return [t for t in cols if t is not None]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"card": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as e:  # noqa: BLE001
        return {"card": torch.cuda.get_device_name(0), "nvidia_smi": f"unavailable: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for chunked_bench.json")
    ap.add_argument("--only", default=None, help="comma-separated shape indices")
    args = ap.parse_args()
    rows = []
    shapes = [SHAPES[int(i)] for i in args.only.split(",")] if args.only else SHAPES
    for which, n, M in shapes:
        L = M - 1
        d = (W.config4_torch(n, L) if which == "large_dfa" else W.config1_torch(n, L)).reshape(-1)
        offs = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
        cfg = handle(which, M)
        outs = {k: H.DeviceOutputs(cfg, n, max_records=8, compact_pitch=64) for k in ("batch", "chunked")}
        for o in outs.values():
            for t in tensors(o):
                t.zero_()
        calls = {"batch": cfg.match_batch_device, "chunked": cfg.match_batch_chunked_device}
        times = {"batch": [], "chunked": []}
        launches = {}
        for it in range(args.iters + 1):                   # the first round warms up (workspace, module load)
            for k in ("batch", "chunked"):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                calls[k](d, offs, outs[k])
                e1.record()
                res = cfg.batch_result(check=False)
                launches[k] = cfg.last_launch_count()
                if it:
                    times[k].append(e0.elapsed_time(e1))
        equal = all(torch.equal(x, y) for x, y in zip(tensors(outs["batch"]), tensors(outs["chunked"])))
        row = {"set": which, "n": n, "M": M, "input_bytes": n * L, "code": res.code, "outputs_equal": equal}
        for k in ("batch", "chunked"):
            ms = sorted(times[k])[len(times[k]) // 2]
            row[k] = {"ms_median": ms, "ms_all": times[k], "input_GBps": n * L / ms / 1e6, "launches": launches[k]}
        row["speedup_chunked"] = row["batch"]["ms_median"] / row["chunked"]["ms_median"]
        print(json.dumps(row), flush=True)
        rows.append(row)
        del outs, d
        torch.cuda.empty_cache()
    doc = {"gpu": gpu_info(), "iters": args.iters, "rows": rows}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "chunked_bench.json"), "w") as f:
            json.dump(doc, f, indent=1)
    assert all(r["outputs_equal"] for r in rows), "chunked outputs differ from b2r_match_batch"


if __name__ == "__main__":
    main()
