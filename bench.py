#!/usr/bin/env python3
"""bench.py — BASELINE.json's metric on BASELINE.json's configs, B200 arm and reference (CPU) arm.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle) on the host cores
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed as DIR/*.npy

metric   : input bytes/sec of DFA witness generation (state column, substr ids, enable bitmaps, masked chars/ids,
           status, records, lookup multiplicities) — bit-exact outputs, see tests/.
headline : BASELINE.json configs[1]: test_regexes regex1_test lookup + substr1, 2^20 synthetic 1 KiB strings per GPU,
           max_chars_size M = 1025 (SURVEY 8(d) config 1).  N > 1: every rank owns 2^20 strings of the same global batch
           (weak scaling, strings are independent); the only exchange is ONE NCCL all-reduce of the multiplicity counters per
           job (the counters are additive: every step accumulates, the K-step job reduces once, inside the timed region).
A step   : one pass of the hot path over the rank's batch.  `value` times it with the inputs resident in HBM; `e2e` times
           the reference-facing C-ABI call b2r_match_batch_host with pinned HOST buffers (H2D and D2H inside the region).
configs  : the other BASELINE configs as sub-records of the same line — "2i"/"2ii" (regex3 + substr1-3, both readings of
           SURVEY 8(d)), "3" (one 64 MiB string, rank 0), "4" (>= 512-state DFA, 2^19 x 4 KiB per GPU) — each with its own
           device-timed ms/step, kernel time, algorithmic bytes, roofline fraction, table/bin placement and parity flags.
parity   : outside every timed region: a 256-string tile of every column of every config against the CPU oracle, bit-exact
           (the checker, never the thing measured); sum(mult) == rows; N > 1: the all-reduced counters row by row against the
           host sum of the all-gathered per-rank counters.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DEFS = os.path.join(ROOT, "tests", "golden", "defs")

LOG2_STRINGS = 20          # per GPU
STRING_LEN = 1024
M = STRING_LEN + 1
METRIC = "input bytes/sec (DFA witness gen)"
UNIT = "GB/s"
REF_SAMPLE_LOG2 = 14       # strings per step of the CPU arm (a bounded sample of the same batch)


def workload_config(log2_strings):
    """The `config` object of both arms: names the workload only (identical for --impl b200 and --impl reference)."""
    return {"workload": "regex1_test + substr1, 2^%d x 1 KiB strings per GPU, M=1025 (BASELINE configs[1])" % log2_strings,
            "strings_per_gpu": 1 << log2_strings, "string_len": STRING_LEN, "max_chars_size": M, "defs": 1, "states": 29,
            "l2_policy": "inputs (1 GiB) + outputs (4.6 GB) per step exceed the 126 MB L2; no flush needed"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled every ~5 ms through NVML while the timed region runs."""

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.stop_flag, self.t, self.err = gpu_index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                try:
                    self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
                except Exception:
                    pass
            time.sleep(0.005)

    def stop(self):
        if self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {self.err}"]}
        self.stop_flag = True
        self.t.join(timeout=2)
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": [k for k, v in names.items() if bits & v], "samples": len(sm)}


def def_paths(spec):
    return [(os.path.join(DEFS, a), [os.path.join(DEFS, s) for s in ss]) for a, ss in spec]


SET_REGEX1 = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"])]
SET_REGEX2 = [("regex2_test_lookup.txt", ["substr2_test_lookup.txt"])]
SET_2I = [("regex3_test_lookup.txt", ["substr1_test_lookup.txt", "substr2_test_lookup.txt", "substr3_test_lookup.txt"])]
SET_2II = [("regex1_test_lookup.txt", ["substr1_test_lookup.txt"]), ("regex2_test_lookup.txt", ["substr2_test_lookup.txt"]),
           ("regex3_test_lookup.txt", ["substr3_test_lookup.txt"])]


def oracle_from_files(spec, m):
    from oracle import oracle as O
    return O.OracleConfig([(O.OracleAllstr.read_from_text(a), [O.OracleSubstr.read_from_text(s) for s in ss]) for a, ss in def_paths(spec)], m)


def oracle_from_texts(allstr, substr, m):
    from oracle import oracle as O
    return O.OracleConfig([(O.OracleAllstr(allstr), [O.OracleSubstr(substr)])], m)


def reference_arm(args):
    """The reference's own CPU algorithm (oracle/oracle.c restatement; the Rust crate cannot be built in this image),
    all host threads, one bounded sample of the same workload per step.  Imports nothing of the product package."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import workloads as W
    cores = os.cpu_count() or 1
    cfg = oracle_from_files(SET_REGEX1, M)
    n = 1 << REF_SAMPLE_LOG2
    data, _ = W.config1_numpy(n, STRING_LEN)
    offs = np.arange(n + 1, dtype=np.uint64) * STRING_LEN
    out = cfg.new_outputs(n, max_records=2, compact_pitch=8)
    flat = data.reshape(-1)
    for _ in range(args.warmup):
        cfg.match_batch(flat, offs, out=out, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cfg.match_batch(flat, offs, out=out, nthreads=cores)
    dt = time.perf_counter() - t0
    gbs = n * STRING_LEN * args.steps / dt / 1e9
    sample = (f"each step walks the first 2^{REF_SAMPLE_LOG2} of the config's 2^{args.log2_strings} strings x {STRING_LEN} B (16 MiB) on {cores} threads: "
              "all witness columns + multiplicities; bytes/s is size-independent for this per-string algorithm")
    assert "halo2_regex_b200" not in sys.modules, "the CPU arm must not load the product package"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.log2_strings),
        "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "C restatement of src/lib.rs:311-888 without halo2 cell assignment / field inversions: faster than the real reference"},
        "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


class Ctx:
    """torch / distributed plumbing shared by the legs of the B200 arm."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"          # the version banner goes to stdout, which carries the JSON line
            dist.init_process_group("nccl", device_id=self.dev)
        assert self.world == args.gpus or self.world == 1, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        self.peak, self.peak_src = measured_peak()

    def stream(self):
        return self.torch.cuda.current_stream(self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok):
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t.item()))

    def timed(self, step, steps, tail=None):
        """barrier + sync, `steps` calls of step() (+ tail()) between two CUDA events on the launching stream, barrier + sync;
        returns (total ms, max over ranks; sorted per-step ms of this rank)."""
        torch = self.torch
        st = self.stream()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        t_begin.record(st)
        for i in range(steps):
            ev[i][0].record(st)
            step()
            ev[i][1].record(st)
        if tail is not None:
            tail()
        t_end.record(st)
        self.barrier()
        return self.max_over_ranks(t_begin.elapsed_time(t_end)), sorted(a.elapsed_time(b) for a, b in ev)


def tile_to_host(H, cfg, out, lo, cnt):
    """Rows [lo, lo+cnt) of every per-string column of a DeviceOutputs as a HostOutputs (no multiplicities)."""
    import numpy as np
    want = set(out.want) - {"mult", "endpoint_mult"}
    h = H.HostOutputs(cnt, out.m, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, row_pitch=out.row_pitch, bitmap_pitch=out.bitmap_pitch,
                      max_records=out.max_records, compact_pitch=out.compact_pitch, want=want)

    def cp(dst, src):
        if dst is not None and src is not None:
            dst.view(np.uint8).reshape(-1)[:] = src[lo:lo + cnt].contiguous().view(-1).view(dtype=__import__("torch").uint8).cpu().numpy()

    for d in range(cfg.n_defs):
        cp(h.states[d], out.states[d]); cp(h.substr_ids[d], out.substr_ids[d])
        cp(h.start_enable[d], out.start_enable[d]); cp(h.end_enable[d], out.end_enable[d])
    cp(h.masked_chars, out.masked_chars); cp(h.masked_substr_ids, out.masked_substr_ids)
    cp(h.status, out.status); cp(h.records, out.records); cp(h.compact_bytes, out.compact_bytes)
    return h


def oracle_tile_check(H, cfg, ocfg, d_bytes, L, out, lo, cnt=256):
    """Strings [lo, lo+cnt) of the batch the GPU just processed: every column bit-exact against the CPU oracle on the same bytes."""
    import numpy as np
    cnt = min(cnt, out.n - lo)
    hb = d_bytes[lo * L:(lo + cnt) * L].cpu().numpy()
    offs = np.arange(cnt + 1, dtype=np.uint64) * L
    want = set(out.want) - {"mult", "endpoint_mult"}
    o, _ = ocfg.match_batch(hb, offs, row_pitch=out.row_pitch, bitmap_pitch=out.bitmap_pitch, max_records=out.max_records, compact_pitch=out.compact_pitch, want=want)
    g = tile_to_host(H, cfg, out, lo, cnt)
    errs = H.compare_outputs(g, o)
    if errs:
        print(f"[bench] PARITY FAILURE (strings {lo}..{lo + cnt}): {errs[:3]}", file=sys.stderr)
    return not errs


DUMP_STRINGS = 1024        # strings in the --dump-outputs sample: ~25 MB as float32 for config 1
DUMP_SEED = 0xB200D0       # the sample is the same strings in every run


def dump_outputs(out, directory):
    """--dump-outputs: the witness of the timed path's last step as DIR/<name>.npy (float32, counters float64) — every column
    of a fixed, seeded sample of the batch's strings, restricted to what include/b2r.h defines (rows [0, M), the first
    n_records records, the first n_compact compacted bytes; the rest of each buffer is left unspecified and zeroed here), and
    every multiplicity counter of the batch."""
    import numpy as np
    import torch
    from b2r_layout import abi as _abi
    os.makedirs(directory, exist_ok=True)
    n, m = out.n, out.m
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_STRINGS), replace=False))
    rows = torch.from_numpy(idx).to(out.mult_all.device)

    def take(t):
        a = t.index_select(0, rows).cpu().numpy()
        return a.view(np.uint16) if a.dtype == np.int16 else a

    def bits(t):
        return np.unpackbits(take(t), axis=1, bitorder="little")[:, :m]

    arrays = {"string_index": idx.astype(np.float64)}
    for d in range(out.cfg.n_defs):
        arrays[f"states{d}"] = take(out.states[d])[:, :m]
        arrays[f"substr_ids{d}"] = take(out.substr_ids[d])[:, :m]
        arrays[f"start_enable{d}"] = bits(out.start_enable[d])
        arrays[f"end_enable{d}"] = bits(out.end_enable[d])
        arrays[f"mult{d}"] = out.mult[d].cpu().numpy().astype(np.float64)
        arrays[f"endpoint_mult{d}"] = out.endpoint_mult[d].cpu().numpy().astype(np.float64)
    arrays["masked_chars"] = take(out.masked_chars)[:, :m]
    arrays["masked_substr_ids"] = take(out.masked_substr_ids)[:, :m]
    status = take(out.status).reshape(-1).view(_abi.STATUS_DTYPE)
    for f in ("flags", "err_pos", "err_state", "err_byte", "err_def", "n_records", "n_compact"):
        arrays["status_" + f] = status[f].astype(np.float64)
    records = take(out.records).view(_abi.RECORD_DTYPE).reshape(len(idx), out.max_records)
    records = np.stack([records[f] for f, _ in _abi.RECORD_DTYPE], axis=-1).astype(np.float64)
    records[np.arange(out.max_records)[None, :] >= status["n_records"][:, None]] = 0
    arrays["records"] = records
    compact = take(out.compact_bytes).astype(np.float32)
    compact[np.arange(out.compact_pitch)[None, :] >= status["n_compact"][:, None]] = 0
    arrays["compact_bytes"] = compact
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def gathered_mult_check(ctx, local, reduced):
    """N > 1: the all-reduced counters against the host sum of the all-gathered per-rank counters, row by row."""
    if ctx.world == 1:
        return None
    torch, dist = ctx.torch, ctx.dist
    parts = [torch.empty_like(local) for _ in range(ctx.world)]
    dist.all_gather(parts, local)
    host_sum = sum(p.cpu().numpy().astype("uint64") for p in parts)
    return bool((host_sum == reduced.cpu().numpy().astype("uint64")).all())


def batch_leg(ctx, H, W, key, workload, cfg, ocfg, d_bytes, n, L, m, steps, warmup, max_records=2, compact_pitch=8, dump_dir=None):
    """One batch config with the inputs resident in HBM: device-timed steps, the kernel alone, parity checks; `dump_dir`: where
    dump_outputs() writes what the last timed step computed."""
    import numpy as np
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    from halo2_regex_b200 import _abi
    from halo2_regex_b200.sharded import allreduce_multiplicities
    d_offs = torch.arange(n + 1, dtype=torch.int64, device=dev) * L
    out = H.DeviceOutputs(cfg, n, max_records=max_records, compact_pitch=compact_pitch, max_chars_size=m)
    in_bytes = n * L
    algo_bytes = in_bytes + (n + 1) * 8 + out.written_bytes()      # input + offsets read, every witness column written (M rows/string)
    flags = _abi.B2R_OUT_ACCUMULATE_MULT if world > 1 else 0

    def enqueue():
        cfg.match_batch_device(d_bytes, d_offs, out, flags=flags, stream=torch.cuda.current_stream(dev))

    for _ in range(warmup):
        enqueue()
    assert cfg.batch_result(stream=ctx.stream()).code == 0
    launches_per_step = cfg.last_launch_count()
    # one step = a handful of launches (memset nodes, walk_kernel, finalize_kernel) captured in ONE CUDA graph; the collective stays outside
    graph = None
    if not ctx.args.no_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                enqueue()
            graph.replay()
            torch.cuda.synchronize()
        except Exception as e:  # pragma: no cover
            print(f"[bench] CUDA graph capture failed ({e!r}); timing plain launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
    step = graph.replay if graph is not None else enqueue
    for _ in range(2):
        step()
    out.mult_all.zero_()
    local = {}

    def tail():     # the job's only exchange: ONE all-reduce of the accumulated counters over NVLink
        if world > 1:
            local["mult"] = out.mult_all.clone()
            allreduce_multiplicities(out.mult + out.endpoint_mult)

    sampler = ClockSampler(ctx.local_rank) if (rank == 0 and key == "1") else None
    if sampler:
        sampler.start()          # before the barrier: NVML start-up on rank 0 must not delay its first step
    if key == "1":
        torch.cuda.profiler.start()      # `ncu --profile-from-start off` lists exactly the launches of the timed region
    total_ms, step_ms = ctx.timed(step, steps, tail)
    if key == "1":
        torch.cuda.profiler.stop()
    clocks = sampler.stop() if sampler else None
    assert cfg.batch_result(stream=ctx.stream()).code == 0
    if dump_dir:
        dump_outputs(out, dump_dir)

    # ---- parity, outside the timed region -------------------------------------------------------------------------------------
    reduced = out.mult_all.clone()
    jobs = steps if world > 1 else 1                                   # accumulated steps
    mult_sum_ok = all(int(out.mult[d].cpu().numpy().astype(np.uint64).sum()) == n * m * jobs * world for d in range(cfg.n_defs))
    gathered_ok = gathered_mult_check(ctx, local["mult"], reduced) if world > 1 else None
    tile_lo = ((rank * 7919 + 13) * 256) % max(n - 256, 1) // 32 * 32    # a different tile on every rank
    tile_ok = oracle_tile_check(H, cfg, ocfg, d_bytes, L, out, tile_lo) and oracle_tile_check(H, cfg, ocfg, d_bytes, L, out, max(n - 256, 0))
    parity = {"oracle_tile_bit_exact": ctx.all_true(tile_ok), "tile": f"strings [{tile_lo}, +256) and the last 256 of every rank, all columns, status, records, compact bytes",
              "mult_sum_equals_rows": ctx.all_true(mult_sum_ok), "allreduce_rows_equal_gathered_host_sum": gathered_ok}

    # ---- the dominant kernel alone (walk_kernel with the emit stage fused in): CUDA events on the launching stream inside the library
    cfg.set_timing(True)
    stages = []
    for _ in range(min(steps, 5)):
        cfg.match_batch_device(d_bytes, d_offs, out, stream=ctx.stream())
        cfg.batch_result(stream=ctx.stream())
        stages.append(cfg.last_stage_ms())
    cfg.set_timing(False)
    # fused: walk_kernel is the whole path.  Emit stage as its own kernel (several defs, large DFAs): the algorithmic bytes are written by
    # walk_kernel AND emit_kernel, so the roofline fraction is taken over both
    split = launches_per_step >= 3
    walk_only_ms = sum(x[0] for x in stages) / len(stages)
    walk_ms = sum(x[0] + (x[1] if split else 0.0) for x in stages) / len(stages)
    plan = cfg.last_plan()
    achieved = algo_bytes / (walk_ms * 1e-3) / 1e9
    rec = {"workload": workload, "strings_per_gpu": n, "string_len": L, "max_chars_size": m, "defs": cfg.n_defs, "states": [int(x) for x in cfg.dummy_states],
           "value": world * in_bytes * steps / (total_ms * 1e-3) / 1e9, "unit": UNIT, "steps": steps, "ms_per_step": total_ms / steps,
           "step_ms_median": step_ms[len(step_ms) // 2], "kernel_ms": walk_ms,
           "stage_ms": {"walk_kernel": walk_only_ms, "emit_kernel": sum(x[1] for x in stages) / len(stages), "finalize": sum(x[2] for x in stages) / len(stages)},
           "emit_stage": "its own kernel after the walk (the walk zero-fills)" if split else "fused into walk_kernel",
           "algorithmic_bytes_per_launch": algo_bytes, "bytes_per_input_byte": algo_bytes / in_bytes, "achieved_gbs": achieved, "frac": achieved / ctx.peak,
           "table_placement": plan[0], "bin_placement": plan[1], "kernels_per_step": launches_per_step, "cuda_graph": graph is not None, "parity": parity}
    return rec, out, d_offs, clocks


def long_leg(ctx, H, W, steps, warmup):
    """BASELINE configs[3]: ONE 64 MiB string through regex2_test (b2r_match_long), rank 0 only."""
    import numpy as np
    torch, dev = ctx.torch, ctx.dev
    length = 1 << ctx.args.log2_long
    m = length + 1
    cfg = make_config(H, SET_REGEX2, 64, ctx.local_rank)
    d, at = W.config3_torch(length, device=dev)
    out = H.DeviceOutputs(cfg, 1, max_records=8, compact_pitch=64, max_chars_size=m)
    algo_bytes = length + out.written_bytes()
    st = ctx.stream()

    def enqueue():
        cfg.match_long_device(d, out, stream=torch.cuda.current_stream(dev))

    for _ in range(warmup):
        enqueue()
    assert cfg.batch_result(stream=st).code == 0
    launches = cfg.last_launch_count()
    # the step (five kernels, the memset nodes of the sparse columns on a side branch) as ONE CUDA graph, like the batch path
    graph = None
    if not ctx.args.no_graph:
        try:
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                enqueue()
            graph.replay()
            torch.cuda.synchronize()
        except Exception as e:  # pragma: no cover
            print(f"[bench] CUDA graph capture of the long-string step failed ({e!r}); timing plain launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    step = graph.replay if graph is not None else enqueue
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    torch.cuda.synchronize()
    for i in range(steps):
        ev[i][0].record(st); step(); ev[i][1].record(st)
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    ms_step = sum(ms) / len(ms)
    assert cfg.batch_result(stream=st).code == 0
    # parity: the whole string against the CPU oracle (a few seconds of CPU), every column
    ok = None
    if not ctx.args.no_long_oracle:
        ocfg = oracle_from_files(SET_REGEX2, m)
        hb = d.cpu().numpy()
        o, _ = ocfg.match_batch(hb, np.array([0, length], dtype=np.uint64), row_pitch=out.row_pitch, bitmap_pitch=out.bitmap_pitch, max_records=8, compact_pitch=64)
        g = out.to_host()
        errs = H.compare_outputs(g, o)
        if errs:
            print(f"[bench] PARITY FAILURE (long string): {errs[:3]}", file=sys.stderr)
        ok = not errs
    mult_ok = int(out.mult[0].cpu().numpy().astype(np.uint64).sum()) == m
    achieved = algo_bytes / (ms_step * 1e-3) / 1e9
    return {"workload": f"ONE {length >> 20} MiB string through regex2_test + substr2 (chunked parallel-prefix composition of the transition vectors), "
                        f"` Also for xyz.` planted at offset {at}; M = len + 1 (BASELINE configs[3]); rank 0 only",
            "string_len": length, "max_chars_size": m, "defs": 1, "states": [13], "value": length / (ms_step * 1e-3) / 1e9, "unit": UNIT, "steps": steps,
            "ms_per_step": ms_step, "step_ms_min": ms[0], "kernels_per_step": launches, "cuda_graph": graph is not None, "algorithmic_bytes_per_launch": algo_bytes,
            "achieved_gbs": achieved, "frac": achieved / ctx.peak, "frac_note": "whole step (every launch of the path), not one kernel",
            "parity": {"oracle_whole_string_bit_exact": ok, "mult_sum_equals_rows": mult_ok}}


def make_config(H, spec, m, device, devices=None):
    defs = [H.RegexDefs(H.AllstrRegexDef.read_from_text(a), [H.SubstrRegexDef.read_from_text(s) for s in ss]) for a, ss in def_paths(spec)]
    return H.RegexVerifyConfig.configure(m, defs, device=device, devices=devices)


def e2e_leg(ctx, H, cfg, d_bytes, n, L, steps):
    """The reference-facing call: b2r_match_batch_host with pinned HOST buffers, dense and sparse D2H."""
    import numpy as np
    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    in_bytes = n * L
    ok, res = 1, {}
    try:
        alloc = H.PinnedAllocator()                                     # b2r_host_alloc: what a host without PyTorch would use
        h_in = alloc(in_bytes)
        h_in[:] = d_bytes.cpu().numpy()
        h_offs = alloc((n + 1) * 8).view(np.uint64)
        h_offs[:] = np.arange(n + 1, dtype=np.uint64) * L
        hout = H.HostOutputs(n, M, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, max_records=2, compact_pitch=8, allocator=alloc)
        cfg.match_batch_host(h_in, h_offs, out=hout)                    # warm-up (device staging allocation)
        cfg.match_batch_host(h_in, h_offs, out=hout, sparse=True)
    except Exception as exc:  # pragma: no cover
        print(f"[bench] end-to-end arm: set-up failed on rank {rank}: {exc!r}", file=sys.stderr)
        ok = 0
    if not ctx.all_true(ok):
        return None
    for mode, sparse, reuse in (("dense", False, False), ("sparse", True, False), ("sparse_reuse", True, True)):
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            cfg.match_batch_host(h_in, h_offs, out=hout, sparse=sparse, reuse=reuse)
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        h2d, d2h = cfg.last_host_bytes()
        assert int(hout.mult[0].sum()) == n * M
        res[mode] = {"value": world * in_bytes * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
                     "ms_per_step": dt / steps * 1e3}
    # the modes must hand the caller the same bytes: a sampled checksum of every column of the last sparse call against a dense one
    sums_sparse = [int(np.add.reduce(a.view(np.uint8).reshape(-1)[::1 << 6].astype(np.uint64))) for a in hout.all_arrays()]
    cfg.match_batch_host(h_in, h_offs, out=hout)
    sums_dense = [int(np.add.reduce(a.view(np.uint8).reshape(-1)[::1 << 6].astype(np.uint64))) for a in hout.all_arrays()]
    e2e = dict(res["sparse_reuse"])
    e2e["api"] = ("b2r_match_batch_host (include/b2r.h), flags = B2R_OUT_SPARSE_D2H | B2R_OUT_SPARSE_REUSE, pinned host buffers from b2r_host_alloc reused batch "
                  "after batch; every column lands dense in the caller's buffers")
    e2e["sparse_fresh_buffers"] = res["sparse"]
    e2e["dense_d2h"] = res["dense"]
    e2e["sparse_equals_dense_sampled_checksum"] = ctx.all_true(sums_sparse == sums_dense)
    alloc.free()
    return e2e


def multi_device_leg(ctx, H, W, n_per_dev_log2=18):
    """The single-process path of the C ABI (b2r_config_new_multi): rank 0 drives every GPU of the box from one process."""
    import numpy as np
    world = ctx.world
    n = world << n_per_dev_log2
    cfg = make_config(H, SET_REGEX1, M, None, devices=list(range(world)))
    alloc = H.PinnedAllocator()
    data, _ = W.config1_numpy(1 << 14, STRING_LEN)
    h_in = alloc(n * STRING_LEN).reshape(n, STRING_LEN)
    for lo in range(0, n, 1 << 14):
        h_in[lo:lo + (1 << 14)] = data
    h_offs = alloc((n + 1) * 8).view(np.uint64)
    h_offs[:] = np.arange(n + 1, dtype=np.uint64) * STRING_LEN
    hout = H.HostOutputs(n, M, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, max_records=2, compact_pitch=8, allocator=alloc)
    flat = h_in.reshape(-1)
    cfg.match_batch_host(flat, h_offs, out=hout, sparse=True)
    cfg.match_batch_host(flat, h_offs, out=hout, sparse=True, reuse=True)
    t0 = time.perf_counter()
    steps = 3
    for _ in range(steps):
        cfg.match_batch_host(flat, h_offs, out=hout, sparse=True, reuse=True)
    dt = (time.perf_counter() - t0) / steps
    # parity: the batch is 2^14 distinct strings repeated; every 2^14-string period of every column must be identical, and the
    # all-reduced counters must be (n / 2^14) x those of one period run on one device
    one = make_config(H, SET_REGEX1, M, 0)
    ref, _ = one.match_batch_host(flat[:(1 << 14) * STRING_LEN], h_offs[:(1 << 14) + 1], max_records=2, compact_pitch=8)
    reps = n >> 14
    ok = bool((hout.mult[0] == ref.mult[0] * np.uint64(reps)).all() and (hout.endpoint_mult[0] == ref.endpoint_mult[0] * np.uint64(reps)).all())
    for k in (0, reps // 2, reps - 1):
        sl = slice(k << 14, (k + 1) << 14)
        ok = ok and bool((hout.states[0][sl] == ref.states[0]).all() and (hout.masked_chars[sl] == ref.masked_chars).all() and (hout.substr_ids[0][sl] == ref.substr_ids[0]).all())
    h2d, d2h = cfg.last_host_bytes()
    rec = {"api": "b2r_config_new_multi + b2r_match_batch_host, flags = B2R_OUT_SPARSE_D2H | B2R_OUT_SPARSE_REUSE (one process, one host thread per device, ONE ncclAllReduce of the counters)", "devices": world,
           "strings": n, "value": n * STRING_LEN / dt / 1e9, "unit": UNIT, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "parity_vs_single_device": ok}
    del cfg, one
    alloc.free()
    return rec


def latency_leg(ctx, H, cfg, ocfg):
    """The reference's real call shape: ONE <= 1 KiB string per match_substrs (examples/regex.rs:96-112), host buffers."""
    import numpy as np
    from halo2_regex_b200 import _abi
    from halo2_regex_b200._ffi import lib
    s = (b"x" * 500 + b"email was meant for @abcd." + b"y" * 498)[:STRING_LEN]
    data = np.frombuffer(s, dtype=np.uint8).copy()
    hout = H.HostOutputs(1, M, cfg.state_widths, cfg.table_num_rows, cfg.endpoint_num_rows, max_records=8, compact_pitch=64)
    st = hout.struct(0)
    res = _abi.BatchStatus()
    ts = []
    for i in range(320):
        t0 = time.perf_counter()
        rc = lib.b2r_match_substrs(cfg._h, data.ctypes.data, len(data), ctypes.byref(st), ctypes.byref(res))
        ts.append(time.perf_counter() - t0)
        assert rc == 0
    ts = sorted(ts[20:])
    offs = np.array([0, len(data)], dtype=np.uint64)
    oout = ocfg.new_outputs(1, max_records=8, compact_pitch=64)
    cs = []
    for i in range(60):
        t0 = time.perf_counter()
        ocfg.match_batch(data, offs, out=oout, nthreads=1)
        cs.append(time.perf_counter() - t0)
    cs = sorted(cs[10:])
    same = not H.compare_outputs(hout, oout)
    return {"api": "b2r_match_substrs (one 1 KiB string, pageable host buffers, every column + multiplicities)", "p50_us": ts[len(ts) // 2] * 1e6,
            "p99_us": ts[int(len(ts) * 0.99)] * 1e6, "cpu_port_1thread_p50_us": cs[len(cs) // 2] * 1e6, "bit_exact_vs_oracle": same,
            "h2d_d2h_bytes": list(cfg.last_host_bytes())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline config (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-strings", type=int, default=LOG2_STRINGS, help="strings per GPU (default: the BASELINE config)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time plain launches instead of one CUDA graph per step")
    ap.add_argument("--configs", default="2i,2ii,3,4", help="other BASELINE configs reported as sub-records ('' = none)")
    ap.add_argument("--side-steps", type=int, default=5)
    ap.add_argument("--log2-strings-c4", type=int, default=19, help="config 4: strings per GPU (x 4 KiB)")
    ap.add_argument("--log2-long", type=int, default=26, help="config 3: log2 of the string length")
    ap.add_argument("--no-long-oracle", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the single-process multi-device leg and the one-string latency leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the headline config's last step computed "
                    "(a fixed sample of its strings, every multiplicity counter) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm has none")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return reference_arm(args)

    # stdout carries exactly one JSON line: everything else that libraries print there (NCCL's version banner) goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import halo2_regex_b200 as H
    import workloads as W
    ctx = Ctx(args)
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    side = [c for c in args.configs.split(",") if c]

    # ---- headline: config 1, device-resident ------------------------------------------------------------------------------------
    n, L = 1 << args.log2_strings, STRING_LEN
    cfg = make_config(H, SET_REGEX1, M, ctx.local_rank)
    ocfg1 = oracle_from_files(SET_REGEX1, M)
    d_bytes = W.config1_torch(n, L, first=rank * n, device=dev).reshape(-1)      # this rank's slice of the global batch
    head, out, d_offs, clocks = batch_leg(ctx, H, W, "1", workload_config(args.log2_strings)["workload"], cfg, ocfg1, d_bytes, n, L, M, args.steps, args.warmup,
                                          dump_dir=args.dump_outputs if rank == 0 else None)
    del out, d_offs

    # ---- end-to-end arm: C-ABI call with pinned host buffers -----------------------------------------------------------------------
    e2e = e2e_leg(ctx, H, cfg, d_bytes, n, L, args.e2e_steps) if args.e2e_steps > 0 else None
    latency = latency_leg(ctx, H, cfg, ocfg1) if (rank == 0 and not args.no_extras) else None
    del d_bytes
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs ----------------------------------------------------------------------------------------------
    configs = {}
    if "2i" in side or "2ii" in side:
        d2 = W.config2_torch(n, L, first=rank * n, device=dev).reshape(-1)
        for key, spec, what in (("2i", SET_2I, "reading (i): ONE RegexDefs{regex3, [substr1, substr2, substr3]}"),
                                ("2ii", SET_2II, "reading (ii): THREE RegexDefs [regex1+substr1, regex2+substr2, regex3+substr3] (TestCircuit1 layout, src/lib.rs:960-987)")):
            if key not in side:
                continue
            c2 = make_config(H, spec, M, ctx.local_rank)
            rec, o2, _, _ = batch_leg(ctx, H, W, key, f"regex3_test header lines (from: address at the end), 2^{args.log2_strings} x 1 KiB strings per GPU, M=1025, {what} (BASELINE configs[2])",
                                      c2, oracle_from_files(spec, M), d2, n, L, M, args.side_steps, 2, max_records=4, compact_pitch=32)
            configs[key] = rec
            del o2, c2
            torch.cuda.empty_cache()
        del d2
        torch.cuda.empty_cache()
    if "4" in side:
        n4, L4 = 1 << args.log2_strings_c4, 4096
        allstr, substr, info = W.large_dfa_texts()
        c4 = H.RegexVerifyConfig.configure(L4 + 1, [H.RegexDefs(H.AllstrRegexDef.read_from_reader(allstr), [H.SubstrRegexDef.read_from_reader(substr)])], device=ctx.local_rank)
        d4 = W.config4_torch(n4, L4, first=rank * n4, device=dev).reshape(-1)
        rec, o4, _, _ = batch_leg(ctx, H, W, "4", f"synthetic e-mail-header DFA with {info['states']} states (2-byte state column, table beyond the replicated shared-memory tiling), "
                                  f"2^{args.log2_strings_c4} x 4 KiB strings per GPU, M=4097 (BASELINE configs[4]; 2^22 strings over 8 GPUs)",
                                  c4, oracle_from_texts(allstr, substr, L4 + 1), d4, n4, L4, L4 + 1, args.side_steps, 2, max_records=2, compact_pitch=64)
        configs["4"] = rec
        del o4, c4, d4
        torch.cuda.empty_cache()
    if "3" in side and rank == 0:
        configs["3"] = long_leg(ctx, H, W, max(args.side_steps, 5), 3)
        torch.cuda.empty_cache()
    ctx.barrier()

    # ---- one process, every GPU of the box through the C ABI (rank 0; the other ranks idle at the barrier) ---------------------------
    single_process = None
    if world > 1 and not args.no_extras:
        if rank == 0:
            try:
                single_process = multi_device_leg(ctx, H, W)
            except Exception as exc:  # pragma: no cover
                single_process = {"error": repr(exc)}
        ctx.barrier()

    if rank != 0:
        if world > 1:
            ctx.dist.destroy_process_group()
        return

    # ---- CPU baseline: the oracle, single thread (the reference's threading model), bounded sample ----------------------
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        ns = 1 << 16
        data, _ = W.config1_numpy(ns, L)
        offs = np.arange(ns + 1, dtype=np.uint64) * L
        oout = ocfg1.new_outputs(ns, max_records=2, compact_pitch=8)
        ocfg1.match_batch(data.reshape(-1)[: 1024 * L], offs[:1025], out=ocfg1.new_outputs(1024, max_records=2, compact_pitch=8))
        t0 = time.perf_counter()
        ocfg1.match_batch(data.reshape(-1), offs, out=oout, nthreads=1)
        dt = time.perf_counter() - t0
        cpu = {"value": ns * L / dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port", "host_cores_available": os.cpu_count(),
               "sample": f"first 2^16 of the 2^{args.log2_strings} strings (64 MiB), all witness columns + multiplicities, {dt:.1f} s",
               "note": "C restatement of src/lib.rs:311-888 (hash-map walk, scans) without halo2 cell assignment / field inversions: faster than the real reference"}

    # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of the same workload (newest round)
    traffic = None
    try:
        import glob
        for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_walk_kernel_traffic.json"))):
            with open(path) as f:
                tj = json.load(f)
            if tj.get("log2_strings") == args.log2_strings:
                traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    wcfg = workload_config(args.log2_strings)
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": wcfg,
        "run": {"parallelism": (f"strings sharded over {world} GPUs, one rank per GPU; every step accumulates its multiplicities on the device, ONE NCCL all-reduce "
                                "of the counters per job, inside the timed region") if world > 1 else "1 GPU",
                "cuda_graph": head["cuda_graph"]},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": head["kernels_per_step"] * args.steps * world,
        "kernels_per_step": head["kernels_per_step"],
        "step_ms_median": head["step_ms_median"],
        "roofline": {"bound": "hbm", "achieved": head["achieved_gbs"], "peak": ctx.peak, "unit": "GB/s", "frac": head["frac"], "traffic": traffic,
                     "kernel": "walk_kernel<1, u8, bank-replicated tables, shared bins> (DFA walk + fused emit stage: every witness column)",
                     "kernel_ms": head["kernel_ms"], "stage_ms": head["stage_ms"],
                     "table_placement": head["table_placement"], "bin_placement": head["bin_placement"], "algorithmic_bytes_per_launch": head["algorithmic_bytes_per_launch"],
                     "bytes_per_input_byte": head["bytes_per_input_byte"], "peak_source": ctx.peak_src,
                     "frac_of_nominal_8tbs": head["achieved_gbs"] / 8000.0},     # SURVEY 8(d): also against the 8 TB/s spec figure
        "parity": head["parity"],
        "configs": configs,
        "single_process_multi_device": single_process,
        "match_substrs_latency": latency,
        "cpu_baseline": cpu,
    }
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
