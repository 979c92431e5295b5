"""CPU: the reference arm of bench.py (`--impl reference`) prints one JSON line with the contract's keys and never loads libb2r.so;
GPU: `--dump-outputs` writes what the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "input bytes/sec (DFA witness gen)" and line["unit"] == "GB/s"
    assert line["higher_is_better"] is True and line["steps"] == 1 and line["warmup"] == 1 and line["value"] > 0
    assert line["config"]["strings_per_gpu"] == 1 << 20 and line["config"]["max_chars_size"] == 1025          # the GPU arm's config object
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_steps_and_dump_outputs_are_checked():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, cwd=ROOT, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error:" in out.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_oracle_computes(tmp_path):
    """--dump-outputs: float32 / float64 arrays of the last timed step, small, and equal to the oracle on the sampled strings."""
    import numpy as np
    import workloads as W
    from conftest import oracle_config
    log2n, L = 11, 1024
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--log2-strings", str(log2n), "--configs", "", "--no-extras",
                          "--e2e-steps", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    idx = d["string_index"].astype(np.int64)
    assert len(idx) == 1024 and (np.diff(idx) > 0).all() and idx[-1] < 1 << log2n
    data, _ = W.config1_numpy(1 << log2n, L)
    o, _ = oracle_config("regex1", L + 1).match_batch(data.reshape(-1), np.arange((1 << log2n) + 1, dtype=np.uint64) * L, max_records=2, compact_pitch=8)
    want = o.defined()
    for k in ("states0", "substr_ids0", "start_enable0", "end_enable0", "masked_chars", "masked_substr_ids"):
        assert np.array_equal(d[k], want[k][idx]), k
    for k in ("mult0", "endpoint_mult0"):
        assert np.array_equal(d[k], want[k].astype(np.float64)), k
    for f in ("flags", "n_records", "n_compact"):
        assert np.array_equal(d["status_" + f], o.status[f][idx]), f


def test_reference_arm_does_not_load_the_cuda_library():
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0']\n"
            "runpy.run_path('bench.py', run_name='__main__')\n"
            "import os\n"
            "maps = open('/proc/self/maps').read()\n"
            "assert 'libb2r.so' not in maps, 'the reference arm mapped libb2r.so'\n"
            "assert 'halo2_regex_b200' not in sys.modules\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
