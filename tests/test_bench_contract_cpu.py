"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the CPU oracle timed on the
host) must run without CUDA and print ONE JSON line with the driver's keys; the GPU arm must refuse to run
without a device instead of falling back to the oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e,
                          capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--seconds", "20", "--batch", "2", "--cpu-threads", "2"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "input_msamples_per_s_decoded" and d["unit"] == "Msamples/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 2 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    assert "configs[3]" in d["config"]["workload"]            # the GPU arm's default workload, same string


def test_reference_arm_single_recording_is_single_threaded_like_the_reference():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--seconds", "20", "--workload", "c2"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["cpu_baseline"]["cores"] == 1 and "configs[1]" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_without_work():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--seconds", "20",
              "--batch", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "3", "--seconds", "20", "--no-cpu-baseline"])
    assert r.returncode != 0                                  # no CPU fallback for the product path
    assert not any(l.strip().startswith("{") for l in r.stdout.splitlines())


def test_dump_arrays_keeps_every_line_or_one_seeded_sample_within_the_budget():
    import torch
    import bench

    class Dec:
        def __init__(self, k):
            self.k = k

        def last_sync(self):
            return np.arange(self.k, self.k + 40, dtype=np.uint64) * 6240

    outs = [torch.arange(k, k + 300 * bench.LINE, dtype=torch.float32) for k in range(3)]
    produced = [300 * bench.LINE] * 3
    decs = [Dec(k) for k in range(3)]
    full = bench.dump_arrays(decs, outs, produced, world=1)
    assert np.array_equal(full["lines_001"], np.arange(300))
    assert np.array_equal(full["rows_001"], outs[1].numpy().reshape(300, bench.LINE))
    assert np.array_equal(full["sync_002"], decs[2].last_sync().astype(np.float64))
    # a world of 500 ranks leaves this rank room for fewer lines than it decoded: a sample, the same on every call
    part = bench.dump_arrays(decs, outs, produced, world=500)
    again = bench.dump_arrays(decs, outs, produced, world=500)
    assert sum(a.nbytes for a in part.values()) <= bench.DUMP_BYTES // 500
    for k in range(3):
        idx = part[f"lines_{k:03d}"].astype(np.int64)
        assert 0 < idx.size < 300 and np.all(np.diff(idx) > 0)
        assert np.array_equal(idx, again[f"lines_{k:03d}"])
        assert np.array_equal(part[f"rows_{k:03d}"], outs[k].numpy().reshape(300, bench.LINE)[idx])
    assert all(a.dtype in (np.float32, np.float64) for a in part.values())
