"""bench.py --dump-outputs on the device: what it writes is what the timed path decoded from the seeded recordings."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from noaa_apt_b200 import synth
import oracle
from _parity import rows_without, sync_ties

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_steps_lines_and_sync_positions(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--seconds", "20",
                        "--batch", "3", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    files = sorted(os.listdir(out))
    assert files == sorted(f"{kind}_{k:03d}.npy" for kind in ("lines", "rows", "sync") for k in range(3))
    assert sum(os.path.getsize(out / f) for f in files) <= 64_000_000
    for k in range(3):                                 # decoder k decoded recording seed k (bench --seed-base 0)
        x = synth.apt_pcm16(48000, 20.0, seed=k).astype(np.float32)
        ref, st = oracle.decode_steps(x, 48000)
        rows, lines, sync = (np.load(out / f"{kind}_{k:03d}.npy") for kind in ("rows", "lines", "sync"))
        assert rows.dtype == np.float32 and lines.dtype == sync.dtype == np.float64
        ties = sync_ties(sync.astype(np.uint64), st["sync_pos"], st["filtered"], 12480)
        assert np.array_equal(lines, np.arange(ref.size // 2080))
        got, want = rows_without(rows.ravel(), ties).astype(np.float64), rows_without(ref, ties)
        assert float(np.max(np.abs(got - want))) / float(np.max(np.abs(want))) <= 1e-5
