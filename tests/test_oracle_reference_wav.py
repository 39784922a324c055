"""Config 1 of BASELINE.json: decode the reference's own test recording on the
CPU (plumbing run).  The reference cannot be executed (no Rust toolchain), so
this checks the oracle against the independent numpy-f32 cross-check numbers
recorded in SURVEY.md Appendix C.  The recording itself (18 MB) is not stored:
tests/golden/make_wav_excerpt.py decoded it whole with the oracle and kept its
sync positions and a sample of the image lines that its two stored excerpts
(tests/golden/test_11025hz_excerpts.npz) cover.  The test decodes those excerpts
and requires the full decode's positions and lines back.
"""
import os

import numpy as np
import pytest

import oracle

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
EXCERPT_START_S = {"start": 0, "dup": 230}
WORK_RATE = 12480


@pytest.fixture(scope="module")
def golden():
    return (np.load(os.path.join(GOLDEN, "test_11025hz_excerpts.npz")),
            np.load(os.path.join(GOLDEN, "test_11025hz_full_decode.npz")))


def test_decode_reference_recording_matches_survey_numbers(golden):
    excerpts, full = golden
    assert str(excerpts["sha256"]) == str(full["sha256"])                 # both cut from the same recording
    # the whole recording's decode, as SURVEY.md Appendix C records it
    assert int(full["samples"]) == 9_067_017
    assert int(full["resampled_size"]) == 10_263_607
    sync = full["sync_pos"]
    assert sync.size == 1644
    assert sync[:4].tolist() == [3989, 13153, 19644, 26047]
    d = np.diff(sync)
    assert (np.median(d), d.min(), d.max()) == (6240, 0, 18708)
    assert int(full["lines"]) == 1642
    r_min, r_max, d_max, o_min, o_max, o_mean = full["extremes"].tolist()
    assert abs(r_min - (-26.86)) < 0.01 and abs(r_max - 32.86) < 0.01 and abs(d_max - 67.60) < 0.01
    assert abs(o_min - (-3.02)) < 0.01 and abs(o_max - 44.78) < 0.01 and abs(o_mean - 9.38) < 0.01
    # the oracle on the stored excerpts finds the same sync positions and the same image lines
    cols = full["cols"]
    for name, t0 in EXCERPT_START_S.items():
        rows, st = oracle.decode_steps(oracle.pcm16_to_f32(excerpts[f"pcm_{name}"]), 11025)
        rows = rows.reshape(-1, 2080)
        pos = st["sync_pos"].astype(np.int64) + t0 * WORK_RATE
        i0, j0, count = full[f"first_{name}"].tolist()
        assert count >= 30 and rows.shape[0] == i0 + count, name
        assert np.array_equal(pos[i0: i0 + count], sync[j0: j0 + count]), name
        mine = rows[i0:]
        assert np.array_equal(mine[:, cols], full[f"rows_{name}"]), name
        stats = full[f"stats_{name}"]
        assert np.array_equal(mine.min(axis=1), stats[:, 0]) and np.array_equal(mine.max(axis=1), stats[:, 1]), name
        assert np.allclose(mine.sum(axis=1, dtype=np.float64), stats[:, 2], rtol=1e-12, atol=0), name
        if name == "dup":                       # the duplicate position and the largest gap of the recording
            assert np.diff(pos).min() == 0 and np.diff(pos).max() == 18708
