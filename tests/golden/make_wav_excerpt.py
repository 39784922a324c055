"""Cuts two excerpts (44 s in total) out of the reference's own test recording, noaa-apt's test/test_11025hz.wav
(11025 Hz, 16-bit mono, 822 s; sha256 50160851becd5997...), and stores the raw PCM16 samples in
tests/golden/test_11025hz_excerpts.npz, so that the one real-world input the reference ships (test/test.sh:45-46)
reaches the CUDA kernels without the reference's source tree.

    [0 s, 24 s)     the recording starts in noise: sync spacings from 1122 to 13454 work samples, the seed peak is
                    refined, several frames are skipped (decode.rs:241-253)
    [230 s, 250 s)  a noisy stretch in which the `while` at decode.rs:244 pushes the same position twice
                    (duplicate sync position -> duplicate image row) and the largest gap of the file (18708)

The file holds reference-owned DATA (a fixture), no reference code.  The sync positions the CPU oracle finds are
stored next to the samples as a drift guard; the GPU tests recompute them with the oracle on the box.

It also decodes the whole recording with the CPU oracle and stores in tests/golden/test_11025hz_full_decode.npz what
tests/test_oracle_reference_wav.py compares the excerpts' decodes with: every sync position of the recording, the
extremes of its stages and, for the image lines of the full decode that each excerpt's decode reproduces, a fixed
seeded sample of 208 of their 2080 values plus each line's min, max and float64 sum.

    python tests/golden/make_wav_excerpt.py <noaa-apt checkout>/test/test_11025hz.wav
"""
import hashlib
import os
import sys
import wave

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
EXCERPTS = {"start": (0, 24), "dup": (230, 250)}
RATE, WORK_RATE, PX = 11025, 12480, 2080


def line_stats(rows):
    return np.stack([rows.min(axis=1), rows.max(axis=1), rows.sum(axis=1, dtype=np.float64)], axis=1).astype(np.float64)


def main(wav):
    import oracle
    with open(wav, "rb") as f:
        digest = hashlib.sha256(f.read()).hexdigest()
    with wave.open(wav) as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate()) == (1, 2, RATE)
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
    full, fst = oracle.decode_steps(oracle.pcm16_to_f32(pcm), RATE)
    full_rows = full.reshape(-1, PX)
    full_sync = fst["sync_pos"].astype(np.int64)
    cols = np.sort(np.random.default_rng(0).choice(PX, PX // 10, replace=False))
    out = {"rate": np.int64(RATE), "sha256": np.array(digest)}
    gold = {"sha256": np.array(digest), "samples": np.int64(pcm.size), "resampled_size": np.int64(fst["resampled"].size),
            "lines": np.int64(full_rows.shape[0]), "sync_pos": full_sync, "cols": cols.astype(np.int64),
            "extremes": np.array([fst["resampled"].min(), fst["resampled"].max(), fst["demodulated"].max(), full.min(),
                                  full.max(), full.mean(dtype=np.float64)], dtype=np.float64)}
    for name, (t0, t1) in EXCERPTS.items():
        cut = pcm[t0 * RATE: t1 * RATE].copy()
        rows, st = oracle.decode_steps(oracle.pcm16_to_f32(cut), RATE)
        rows = rows.reshape(-1, PX)
        pos = st["sync_pos"].astype(np.int64) + t0 * WORK_RATE        # t0 * RATE samples in = t0 * WORK_RATE out
        out[f"pcm_{name}"] = cut
        out[f"sync_{name}"] = st["sync_pos"]
        # the excerpt's decode locks onto the full decode's sync positions after its first few frames and keeps them
        # (with bit-identical image lines) to its last complete line
        i0 = next(i for i in range(len(pos)) if pos[i] in full_sync)
        j0 = int(np.nonzero(full_sync == pos[i0])[0][0])
        count = rows.shape[0] - i0
        assert np.array_equal(pos[i0: i0 + count], full_sync[j0: j0 + count])
        assert np.array_equal(rows[i0:], full_rows[j0: j0 + count])
        gold[f"first_{name}"] = np.array([i0, j0, count], dtype=np.int64)
        gold[f"rows_{name}"] = full_rows[j0: j0 + count][:, cols]
        gold[f"stats_{name}"] = line_stats(full_rows[j0: j0 + count])
        print(name, cut.size, "samples,", pos.size, "sync positions, min spacing", int(np.diff(pos).min()),
              f"max spacing {int(np.diff(pos).max())}; lines {j0}..{j0 + count} of the full decode from excerpt line {i0}")
    np.savez_compressed(os.path.join(HERE, "test_11025hz_excerpts.npz"), **out)
    np.savez_compressed(os.path.join(HERE, "test_11025hz_full_decode.npz"), **gold)


if __name__ == "__main__":
    main(sys.argv[1])
