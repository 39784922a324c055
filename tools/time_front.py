"""Times the resample+envelope kernel alone (decoder profiling events) on a device-resident synthetic recording.
RATE, SECS and ITERS set the input; APTB200_NO_UNIFORM_TAPS=1 times the tiled kernel (k_polyphase_ws) instead of the
uniform-tap one."""
import os, sys, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import noaa_apt_b200 as apt
from noaa_apt_b200 import synth

rate = int(os.environ.get("RATE", "48000"))
secs = float(os.environ.get("SECS", "900"))
x = synth.apt_signal(rate, secs, seed=3).astype(np.float32)
dx = torch.from_numpy(x).cuda()
dec = apt.Decoder(rate, max_samples=x.size)
out = torch.empty(dec.out_bound(x.size), dtype=torch.float32, device="cuda")
dec.set_profiling(True)
times = []
for it in range(int(os.environ.get("ITERS", "12"))):
    dec.submit_device(dx.data_ptr(), 0, x.size, True, out.data_ptr(), out.numel())
    dec.wait()
    t = dict(dec.kernel_times_ms())
    times.append(t.get("resample_envelope", float("nan")))
print("resample_envelope ms: median %.4f  min %.4f  (n=%d)" % (float(np.median(times[2:])), min(times[2:]), len(times) - 2))
