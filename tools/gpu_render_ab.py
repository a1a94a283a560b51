"""A/B of the render routes on a device-resident 10-minute 32-channel signal: fused overlap-save kernel
(default) against the cuFFT + multiply-accumulate route (EMAGLS_RENDER_FUSED=0), with the maximum
deviation between the two.  usage (GPU box): python tools/gpu_render_ab.py [seconds]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import emagls_b200 as em  # noqa: E402

secs = float(sys.argv[1]) if len(sys.argv) > 1 else 600.0
n, ch, ln = int(secs * 48000), 32, 512
dev = torch.device("cuda", 0)
h = em.Handle(0)
stream = torch.cuda.ExternalStream(h.stream, device=dev)
x = torch.randn((ch, n), dtype=torch.float64, device=dev)
y = torch.empty((2, n), dtype=torch.float64, device=dev)
rng = np.random.default_rng(0)
wl = torch.from_numpy(rng.standard_normal((ch, ln))).to(dev)
wr = torch.from_numpy(rng.standard_normal((ch, ln))).to(dev)


def run(reps=5):
    def step():
        h.check(h.lib.emagls_binaural_decode_dev(h.ptr, x.data_ptr(), n, ch, wl.data_ptr(), wr.data_ptr(), ln, 0,
                                                 y.data_ptr()))
    step(); step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        step()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


ref = None
ffts = [int(v) for v in os.environ.get("AB_FFTS", "0").split(",")]
for fused, fft in [(f, n_) for n_ in ffts for f in os.environ.get("AB_ROUTES", "0,2").split(",")]:
    os.environ["EMAGLS_RENDER_FUSED"] = fused
    if fft:
        os.environ["EMAGLS_RENDER_FFT"] = str(fft)
    ms = run()
    yy = y.clone()
    dev_ = 0.0 if ref is None else float((yy - ref).abs().max() / ref.abs().max())
    if ref is None:
        ref = yy
    print(f"fft={fft or 'default'} fused={fused}  {ms:8.3f} ms  {n / ms / 1e3:9.1f} Msamples/s  "
          f"{(n * (ch + 2) * 8) / ms / 1e6:7.1f} GB/s algorithmic  max deviation from the cuFFT route {dev_:.1e}", flush=True)
