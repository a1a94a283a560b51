"""Per-repetition timings of one render route on a device-resident signal (variance check).
usage (GPU box): [EMAGLS_RENDER_FUSED=0] python tools/gpu_render_reps.py [seconds] [reps]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import emagls_b200 as em  # noqa: E402

secs = float(sys.argv[1]) if len(sys.argv) > 1 else 600.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 12
n, ch, ln = int(secs * 48000), 32, 512
dev = torch.device("cuda", 0)
h = em.Handle(0)
stream = torch.cuda.ExternalStream(h.stream, device=dev)
x = torch.randn((ch, n), dtype=torch.float64, device=dev)
y = torch.empty((2, n), dtype=torch.float64, device=dev)
rng = np.random.default_rng(0)
wl = torch.from_numpy(rng.standard_normal((ch, ln))).to(dev)
wr = torch.from_numpy(rng.standard_normal((ch, ln))).to(dev)
times = []
for i in range(reps + 2):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    h.check(h.lib.emagls_binaural_decode_dev(h.ptr, x.data_ptr(), n, ch, wl.data_ptr(), wr.data_ptr(), ln, 0, y.data_ptr()))
    b.record(stream)
    torch.cuda.synchronize()
    if i >= 2:
        times.append(a.elapsed_time(b))
print(f"route {os.environ.get('EMAGLS_RENDER_FUSED', 'default')} secs {secs:.0f} x ptr % 2MiB = {x.data_ptr() % (1 << 21)}: "
      + " ".join(f"{t:.2f}" for t in times) + f"  | median {np.median(times):.2f} ms")
