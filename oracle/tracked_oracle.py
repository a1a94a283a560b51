"""Head-tracked render oracle (TEST INFRASTRUCTURE ONLY): the contract of emagls_binaural_decode_tracked
(include/emagls_cuda.h) in FP64 NumPy, built from the static binauralDecode restatement."""
from __future__ import annotations

import numpy as np

from .emagls_oracle import binauralDecode

__all__ = ["binauralDecodeTracked"]


def binauralDecodeTracked(inp, wL, wR, track, hop, fade=None, compensateDelay=False, firstSample=0):
    """Head-tracked binauralDecode (the contract of emagls_binaural_decode_tracked, include/emagls_cuda.h), straight
    from its definition: one static render y_p per referenced page p of the bank [len, ch, pages], mixed per sample as
    out[n] = (1 - g) y_a[n] + g y_c[n] with t = firstSample + n, f = t // hop, i = t - f hop, c = track[f],
    a = track[max(f - 1, 0)], g = (i + 0.5) / fade for i < fade else 1 (and exactly y_c where a == c)."""
    x = np.asarray(inp)
    wL, wR = np.asarray(wL), np.asarray(wR)
    if wL.ndim == 2:
        wL, wR = wL[:, :, None], wR[:, :, None]
    track = np.asarray(track).astype(np.int64)
    hop = int(hop)
    fade = hop if fade is None else int(fade)
    n = x.shape[0]
    t = int(firstSample) + np.arange(n)
    f = t // hop
    i = t - f * hop
    c = track[f]
    a = track[np.maximum(f - 1, 0)]
    g = np.where(i < fade, (i + 0.5) / max(fade, 1), 1.0)
    g = np.where(a == c, 1.0, g)
    out = np.zeros((n, 2))
    for p in np.unique(np.concatenate([c, a[g < 1.0]])):
        wgt = np.where(c == p, g, 0.0) + np.where(a == p, 1.0 - g, 0.0)
        y = binauralDecode(x, 1, wL[:, :, p], wR[:, :, p], 1)
        out += wgt[:, None] * y
    if compensateDelay:
        out = out[wL.shape[0] // 2 - 1:, :]
    return out
