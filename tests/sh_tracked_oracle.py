"""FP64 reference of the head-tracked render of SH signals (the contract of emagls_binaural_decode_sh_tracked,
include/emagls_cuda.h), written straight from its definition with the oracle's getSHrotMtx and binauralDecode.
Test infrastructure only: imported by the tests next to it, never by the product package."""
from __future__ import annotations

import math

import numpy as np

from oracle import binauralDecode, getSHrotMtx

__all__ = ["binauralDecodeShTracked", "frame_times"]


def frame_times(n, hop, fade, firstSample=0):
    """Per input sample n: (c, a, g) of the contract, t = firstSample + n, f = t // hop, i = t - f hop, c = f,
    a = max(f - 1, 0), g = (i + 0.5) / fade for i < fade else 1."""
    t = int(firstSample) + np.arange(n)
    f = t // hop
    i = t - f * hop
    g = np.where(i < fade, (i + 0.5) / max(fade, 1), 1.0)
    return f, np.maximum(f - 1, 0), g


def binauralDecodeShTracked(inp, wL, wR, rotations, hop, fade=None, compensateDelay=False, firstSample=0):
    """x'[n] = inp[n, :] @ M(n) with M(n) = (1 - g) Q_a + g Q_c, Q_f = getSHrotMtx(rotations[f], order, 'real'),
    M(n) = Q_c exactly when rotations[a] and rotations[c] are bitwise equal; then the static binauralDecode of x'."""
    x = np.asarray(inp, dtype=float)
    n, ch = x.shape
    order = math.isqrt(ch) - 1
    assert (order + 1) ** 2 == ch
    R = np.ascontiguousarray(np.asarray(rotations, dtype=float).reshape(-1, 3, 3))
    hop = int(hop)
    fade = hop if fade is None else int(fade)
    c, a, g = frame_times(n, hop, fade, firstSample)
    Q = {f: getSHrotMtx(R[f], order, "real") for f in np.unique(np.concatenate([c, a]))}
    bits = R.view(np.uint64).reshape(R.shape[0], 9)
    xr = np.empty_like(x)
    for k in range(n):
        if np.array_equal(bits[a[k]], bits[c[k]]):
            M = Q[c[k]]
        else:
            M = (1.0 - g[k]) * Q[a[k]] + g[k] * Q[c[k]]
        xr[k] = x[k] @ M
    return binauralDecode(xr, 1, np.asarray(wL), np.asarray(wR), 1, compensateDelay)
