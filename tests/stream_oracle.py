"""NumPy restatement of the render sessions' algorithm (emagls_render_stream_*, emagls_b200/csrc/stream_render.cu):
uniformly partitioned overlap-save with a frequency-domain delay line, the per-block page selection of the bank render
and the contract's crossfade.  Test infrastructure only: imported by the tests next to it, never by the product
package.  It mirrors the kernels step by step, so that the bookkeeping (FDL slots, partitions, pages of a block, frames
across call boundaries) can be checked against the whole-signal oracles without a GPU."""
from __future__ import annotations

import math

import numpy as np

from oracle import getSHrotMtx

__all__ = ["StreamOracle"]


class StreamOracle:
    """kind 'static' (wL, wR [len, ch]), 'bank' ([len, ch, pages]) or 'sh' ([len, (order+1)^2]); process() takes
    blocks' worth of samples and the next tracker entries, exactly like emagls_render_stream_process."""

    def __init__(self, kind, wL, wR, block, hop=1, fade=0):
        wL, wR = np.asarray(wL, dtype=float), np.asarray(wR, dtype=float)
        if wL.ndim == 2:
            wL, wR = wL[:, :, None], wR[:, :, None]
        self.kind, self.B, self.hop, self.fade = kind, int(block), int(hop), int(fade)
        ln, self.ch, self.pages = wL.shape
        B = self.B
        self.N, self.F, self.P = 2 * B, B + 1, -(-ln // B)
        # H[page][ear][ch][q][F]: partition q = taps [q B, (q + 1) B) zero-padded to N
        wp = np.zeros((self.pages, 2, self.ch, self.P * B))
        wp[:, 0, :, :ln] = wL.transpose(2, 1, 0)
        wp[:, 1, :, :ln] = wR.transpose(2, 1, 0)
        part = np.zeros((self.pages, 2, self.ch, self.P, self.N))
        part[..., :B] = wp.reshape(self.pages, 2, self.ch, self.P, B)
        self.H = np.fft.rfft(part, axis=-1)
        self.X = np.zeros((self.P, self.ch, self.F), dtype=complex)   # FDL ring
        self.prev = np.zeros((self.ch, B))
        self.T = 0
        self.entries = []           # all tracker entries so far (pages, or 3x3 rotations)
        if kind == "sh":
            self.order = math.isqrt(self.ch) - 1

    def _pages(self, t_lo):
        """Distinct pages of the block starting at t_lo (the rule of build_pairs), sorted."""
        hop, fade, trk = self.hop, self.fade, self.entries
        cand = set()
        for f in range(t_lo // hop, (t_lo + self.B - 1) // hop + 1):
            cand.add(int(trk[f]))
            if f > 0 and fade > 0 and f * hop + fade - 1 >= t_lo:
                cand.add(int(trk[f - 1]))
        return sorted(cand)

    def _rotate(self, x, t_lo):
        hop, fade = self.hop, self.fade
        R = np.asarray(self.entries, dtype=float)
        bits = R.reshape(-1, 9).view(np.uint64)
        out = np.empty_like(x)
        Q = {}
        for i in range(self.B):
            t = t_lo + i
            f = t // hop
            ii = t - f * hop
            for fr in (f, max(f - 1, 0)):
                if fr not in Q:
                    Q[fr] = getSHrotMtx(R[fr], self.order, "real")
            blend = f > 0 and ii < fade and not np.array_equal(bits[f], bits[f - 1])
            if blend:
                g = (ii + 0.5) / fade
                out[i] = (1.0 - g) * (x[i] @ Q[f - 1]) + g * (x[i] @ Q[f])
            else:
                out[i] = x[i] @ Q[f]
        return out

    def process(self, x, entries=()):
        x = np.asarray(x, dtype=float)
        n = x.shape[0]
        assert n > 0 and n % self.B == 0
        self.entries.extend(list(entries))
        if self.kind != "static":
            assert len(self.entries) > (self.T + n - 1) // self.hop, "entries do not cover the call"
        B, N, P = self.B, self.N, self.P
        out = np.zeros((n, 2))
        for b in range(n // B):
            t_lo = self.T
            k = t_lo // B
            xb = x[b * B:(b + 1) * B]
            if self.kind == "sh":
                xb = self._rotate(xb, t_lo)
            seg = np.concatenate([self.prev, xb.T], axis=1)               # [ch][N]
            self.prev = xb.T.copy()
            self.X[k % P] = np.fft.rfft(seg, axis=-1)
            pages = self._pages(t_lo) if self.kind == "bank" else [0]
            y = np.zeros((len(pages), 2, N))
            for j, pg in enumerate(pages):
                Y = np.zeros((2, self.F), dtype=complex)
                for q in range(P):
                    Y += np.einsum("cf,ecf->ef", self.X[(k - q) % P], self.H[pg, :, :, q, :])
                y[j] = np.fft.irfft(Y, n=N, axis=-1)
            t = t_lo + np.arange(B)
            if self.kind == "bank":
                trk = np.asarray(self.entries, dtype=np.int64)
                f = t // self.hop
                ii = t - f * self.hop
                c, a = trk[f], trk[np.maximum(f - 1, 0)]
                g = np.where((a != c) & (ii < self.fade), (ii + 0.5) / max(self.fade, 1), 1.0)
            else:
                c = a = np.zeros(B, dtype=np.int64)
                g = np.ones(B)
            for j, pg in enumerate(pages):
                w = np.where(c == pg, g, 0.0) + np.where(a == pg, 1.0 - g, 0.0)
                out[b * B:(b + 1) * B] += w[:, None] * y[j][:, B:].T
            self.T += B
        return out
