"""The render sessions' algorithm (tests/stream_oracle.py: partitioned overlap-save with a frequency-domain delay line,
per-block page selection, crossfades across call boundaries) equals the whole-signal oracles of the three renders for
random splits of the signal and of the tracker entries, to 1e-12 relative max-norm.  CPU only."""
import os
import sys

import numpy as np
import pytest

import oracle
from oracle.tracked_oracle import binauralDecodeTracked

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sh_tracked_oracle import binauralDecodeShTracked  # noqa: E402
from stream_oracle import StreamOracle  # noqa: E402


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def random_split(rng, nblocks, block):
    """Call lengths (multiples of block) that add up to nblocks blocks: 1, 3 and 7 blocks mixed."""
    sizes = []
    left = nblocks
    while left:
        k = min(left, int(rng.choice([1, 3, 7])))
        sizes.append(k * block)
        left -= k
    return sizes


def random_rotations(rng, nf):
    q = rng.standard_normal((nf, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(nf, 3, 3)


def stream(so, x, entries, sizes, rng, hop):
    """Feed x in calls of `sizes`, appending entries so that each call has what it needs plus a random look-ahead."""
    out, t, given = [], 0, 0
    for n in sizes:
        need = (t + n - 1) // hop + 1
        upto = min(len(entries), need + int(rng.integers(0, 3)))
        new = entries[given:max(upto, given)]
        given += len(new)
        out.append(so.process(x[t:t + n], new))
        t += n
    return np.concatenate(out)


@pytest.mark.parametrize("block,ln,ch", [(64, 512, 8), (48, 100, 4), (32, 33, 3), (64, 1, 2), (128, 128, 2)])
def test_static_stream_equals_the_static_render(block, ln, ch):
    rng = np.random.default_rng(block + ln + ch)
    nb = 20
    x = rng.standard_normal((nb * block, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    so = StreamOracle("static", wL, wR, block)
    y = stream(so, x, [], random_split(rng, nb, block), rng, 1)
    yo = oracle.binauralDecode(x, 1, wL, wR, 1)
    assert rel(y, yo) < 1e-12


@pytest.mark.parametrize("block,hop,fade,kind", [
    (64, 37, 37, "random"), (64, 37, 1, "random"), (64, 37, 0, "random"),
    (48, 48, 48, "random"), (32, 48, 20, "constant"), (64, 300, 300, "random"), (64, 300, 0, "walk"),
])
def test_bank_stream_equals_the_tracked_render(block, hop, fade, kind):
    rng = np.random.default_rng(block * 7 + hop + fade)
    ln, ch, pages, nb = 150, 3, 9, 24
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))
    nf = (n - 1) // hop + 1 + 3
    if kind == "random":
        track = rng.integers(0, pages, nf)
    elif kind == "constant":
        track = np.full(nf, 4)
    else:
        track = np.cumsum(rng.integers(-1, 2, nf)) % pages
    so = StreamOracle("bank", wL, wR, block, hop, fade)
    y = stream(so, x, list(track.astype(np.int32)), random_split(rng, nb, block), rng, hop)
    yo = binauralDecodeTracked(x, wL, wR, track, hop, fade)
    assert rel(y, yo) < 1e-12


@pytest.mark.parametrize("order,block,hop,fade", [(0, 32, 20, 20), (1, 32, 50, 7), (2, 16, 16, 0)])
def test_sh_stream_equals_the_sh_tracked_render(order, block, hop, fade):
    rng = np.random.default_rng(order * 11 + block + hop)
    ch = (order + 1) ** 2
    ln, nb = 40, 12
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    nf = (n - 1) // hop + 1 + 2
    R = random_rotations(rng, nf)
    R[3] = R[2]                               # bitwise-equal frames: exactly Q_c, also across call boundaries
    R[4] = R[3]
    so = StreamOracle("sh", wL, wR, block, hop, fade)
    y = stream(so, x, list(R), random_split(rng, nb, block), rng, hop)
    yo = binauralDecodeShTracked(x, wL, wR, R, hop, fade)
    assert rel(y, yo) < 1e-12
