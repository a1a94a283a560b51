"""The head-tracked render oracle (oracle/tracked_oracle.py) against its own definition: a constant track is the
static render, the crossfade weights of the two pages sum to one and change linearly, a hard switch is the two static
renders on either side of the frame boundary."""
import numpy as np

import oracle
from oracle.tracked_oracle import binauralDecodeTracked


def _bank(rng, ln, ch, pages):
    return rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))


def test_constant_track_is_the_static_render():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((3001, 4))
    wL, wR = _bank(rng, 64, 4, 3)
    for comp in (False, True):
        y = binauralDecodeTracked(x, wL, wR, np.full(8, 2), 400, 400, comp)
        yo = oracle.binauralDecode(x, 1, wL[:, :, 2], wR[:, :, 2], 1, comp)
        assert y.shape == yo.shape and np.array_equal(y, yo)


def test_full_fade_weights_sum_to_one_and_are_linear():
    """With the same filter on every channel of page p scaled by s_p, the render of a signal is s_p times one static
    render, so the tracked output divided by that render is the weighted sum of the scales."""
    rng = np.random.default_rng(2)
    hop, n = 50, 400
    x = rng.standard_normal((n, 1))
    w = rng.standard_normal((16, 1, 1))
    scales = np.array([1.0, 3.0])
    wL = w * scales[None, None, :]
    track = np.array([0, 1, 0, 1, 1, 0, 1, 0])
    y = binauralDecodeTracked(x, wL, wL, track, hop)
    base = oracle.binauralDecode(x, 1, w[:, :, 0], w[:, :, 0], 1)
    mix = y[:, 0] / base[:, 0]                         # = (1 - g) s_a + g s_c
    t = np.arange(n)
    f, i = t // hop, t % hop
    c, a = track[f], track[np.maximum(f - 1, 0)]
    g = np.where(a == c, 1.0, (i + 0.5) / hop)
    assert np.allclose(mix, (1 - g) * scales[a] + g * scales[c], rtol=1e-9, atol=1e-9)
    # the weights of the two pages sum to one: two pages with the same filter render exactly that filter
    y1 = binauralDecodeTracked(x, np.concatenate([w, w], 2), np.concatenate([w, w], 2), track, hop)
    assert np.allclose(y1, base, rtol=0, atol=1e-12 * np.abs(base).max())
    # and g rises by 1/hop per sample inside a switching frame
    sw = (f == 1)
    assert np.allclose(np.diff(g[sw]), 1.0 / hop)


def test_hard_switch_reproduces_the_static_renders():
    rng = np.random.default_rng(3)
    hop = 300
    x = rng.standard_normal((1200, 3))
    wL, wR = _bank(rng, 32, 3, 4)
    track = np.array([3, 1, 1, 0])
    y = binauralDecodeTracked(x, wL, wR, track, hop, 0)
    for f, p in enumerate(track):
        yo = oracle.binauralDecode(x, 1, wL[:, :, p], wR[:, :, p], 1)
        assert np.array_equal(y[f * hop:(f + 1) * hop], yo[f * hop:(f + 1) * hop])
