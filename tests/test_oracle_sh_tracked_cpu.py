"""The SH head-tracked render reference (tests/sh_tracked_oracle.py) against its own definition and the two
identities that pin its orientation convention: a constant track R equals the static render with the LS filters
designed on the HRIR grid rotated by R, and horRotAngleRad = a equals the constant track of a yaw of -a."""
import math
import os
import sys

import numpy as np

import oracle
from emagls_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sh_tracked_oracle import binauralDecodeShTracked  # noqa: E402


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def rot_xyz(yaw_deg, pitch_deg, roll_rad):
    """Rz(yaw) Ry(pitch) Rx(roll)."""
    c, s = math.cos(roll_rad), math.sin(roll_rad)
    return synth.rotation_yaw_pitch(yaw_deg, pitch_deg) @ np.array([[1, 0, 0], [0, c, -s], [0, s, c]])


def random_rotations(rng, nf):
    q = rng.standard_normal((nf, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(nf, 3, 3)


def test_constant_track_is_the_rotated_static_render():
    rng = np.random.default_rng(1)
    order, n, hop = 3, 2000, 150
    x = rng.standard_normal((n, 16))
    wL, wR = rng.standard_normal((64, 16)), rng.standard_normal((64, 16))
    R = rot_xyz(37.0, -20.0, 0.3)
    nf = (n - 1) // hop + 1
    for comp in (False, True):
        y = binauralDecodeShTracked(x, wL, wR, np.repeat(R[None], nf, 0), hop, hop, comp)
        yo = oracle.binauralDecode(x @ oracle.getSHrotMtx(R, order, "real"), 1, wL, wR, 1, comp)
        assert y.shape == yo.shape and rel(y, yo) < 1e-13


def test_ls_filters_on_the_rotated_grid_are_the_constant_track():
    order = 3
    az, ze = synth.fibonacci_sphere(200)
    hL, hR = synth.synth_hrirs(az, ze, taps=64, delay=16)
    R = rot_xyz(37.0, -20.0, 0.3)
    w0L, w0R = oracle.getLsFilters(hL, hR, az, ze, order)
    raz, rze = synth.rotate_grid(az, ze, R)
    wrL, wrR = oracle.getLsFilters(hL, hR, raz, rze, order)
    Q = oracle.getSHrotMtx(R, order, "real")
    assert rel(wrL, w0L @ Q.T) < 1e-12 and rel(wrR, w0R @ Q.T) < 1e-12
    x = np.random.default_rng(2).standard_normal((1500, 16))
    y = binauralDecodeShTracked(x, w0L, w0R, np.repeat(R[None], 4, 0), 480)
    ys = oracle.binauralDecode(x, 1, wrL, wrR, 1)
    assert rel(y, ys) < 1e-12


def test_horizontal_rotation_angle_is_a_constant_yaw_track():
    x = np.random.default_rng(3).standard_normal((1200, 25))
    rng = np.random.default_rng(4)
    wL, wR = rng.standard_normal((32, 25)), rng.standard_normal((32, 25))
    for a in (0.7, -2.1):
        R = synth.rotation_yaw_pitch(-math.degrees(a), 0.0)
        y = binauralDecodeShTracked(x, wL, wR, np.repeat(R[None], 3, 0), 500)
        yo = oracle.binauralDecode(x, 1, wL, wR, 1, horRotAngleRad=a)
        assert rel(y, yo) < 1e-13


def test_bitwise_equal_frames_do_not_blend():
    rng = np.random.default_rng(5)
    hop, n = 100, 800
    x = rng.standard_normal((n, 9))
    wL, wR = rng.standard_normal((16, 9)), rng.standard_normal((16, 9))
    R = random_rotations(rng, 1)[0]
    track = np.stack([R.copy() for _ in range(8)])
    assert np.array_equal(binauralDecodeShTracked(x, wL, wR, track, hop, hop),
                          binauralDecodeShTracked(x, wL, wR, track, hop, 0))
    # one ulp apart: the frames blend
    track[3, 0, 0] = np.nextafter(track[3, 0, 0], 2.0)
    assert not np.array_equal(binauralDecodeShTracked(x, wL, wR, track, hop, hop),
                              binauralDecodeShTracked(x, wL, wR, track, hop, 0))


def test_pieces_with_a_halo_compose_into_the_whole_render():
    rng = np.random.default_rng(6)
    hop, n, ln = 70, 1500, 48
    x = rng.standard_normal((n, 4))
    wL, wR = rng.standard_normal((ln, 4)), rng.standard_normal((ln, 4))
    track = random_rotations(rng, (n - 1) // hop + 1)
    whole = binauralDecodeShTracked(x, wL, wR, track, hop, 30)
    cut = 811
    first = binauralDecodeShTracked(x[:cut], wL, wR, track, hop, 30)
    lo = cut - (ln - 1)
    second = binauralDecodeShTracked(x[lo:], wL, wR, track, hop, 30, firstSample=lo)[ln - 1:]
    assert rel(np.concatenate([first, second]), whole) < 1e-13
