"""Head-tracked render of SH signals (emagls_binaural_decode_sh_tracked) against tests/sh_tracked_oracle.py and the
existing static paths, B200 only.  Tolerance: 1e-9 relative max-norm against the oracle, the bar of
test_gpu_render.py."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sh_tracked_oracle import binauralDecodeShTracked  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def h(em):
    return em.Handle(0)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def frames_needed(n, hop, first=0):
    return (first + n - 1) // hop + 1


def random_rotations(rng, nf):
    q = rng.standard_normal((nf, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(nf, 3, 3)


def filters(rng, ln, ch):
    return rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))


@pytest.mark.parametrize("n,order,ln,hop,fade,comp", [
    (20000, 1, 512, 37, 37, False),       # hop shorter than the filter and than a warp's sample span
    (20000, 4, 512, 37, 0, True),         # hard switch
    (30001, 4, 256, 441, 1, False),       # odd hop, one-sample fade, odd length (cuFFT route)
    (30000, 7, 256, 441, 200, True),      # partial fade
    (40000, 4, 512, 9000, 9000, False),   # frames longer than a render block
    (40000, 0, 512, 9000, 0, True),
    (300, 4, 128, 1000, 500, False),      # signal shorter than one frame
    (12000, 7, 512, 480, 480, False),
])
def test_sh_tracked_render_matches_oracle(em, h, n, order, ln, hop, fade, comp):
    rng = np.random.default_rng(n + hop + fade + order)
    ch = (order + 1) ** 2
    x = rng.standard_normal((n, ch))
    wL, wR = filters(rng, ln, ch)
    R = random_rotations(rng, frames_needed(n, hop))          # exactly as long as needed, a large step every frame
    y = em.binauralDecodeShTracked(x, wL, wR, R, hop, fade, comp, handle=h)
    yo = binauralDecodeShTracked(x, wL, wR, R, hop, fade, comp)
    assert y.shape == yo.shape
    assert rel(y, yo) < 1e-9


def test_constant_track_is_rotate_sh_and_the_static_render(em, h):
    rng = np.random.default_rng(4)
    order, n, hop = 4, 50000, 480
    x = rng.standard_normal((n, 25))
    wL, wR = filters(rng, 512, 25)
    yaw, pitch, roll = 0.7, -0.3, 0.2
    R = oracle.euler2rotationMatrix(-yaw, -pitch, roll, "zyx").T
    track = np.repeat(R[None], frames_needed(n, hop), 0)
    for comp in (False, True):
        y = em.binauralDecodeShTracked(x, wL, wR, track, hop, None, comp, handle=h)
        ys = em.binauralDecode(em.rotateSH(x, yaw, pitch, roll, handle=h), 48000, wL, wR, 48000, comp, handle=h)
        assert y.shape == ys.shape and rel(y, ys) < 1e-12
    a = -1.3
    from emagls_b200 import synth
    Ry = synth.rotation_yaw_pitch(-math.degrees(a), 0.0)
    y = em.binauralDecodeShTracked(x, wL, wR, np.repeat(Ry[None], frames_needed(n, hop), 0), hop, handle=h)
    ys = em.binauralDecode(x, 48000, wL, wR, 48000, horRotAngleRad=a, handle=h)
    assert rel(y, ys) < 1e-12


def test_ls_filters_on_the_rotated_grid(em, h):
    from emagls_b200 import synth
    order = 3
    az, ze = synth.fibonacci_sphere(200)
    hL, hR = synth.synth_hrirs(az, ze, taps=256, delay=40)
    R = synth.rotation_yaw_pitch(37.0, -20.0) @ np.array([[1, 0, 0], [0, math.cos(0.3), -math.sin(0.3)],
                                                         [0, math.sin(0.3), math.cos(0.3)]])
    w0L, w0R = em.getLsFilters(hL, hR, az, ze, order, handle=h)
    raz, rze = synth.rotate_grid(az, ze, R)
    wrL, wrR = em.getLsFilters(hL, hR, raz, rze, order, handle=h)
    x = np.random.default_rng(5).standard_normal((24000, 16))
    y = em.binauralDecodeShTracked(x, w0L, w0R, np.repeat(R[None], frames_needed(24000, 480), 0), 480, handle=h)
    ys = em.binauralDecode(x, 48000, wrL, wrR, 48000, handle=h)
    assert rel(y, ys) < 1e-10


def test_chunked_workspace_gives_the_same_output(em, h, monkeypatch):
    rng = np.random.default_rng(6)
    n, order, hop, ln = 60000, 4, 441, 512
    x = rng.standard_normal((n, 25))
    wL, wR = filters(rng, ln, 25)
    R = random_rotations(rng, frames_needed(n, hop))
    for comp in (False, True):
        l0 = h.launches
        whole = em.binauralDecodeShTracked(x, wL, wR, R, hop, 300, comp, handle=h)
        one_call = h.launches - l0
        monkeypatch.setenv("EMAGLS_TRACK_WS_MB", "1")     # 1 MB: about 5000 samples of 25 channels per chunk
        l0 = h.launches
        chunked = em.binauralDecodeShTracked(x, wL, wR, R, hop, 300, comp, handle=h)
        many = h.launches - l0
        monkeypatch.delenv("EMAGLS_TRACK_WS_MB")
        # every chunk launches the frame matrices, the rotation and a static render
        assert many >= 5 * one_call
        assert chunked.shape == whole.shape and rel(chunked, whole) < 1e-12


def test_dev_variant_equals_host_variant(em, h):
    import torch
    rng = np.random.default_rng(7)
    n, order, ln, hop, fade = 30000, 4, 512, 480, 200
    ch = (order + 1) ** 2
    x = rng.standard_normal((n, ch))
    wL, wR = filters(rng, ln, ch)
    R = random_rotations(rng, frames_needed(n, hop) + 3)
    y = em.binauralDecodeShTracked(x, wL, wR, R, hop, fade, True, handle=h)
    dev = torch.device("cuda", 0)
    xd = torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)                 # [n, ch] column-major
    wd = [torch.from_numpy(np.ascontiguousarray(w.T)).to(dev) for w in (wL, wR)]
    rd = torch.from_numpy(np.ascontiguousarray(R.reshape(-1, 9))).to(dev)
    rows = n - ln // 2 + 1
    out = torch.empty((2, rows), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    h.check(h.lib.emagls_binaural_decode_sh_tracked_dev(h.ptr, xd.data_ptr(), n, order, wd[0].data_ptr(),
                                                        wd[1].data_ptr(), ln, rd.data_ptr(), R.shape[0], hop, fade, 0,
                                                        1, out.data_ptr()))
    torch.cuda.ExternalStream(h.stream, device=dev).synchronize()
    assert np.array_equal(out.cpu().numpy().T, y)


def test_consecutive_pieces_compose(em, h):
    rng = np.random.default_rng(8)
    n, m, ln, hop = 40000, 17001, 512, 480
    x = rng.standard_normal((n, 16))
    wL, wR = filters(rng, ln, 16)
    R = random_rotations(rng, frames_needed(n, hop))
    whole = em.binauralDecodeShTracked(x, wL, wR, R, hop, handle=h)
    first = em.binauralDecodeShTracked(x[:m], wL, wR, R, hop, handle=h)
    halo = ln - 1
    second = em.binauralDecodeShTracked(x[m - halo:], wL, wR, R, hop, firstSample=m - halo, handle=h)[halo:]
    assert rel(np.concatenate([first, second], 0), whole) < 1e-12


def test_time_block_sharded_sh_tracked_render(em, h):
    from emagls_b200 import dist as emdist
    rng = np.random.default_rng(9)
    n, taps, ch, hop = 50000, 512, 25, 480
    x = rng.standard_normal((n, ch))
    wL, wR = filters(rng, taps, ch)
    R = random_rotations(rng, frames_needed(n, hop))
    ref = em.binauralDecodeShTracked(x, wL, wR, R, hop, handle=h)
    # world size 1 through for_signal, then the shards of a world of 3 reassembled
    sr = emdist.ShardedRenderer.for_signal(h, x, wL, wR, rotations=R, hop=hop)
    sr.step()
    assert rel(sr.wait(), ref) < 1e-12
    parts = []
    for r in range(3):
        lo, hi, halo = emdist.render_shard(n, taps, r, 3)
        sr = emdist.ShardedRenderer(h, x[lo - halo:hi], wL, wR, halo, rotations=R, hop=hop, first_sample=lo - halo)
        sr.step()
        parts.append(sr.wait().copy())
    got = np.concatenate(parts, 0)
    assert got.shape == ref.shape and rel(got, ref) < 1e-12
    with pytest.raises(ValueError):
        emdist.ShardedRenderer(h, x, wL, wR, 0, rotations=R, track=np.zeros(R.shape[0], np.int32), hop=hop)


def test_rejected_arguments_launch_nothing(em, h):
    rng = np.random.default_rng(10)
    n, order, ln, hop = 2000, 2, 64, 100
    ch = (order + 1) ** 2
    x = np.asfortranarray(rng.standard_normal((n, ch)))
    wL, wR = (np.asfortranarray(w) for w in filters(rng, ln, ch))
    R = np.ascontiguousarray(random_rotations(rng, frames_needed(n, hop)).reshape(-1, 9))
    out = np.zeros((n, 2))
    P = [a.ctypes.data_as(C.c_void_p) for a in (x, wL, wR, R, out)]
    base = dict(n=n, order=order, ln=ln, nf=R.shape[0], hop=hop, fade=hop, first=0, comp=0)

    def call(p=P, **kw):
        a = dict(base, **kw)
        return h.lib.emagls_binaural_decode_sh_tracked(h.ptr, p[0], a["n"], a["order"], p[1], p[2], a["ln"], p[3],
                                                       a["nf"], a["hop"], a["fade"], a["first"], a["comp"], p[4])
    cases = [dict(order=-1), dict(order=8), dict(hop=0), dict(fade=-1), dict(fade=hop + 1), dict(first=-1),
             dict(nf=R.shape[0] - 1), dict(ln=ln - 1, comp=1), dict(n=ln // 2 - 1, comp=1)]
    for c in cases:
        l0 = h.launches
        assert call(**c) == -1 and h.launches == l0, c
    for k in range(5):
        p = list(P)
        p[k] = None
        l0 = h.launches
        assert call(p) == -1 and h.launches == l0, k
        assert h.lib.emagls_binaural_decode_sh_tracked_dev(h.ptr, *([p[0], n, order, p[1], p[2], ln, p[3], R.shape[0],
                                                                      hop, hop, 0, 0, p[4]])) == -1
        assert h.launches == l0
    with pytest.raises(ValueError):
        em.binauralDecodeShTracked(rng.standard_normal((100, 5)), np.ones((8, 5)), np.ones((8, 5)), R.reshape(-1, 3, 3),
                                   hop, handle=h)
    with pytest.raises(NotImplementedError):
        em.binauralDecodeShTracked(x + 1j, wL, wR, R.reshape(-1, 3, 3), hop, handle=h)
    assert call() == 0


def test_benchmark_script_runs(tmp_path):
    out = tmp_path / "sh_tracked.json"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_sh_tracked_render.py"), "--seconds", "1",
                        "--out", str(out)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stdout + r.stderr
    res = json.loads(out.read_text())
    assert res["device"]["name"] and "power_limit_w" in res["device"] and res["ok"]
    for order in ("4", "7"):
        o = res["orders"][order]
        for name in ("static_head", "natural", "random"):
            t = o["tracks"][name]
            for key in ("ms_per_call", "msamples_per_s", "profile_ms", "rotation_stage_ms", "rotation_stage_bytes",
                        "rotation_stage_hbm_fraction", "max_rel_diff_vs_reference"):
                assert key in t, (order, name, key)
            assert t["max_rel_diff_vs_reference"] < 1e-12
        assert o["static_render"]["ms_per_call"] > 0
    assert res["orders"]["4"]["bank_render_natural"]["ms_per_call"] > 0
