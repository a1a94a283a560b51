"""Head-tracked render (emagls_binaural_decode_tracked) against oracle/tracked_oracle.py, B200 only.
Tolerance: 1e-9 relative max-norm, the bar of test_gpu_render.py."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from oracle.tracked_oracle import binauralDecodeTracked

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


def bank(rng, ln, ch, pages):
    return rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))


@pytest.mark.parametrize("n,ch,ln,pages,hop,fade,comp", [
    (20000, 8, 512, 5, 37, 37, False),      # hop shorter than the filter
    (20000, 8, 512, 5, 37, 0, True),        # hard switch
    (30001, 6, 256, 4, 441, 1, False),      # odd hop, one-sample fade, odd length (staged forward route)
    (30000, 6, 256, 4, 441, 441, True),
    (40000, 4, 512, 3, 9000, 9000, False),  # frames longer than a block
    (40000, 4, 512, 3, 9000, 0, True),
    (300, 5, 128, 3, 1000, 500, False),     # signal shorter than one frame
    (5000, 1, 64, 4, 100, 100, False),      # single channel
])
def test_tracked_render_matches_oracle(em, h, n, ch, ln, pages, hop, fade, comp):
    rng = np.random.default_rng(n + hop + fade)
    x = rng.standard_normal((n, ch))
    wL, wR = bank(rng, ln, ch, pages)
    track = rng.integers(0, pages, frames_needed(n, hop))          # exactly as long as needed
    y = em.binauralDecodeTracked(x, wL, wR, track, hop, fade, comp, handle=h)
    yo = binauralDecodeTracked(x, wL, wR, track, hop, fade, comp)
    assert y.shape == yo.shape
    assert rel(y, yo) < 1e-9


def test_constant_track_is_the_static_render(em, h):
    rng = np.random.default_rng(4)
    x = rng.standard_normal((50000, 12))
    wL, wR = bank(rng, 512, 12, 4)
    for comp in (False, True):
        y = em.binauralDecodeTracked(x, wL, wR, np.full(frames_needed(50000, 480), 2), 480, None, comp, handle=h)
        ys = em.binauralDecode(x, 48000, wL[:, :, 2], wR[:, :, 2], 48000, comp, handle=h)
        assert y.shape == ys.shape and rel(y, ys) < 1e-12


@pytest.mark.parametrize("kind", ["every_frame", "returning"])
def test_switching_tracks(em, h, kind):
    rng = np.random.default_rng(5)
    n, hop, pages = 30000, 480, 6
    x = rng.standard_normal((n, 8))
    wL, wR = bank(rng, 512, 8, pages)
    nf = frames_needed(n, hop)
    track = np.arange(nf) % pages if kind == "every_frame" else np.array([0, 1, 0, 2, 2, 1, 0] * nf)[:nf]
    y = em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h)
    assert rel(y, binauralDecodeTracked(x, wL, wR, track, hop)) < 1e-9


def test_fft_sizes_and_chunking_give_the_same_output(em, h, monkeypatch):
    rng = np.random.default_rng(6)
    n, hop, ch = 60000, 441, 6
    x = rng.standard_normal((n, ch))
    wL, wR = bank(rng, 512, ch, 5)
    track = rng.integers(0, 5, frames_needed(n, hop))
    yo = binauralDecodeTracked(x, wL, wR, track, hop)
    l0 = h.launches
    em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h)
    one_call = h.launches - l0
    for fft in ("1024", "2048", "4096", "16384"):
        monkeypatch.setenv("EMAGLS_TRACK_FFT", fft)
        assert rel(em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h), yo) < 1e-9
    monkeypatch.delenv("EMAGLS_TRACK_FFT")
    monkeypatch.setenv("EMAGLS_TRACK_WS_MB", "1")
    l0 = h.launches
    assert rel(em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h), yo) < 1e-9
    # every chunk adds at least a gather, a multiply-accumulate and a combine launch: at least three chunks
    assert h.launches - l0 >= one_call + 6


def test_consecutive_pieces_compose(em, h):
    rng = np.random.default_rng(7)
    n, m, ln, hop = 40000, 17001, 512, 480
    x = rng.standard_normal((n, 8))
    wL, wR = bank(rng, ln, 8, 4)
    track = rng.integers(0, 4, frames_needed(n, hop))
    whole = em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h)
    first = em.binauralDecodeTracked(x[:m], wL, wR, track, hop, handle=h)
    halo = ln - 1
    second = em.binauralDecodeTracked(x[m - halo:], wL, wR, track, hop, firstSample=m - halo, handle=h)[halo:]
    assert rel(np.concatenate([first, second], 0), whole) < 1e-12


def test_time_block_sharded_tracked_render(em, h):
    from emagls_b200 import dist as emdist
    rng = np.random.default_rng(8)
    n, taps, ch, world, hop = 50000, 512, 16, 4, 480
    x = rng.standard_normal((n, ch))
    wL, wR = bank(rng, taps, ch, 5)
    track = rng.integers(0, 5, frames_needed(n, hop))
    ref = binauralDecodeTracked(x, wL, wR, track, hop)
    parts = []
    for r in range(world):
        lo, hi, halo = emdist.render_shard(n, taps, r, world)
        sr = emdist.ShardedRenderer(h, x[lo - halo:hi], wL, wR, halo, track=track, hop=hop, first_sample=lo - halo)
        sr.step()
        parts.append(sr.wait().copy())
    got = np.concatenate(parts, 0)
    assert got.shape == ref.shape and rel(got, ref) < 1e-9


def test_designed_bank_end_to_end(em, h, grids):
    """A bank designed on the device over k head orientations, rendered with a track over its k pages."""
    from emagls_b200 import synth
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    k = 6
    wL, wR = em.getEMagLs2Filters(hL, hR, az, ze, grids["micRadius"], grids["micGridAziRad"], grids["micGridZenRad"],
                                  4, grids["fs"], 512, rotations=synth.orientation_grid()[:k], handle=h)
    assert wL.shape[2] == k
    rng = np.random.default_rng(9)
    n, hop = 24000, 480
    x = rng.standard_normal((n, wL.shape[1]))
    track = rng.integers(0, k, frames_needed(n, hop))
    y = em.binauralDecodeTracked(x, wL, wR, track, hop, None, True, handle=h)
    yo = binauralDecodeTracked(x, wL, wR, track, hop, None, True)
    assert y.shape == (n - 255, 2) and rel(y, yo) < 1e-9


def test_complex_bank_and_signal(em, h):
    rng = np.random.default_rng(10)
    n, ch, ln, pages, hop = 12000, 9, 256, 3, 300
    x = rng.standard_normal((n, ch)) + 1j * rng.standard_normal((n, ch))
    wL = rng.standard_normal((ln, ch, pages)) + 1j * rng.standard_normal((ln, ch, pages))
    wR = rng.standard_normal((ln, ch, pages)) + 1j * rng.standard_normal((ln, ch, pages))
    track = rng.integers(0, pages, frames_needed(n, hop))
    y = em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h)
    yo = binauralDecodeTracked(x, wL, wR, track, hop)
    assert not np.iscomplexobj(y) and rel(y, yo) < 1e-9


def test_dev_variant_equals_host_variant(em, h):
    import torch
    rng = np.random.default_rng(11)
    n, ch, ln, pages, hop, fade = 30000, 8, 512, 4, 480, 200
    x = rng.standard_normal((n, ch))
    wL, wR = bank(rng, ln, ch, pages)
    track = rng.integers(0, pages, frames_needed(n, hop)).astype(np.int32)
    y = em.binauralDecodeTracked(x, wL, wR, track, hop, fade, True, handle=h)
    dev = torch.device("cuda", 0)
    xd = torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)                 # [n, ch] column-major
    wd = [torch.from_numpy(np.ascontiguousarray(w.T)).to(dev) for w in (wL, wR)]
    rows = n - ln // 2 + 1
    out = torch.empty((2, rows), dtype=torch.float64, device=dev)
    h.check(h.lib.emagls_binaural_decode_tracked_dev(h.ptr, xd.data_ptr(), n, ch, wd[0].data_ptr(), wd[1].data_ptr(),
                                                     ln, pages, track.ctypes.data_as(C.c_void_p), track.size, hop,
                                                     fade, 0, 1, out.data_ptr()))
    torch.cuda.ExternalStream(h.stream, device=dev).synchronize()
    assert np.array_equal(out.cpu().numpy().T, y)


def test_rejected_arguments_launch_nothing(em, h):
    rng = np.random.default_rng(12)
    n, ch, ln, pages, hop = 2000, 3, 64, 3, 100
    x = rng.standard_normal((n, ch))
    wL, wR = bank(rng, ln, ch, pages)
    track = rng.integers(0, pages, frames_needed(n, hop))
    cases = [
        dict(hop=0),
        dict(fade=-1),
        dict(fade=hop + 1),
        dict(firstSample=-1),
        dict(track=track[:-1]),
        dict(track=np.where(np.arange(track.size) == 7, pages, track)),
        dict(track=np.where(np.arange(track.size) == 3, -1, track)),
        dict(wL=wL[:-1], wR=wR[:-1], compensateDelay=True),        # odd length with the compensated delay
    ]
    for c in cases:
        args = dict(wL=wL, wR=wR, track=track, hop=hop, fade=None, compensateDelay=False, firstSample=0)
        args.update(c)
        l0 = h.launches
        with pytest.raises(em.EmaglsError) as e:
            em.binauralDecodeTracked(x, args["wL"], args["wR"], args["track"], args["hop"], args["fade"],
                                     args["compensateDelay"], firstSample=args["firstSample"], handle=h)
        assert e.value.code == -1 and h.launches == l0, c
    tr = track.astype(np.int32)
    xf, wf = np.asfortranarray(x), np.asfortranarray(wL)
    ptrs = [xf.ctypes.data_as(C.c_void_p), wf.ctypes.data_as(C.c_void_p), wf.ctypes.data_as(C.c_void_p),
            tr.ctypes.data_as(C.c_void_p), np.zeros((n, 2)).ctypes.data_as(C.c_void_p)]
    for k in range(5):
        p = list(ptrs)
        p[k] = None
        l0 = h.launches
        rc = h.lib.emagls_binaural_decode_tracked(h.ptr, p[0], n, ch, p[1], p[2], ln, pages, p[3], tr.size, hop, hop,
                                                  0, 0, p[4])
        assert rc == -1 and h.launches == l0


def test_benchmark_script_runs(tmp_path):
    out = tmp_path / "tracked.json"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_tracked_render.py"), "--seconds", "1",
                        "--pages", "360", "--out", str(out)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stdout + r.stderr
    res = json.loads(out.read_text())
    assert res["device"]["name"] and "power_limit_w" in res["device"]
    for name in ("static_head", "natural", "worst_case"):
        t = res["tracks"][name]
        for key in ("ms_per_call", "msamples_per_s", "pages_per_block_mean", "pages_per_block_max", "distinct_pages",
                    "hbm_bytes_algorithmic", "hbm_fraction_algorithmic", "profile_ms"):
            assert key in t, (name, key)
    for name in ("natural", "worst_case"):
        assert res["tracks"][name]["max_rel_diff_vs_composed_static"] < 1e-9
    assert res["static_render"]["default"]["ms_per_call"] > 0 and res["static_render"]["cufft"]["ms_per_call"] > 0
