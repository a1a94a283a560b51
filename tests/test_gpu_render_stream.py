"""Render sessions (emagls_render_stream_*): the concatenated block outputs equal the whole-signal renders, B200 only.
Against the device's whole-signal renders: 1e-12 relative max-norm; against the FP64 oracles: 1e-9, the bar of
test_gpu_render.py."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from oracle.tracked_oracle import binauralDecodeTracked as tracked_oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sh_tracked_oracle import binauralDecodeShTracked as sh_oracle  # noqa: E402

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


def splits(nblocks, block, pattern=(1, 3, 7)):
    sizes, k = [], 0
    while nblocks:
        m = min(nblocks, pattern[k % len(pattern)])
        sizes.append(m * block)
        nblocks -= m
        k += 1
    return sizes


def random_rotations(rng, nf):
    q = rng.standard_normal((nf, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(nf, 3, 3)


def run(s, x, sizes, entries=None, hop=1, lookahead=0, kw="track"):
    """Feed x in calls of `sizes`; each call appends the entries it needs plus `lookahead` more."""
    out, t, given = [], 0, 0
    for n in sizes:
        new = None
        if entries is not None:
            upto = min(len(entries), (t + n - 1) // hop + 1 + lookahead)
            new = entries[given:max(upto, given)]
            given += len(new)
        out.append(s.process(x[t:t + n], **({kw: new} if entries is not None else {})))
        t += n
    return np.concatenate(out)


def make_track(kind, rng, nf, pages):
    if kind == "random":
        return rng.integers(0, pages, nf).astype(np.int32)
    if kind == "constant":
        return np.full(nf, pages // 2, np.int32)
    t = np.arange(nf)                              # natural: a slow smooth sweep over neighbouring pages
    return np.mod(np.rint(pages / 2 + (pages / 2 - 1) * np.sin(2 * np.pi * t / 97)), pages).astype(np.int32)


@pytest.mark.parametrize("block,ln,ch", [(64, 512, 8), (480, 512, 32), (512, 512, 32), (1024, 100, 4), (256, 333, 3),
                                         (256, 1, 2)])
def test_static_session_equals_the_static_render(em, h, block, ln, ch):
    rng = np.random.default_rng(block + ln + ch)
    nb = 33
    x = rng.standard_normal((nb * block, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    with em.RenderStream(wL, wR, block, handle=h) as s:
        y = run(s, x, splits(nb, block))
    yd = em.binauralDecode(x, 1, wL, wR, 1, handle=h)
    yo = oracle.binauralDecode(x, 1, wL, wR, 1)
    assert rel(y, yd) < 1e-12
    assert rel(y, yo) < 1e-9


BANK_CASES = [(256, 37), (256, 480), (480, 480), (512, 480), (512, 9000)]


@pytest.mark.parametrize("track_kind", ["random", "constant", "natural"])
@pytest.mark.parametrize("fade_kind", ["hop", "one", "zero"])
@pytest.mark.parametrize("block,hop", BANK_CASES)
def test_bank_session_equals_the_tracked_render(em, h, block, hop, fade_kind, track_kind):
    fade = {"hop": hop, "one": 1, "zero": 0}[fade_kind]
    rng = np.random.default_rng(block + hop + fade + len(track_kind))
    ln, ch, pages = 512, 4, 12
    nb = max(24, 3 * hop // block + 4)
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))
    track = make_track(track_kind, rng, (n - 1) // hop + 1, pages)
    with em.RenderStream(wL, wR, block, hop, fade, handle=h) as s:
        y = run(s, x, splits(nb, block), track, hop)
    yd = em.binauralDecodeTracked(x, wL, wR, track, hop, fade, handle=h)
    assert rel(y, yd) < 1e-12
    yo = tracked_oracle(x, wL, wR, track, hop, fade)
    assert rel(y, yo) < 1e-9


def test_tracker_entry_spread_gives_identical_bits(em, h):
    rng = np.random.default_rng(5)
    block, hop, ln, ch, pages, nb = 256, 100, 300, 4, 10, 30
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))
    track = rng.integers(0, pages, (n - 1) // hop + 1 + 40).astype(np.int32)
    with em.RenderStream(wL, wR, block, hop, handle=h) as s:
        exact = run(s, x, splits(nb, block), track, hop)
    with em.RenderStream(wL, wR, block, hop, handle=h) as s:
        ahead = run(s, x, splits(nb, block), track, hop, lookahead=9)
    # everything up front, then calls with zero new entries
    with em.RenderStream(wL, wR, block, hop, handle=h) as s:
        parts = [s.process(x[:block], track)]
        parts += [s.process(x[t:t + block], np.zeros(0, np.int32)) for t in range(block, n, block)]
        upfront = np.concatenate(parts)
    assert np.array_equal(exact, ahead)
    assert np.array_equal(exact, upfront)


@pytest.mark.parametrize("order,block,hop,fade", [(0, 256, 480, 480), (1, 480, 480, 480), (4, 512, 480, 480),
                                                  (4, 128, 37, 0), (7, 256, 441, 200)])
def test_sh_session_equals_the_sh_tracked_render(em, h, order, block, hop, fade):
    rng = np.random.default_rng(order * 13 + block + hop)
    ch = (order + 1) ** 2
    ln, nb = 256, 24
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    nf = (n - 1) // hop + 1
    R = random_rotations(rng, nf)
    # bitwise-equal rotations across a call boundary: the frame that holds sample 4 block (a call boundary of
    # splits()) repeats its predecessor, so M is exactly Q_c there
    f = (4 * block) // hop
    if f > 0:
        R[f] = R[f - 1]
    with em.ShRenderStream(wL, wR, block, hop, fade, handle=h) as s:
        y = run(s, x, splits(nb, block), R, hop, kw="rotations")
    yd = em.binauralDecodeShTracked(x, wL, wR, R, hop, fade, handle=h)
    assert rel(y, yd) < 1e-12
    if order <= 4:
        yo = sh_oracle(x, wL, wR, R, hop, fade)
        assert rel(y, yo) < 1e-9


def _dev_run(em, h, s, x, sizes, entries, hop, kind):
    import torch
    dev = torch.device("cuda", 0)
    outs, t, given = [], 0, 0
    for n in sizes:
        upto = min(len(entries), (t + n - 1) // hop + 1) if entries is not None else 0
        xin = torch.from_numpy(np.ascontiguousarray(x[t:t + n].T)).to(dev)
        out = torch.empty((2, n), dtype=torch.float64, device=dev)
        trk, rot, nnew = None, None, 0
        if entries is not None:
            new = np.ascontiguousarray(entries[given:max(upto, given)])
            given += len(new)
            nnew = len(new)
            if kind == "bank":
                trk = new.ctypes.data_as(C.c_void_p)
            else:
                rot = new.ctypes.data_as(C.c_void_p)
        h.check(h.lib.emagls_render_stream_process_dev(s.ptr, C.c_void_p(xin.data_ptr()), n, trk, rot, nnew,
                                                       C.c_void_p(out.data_ptr())))
        torch.cuda.synchronize(dev)
        outs.append(out.cpu().numpy().T)
        t += n
    return np.concatenate(outs)


@pytest.mark.parametrize("kind", ["static", "bank", "sh"])
def test_dev_variant_equals_host_variant(em, h, kind):
    rng = np.random.default_rng(len(kind))
    block, hop, nb = 480, 300, 20
    n = nb * block
    if kind == "sh":
        ch = 16
        wL, wR = rng.standard_normal((200, ch)), rng.standard_normal((200, ch))
        entries = random_rotations(rng, (n - 1) // hop + 1)
        mk = lambda: em.ShRenderStream(wL, wR, block, hop, handle=h)   # noqa: E731
    else:
        ch = 6
        pages = 5 if kind == "bank" else 1
        wL, wR = rng.standard_normal((700, ch, pages)), rng.standard_normal((700, ch, pages))
        entries = rng.integers(0, pages, (n - 1) // hop + 1).astype(np.int32) if kind == "bank" else None
        mk = lambda: em.RenderStream(wL, wR, block, hop if kind == "bank" else None, handle=h)   # noqa: E731
    x = rng.standard_normal((n, ch))
    sizes = splits(nb, block)
    with mk() as s:
        yh = run(s, x, sizes, entries, hop, kw="rotations" if kind == "sh" else "track")
    with mk() as s:
        yd = _dev_run(em, h, s, x, sizes, entries, hop, kind)
    assert np.array_equal(yh, yd)


def test_sessions_on_one_handle_are_isolated(em, h):
    rng = np.random.default_rng(9)
    block, hop, nb = 256, 480, 20
    n = nb * block
    xb = rng.standard_normal((n, 4))
    bL, bR = rng.standard_normal((300, 4, 7)), rng.standard_normal((300, 4, 7))
    track = rng.integers(0, 7, (n - 1) // hop + 1).astype(np.int32)
    xs = rng.standard_normal((n, 9))
    sL, sR = rng.standard_normal((300, 9)), rng.standard_normal((300, 9))
    R = random_rotations(rng, (n - 1) // hop + 1)
    with em.RenderStream(bL, bR, block, hop, handle=h) as s:
        alone_b = run(s, xb, [block] * nb, track, hop)
    with em.ShRenderStream(sL, sR, block, hop, handle=h) as s:
        alone_s = run(s, xs, [block] * nb, R, hop, kw="rotations")
    sb = em.RenderStream(bL, bR, block, hop, handle=h)
    ss = em.ShRenderStream(sL, sR, block, hop, handle=h)
    yb, ys, given_b, given_s = [], [], 0, 0
    for k in range(nb):
        t = k * block
        need = (t + block - 1) // hop + 1
        yb.append(sb.process(xb[t:t + block], track[given_b:need]))
        ys.append(ss.process(xs[t:t + block], R[given_s:need]))
        given_b = given_s = need
    sb.close()
    ss.close()
    assert np.array_equal(np.concatenate(yb), alone_b)
    assert np.array_equal(np.concatenate(ys), alone_s)


def test_rejected_calls_change_nothing(em, h):
    rng = np.random.default_rng(11)
    block, hop, pages, ch = 256, 480, 6, 3
    nb = 12
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((200, ch, pages)), rng.standard_normal((200, ch, pages))
    track = rng.integers(0, pages, (n - 1) // hop + 1).astype(np.int32)
    with em.RenderStream(wL, wR, block, hop, handle=h) as s:
        ref = run(s, x, [block] * nb, track, hop)
    lib = h.lib
    s = em.RenderStream(wL, wR, block, hop, handle=h)
    out = np.zeros((block, 2), order="F")
    xa = np.asfortranarray(x[:block])
    bad_track = track[:2].copy()
    bad_track[1] = pages                   # page out of range
    l0 = h.launches
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block - 1, p(track), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(bad_track), None, 2, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, None, None, 0, p(out)) == -1      # no entries
    rot = np.eye(3).reshape(1, 9)
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(track), p(rot), 1, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, None, block, p(track), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(track), None, 1, None) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(track), None, -1, p(out)) == -1
    assert lib.emagls_render_stream_process(None, p(xa), block, p(track), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_process_dev(None, p(xa), block, p(track), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_destroy(None) == -1
    assert h.launches == l0
    got = run(s, x, [block] * nb, track, hop)
    s.close()
    assert np.array_equal(got, ref)
    # a track on a static session, rotations on a bank session, a track on an SH session
    with em.RenderStream(wL[:, :, 0], wR[:, :, 0], block, handle=h) as st:
        assert lib.emagls_render_stream_process(st.ptr, p(xa), block, p(track), None, 1, p(out)) == -1
    sL, sR = rng.standard_normal((50, 4)), rng.standard_normal((50, 4))
    with em.ShRenderStream(sL, sR, block, hop, handle=h) as ss:
        x4 = np.asfortranarray(rng.standard_normal((block, 4)))
        assert lib.emagls_render_stream_process(ss.ptr, p(x4), block, p(track), None, 1, p(out)) == -1
    # create: null pointers and arguments out of range launch nothing and return no session
    sp = C.c_void_p()
    wl0 = np.asfortranarray(wL)
    l0 = h.launches
    for args in [(None, p(wl0), 200, ch, pages, block, hop, hop), (p(wl0), p(wl0), 200, ch, pages, 15, hop, hop),
                 (p(wl0), p(wl0), 200, ch, pages, 8193, hop, hop), (p(wl0), p(wl0), 200, ch, pages, block, 0, 0),
                 (p(wl0), p(wl0), 200, ch, pages, block, hop, hop + 1), (p(wl0), p(wl0), 200, ch, pages, block, hop, -1)]:
        assert lib.emagls_render_stream_create(h.ptr, *args, C.byref(sp)) == -1
        assert not sp.value
    assert lib.emagls_render_stream_create(h.ptr, p(wl0), p(wl0), 200, ch, pages, block, hop, hop, None) == -1
    for order in (-1, 8):
        assert lib.emagls_render_stream_create_sh(h.ptr, p(wl0), p(wl0), 50, order, block, hop, hop, C.byref(sp)) == -1
    assert h.launches == l0


def test_create_destroy_cycles_do_not_leak(em):
    hh = em.Handle(0)
    rng = np.random.default_rng(2)
    # 1024 pages x 2 ears x 4 channels x 8193 bins x 16 B = 1.07 GB of filter spectra per session
    wL, wR = rng.standard_normal((1, 4, 1024)), rng.standard_normal((1, 4, 1024))
    x = rng.standard_normal((8192, 4))
    for _ in range(100):
        with em.RenderStream(wL, wR, 8192, 8192, handle=hh) as s:
            s.process(x, np.zeros(1, np.int32))
    # destroying the handle frees the sessions still open
    s1 = em.RenderStream(wL, wR, 8192, 8192, handle=hh)
    s2 = em.ShRenderStream(rng.standard_normal((10, 4)), rng.standard_normal((10, 4)), 64, 64, handle=hh)
    assert hh.lib.emagls_destroy(hh.ptr) == 0
    hh._h = None
    s1.close()
    s2.close()


def test_benchmark_script_runs_at_a_tiny_size(tmp_path):
    out = tmp_path / "stream.json"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_render_stream.py"), "--tiny",
                        "--out", str(out)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.loads(out.read_text())
    assert d["device"] and "power_limit_w" in d
    assert d["workloads"]
    for w in d["workloads"]:
        for key in ("workload", "block", "create_ms", "latency_ms_median", "latency_ms_p99", "latency_ms_max",
                    "device_ms_per_block", "launches_per_block", "realtime_factor", "stream_ms", "whole_ms",
                    "stream_over_whole", "max_rel_diff"):
            assert key in w, key
        assert w["max_rel_diff"] < 1e-12


def test_bank_whose_pages_leave_a_partial_last_batch(em, h):
    """1025 pages of 1.05 MB of spectra each: creation transforms them in batches of 256 and a last batch of one page.
    The bank renders the tracked render, and a session opened before it keeps its output bit for bit."""
    rng = np.random.default_rng(13)
    block, hop, pages, ch = 8192, 512, 1025, 4
    wL, wR = rng.standard_normal((1, ch, pages)), rng.standard_normal((1, ch, pages))
    nb = 6
    n = nb * block
    x = rng.standard_normal((n, ch))
    track = rng.integers(0, pages, (n - 1) // hop + 1).astype(np.int32)
    track[:4] = [pages - 1, 0, pages - 1, pages - 2]            # the pages of the last batch, early and often
    track[-3:] = pages - 1
    oL, oR = rng.standard_normal((300, 3, 5)), rng.standard_normal((300, 3, 5))
    xo = rng.standard_normal((8 * 256, 3))
    to = rng.integers(0, 5, (8 * 256 - 1) // 100 + 1).astype(np.int32)
    with em.RenderStream(oL, oR, 256, 100, handle=h) as ref:
        other_ref = run(ref, xo, [256] * 8, to, 100)
    other = em.RenderStream(oL, oR, 256, 100, handle=h)
    first = run(other, xo[:1024], [256] * 4, to, 100)
    with em.RenderStream(wL, wR, block, hop, handle=h) as s:
        y = run(s, x, splits(nb, block), track, hop)
        given = (1024 - 1) // 100 + 1
        rest = []
        for k in range(4, 8):
            need = (k * 256 + 255) // 100 + 1
            rest.append(other.process(xo[k * 256:(k + 1) * 256], to[given:need]))
            given = need
    other.close()
    assert np.array_equal(np.concatenate([first] + rest), other_ref)
    yd = em.binauralDecodeTracked(x, wL, wR, track, hop, handle=h)
    assert rel(y, yd) < 1e-12
    yo = tracked_oracle(x, wL, wR, track, hop)
    assert rel(y, yo) < 1e-9


def test_sh_bitwise_equal_rotations_give_exactly_q_c_across_calls(em, h):
    """Frames whose rotations are bitwise equal take exactly Q_c, also where the previous frame lies in an earlier call:
    a constant track with a frame every 37 samples, one block per call, gives the bits of a single frame."""
    rng = np.random.default_rng(17)
    order, block, nb = 4, 128, 20
    ch = (order + 1) ** 2
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((200, ch)), rng.standard_normal((200, ch))
    R1 = random_rotations(rng, 1)
    R = np.repeat(R1, (n - 1) // 37 + 1, axis=0)
    with em.ShRenderStream(wL, wR, block, 37, 37, handle=h) as s:
        many = run(s, x, [block] * nb, R, 37, kw="rotations")
    with em.ShRenderStream(wL, wR, block, n, 0, handle=h) as s:
        one = s.process(x, R1)
    assert np.array_equal(many, one)


def test_sh_output_bits_do_not_depend_on_the_call_split(em, h):
    rng = np.random.default_rng(19)
    order, block, hop, nb = 2, 256, 441, 24
    ch = (order + 1) ** 2
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((300, ch)), rng.standard_normal((300, ch))
    R = random_rotations(rng, (n - 1) // hop + 1)
    R[1::3] = R[0::3][:len(R[1::3])]                # every third frame repeats its predecessor bit for bit
    outs = []
    for sizes in (splits(nb, block), [block] * nb, [n]):
        with em.ShRenderStream(wL, wR, block, hop, handle=h) as s:
            outs.append(run(s, x, sizes, R, hop, kw="rotations"))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
