"""Render sessions for many listeners (emagls_render_stream_create_listeners / _create_sh_listeners), B200 only: every
listener's output equals a one-listener session on the same input and that listener's entries, and so the
whole-signal renders.  Against one-listener bank sessions 1e-14 relative max-norm (the pair transforms may run in
batches of another size), against the device's whole-signal renders 1e-12 and against the FP64 oracles 1e-9."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.tracked_oracle import binauralDecodeTracked as tracked_oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sh_tracked_oracle import binauralDecodeShTracked as sh_oracle  # noqa: E402
from test_gpu_render_stream import BANK_CASES, make_track, random_rotations, splits  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACK_KINDS = ("random", "constant", "natural")


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def h(em):
    return em.Handle(0)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def run(s, x, sizes, entries=None, hop=1, lookahead=0, kw="track"):
    """Feed x in calls of `sizes`; each call appends the entries (frames on axis 0) it needs plus `lookahead` more."""
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


def mixed_tracks(rng, nf, pages, L):
    """[nf, L]: listener l follows a random, constant or natural track (TRACK_KINDS[l % 3]); the constant and natural
    tracks are shifted per listener so that listeners differ"""
    cols = []
    for l in range(L):
        t = make_track(TRACK_KINDS[l % 3], rng, nf, pages)
        cols.append(t if l % 3 == 0 else np.mod(t + l // 3, pages).astype(np.int32))
    return np.stack(cols, 1)


BANK_LISTENER_CASES = [(2, *BANK_CASES[0]), (5, *BANK_CASES[2]), (37, *BANK_CASES[3]), (5, *BANK_CASES[4])]


@pytest.mark.parametrize("fade_kind", ["hop", "one", "zero"])
@pytest.mark.parametrize("L,block,hop", BANK_LISTENER_CASES)
def test_bank_listeners_equal_one_listener_sessions(em, h, L, block, hop, fade_kind):
    fade = {"hop": hop, "one": 1, "zero": 0}[fade_kind]
    rng = np.random.default_rng(L * 1000 + block + hop + fade)
    ln, ch, pages = 512, 4, 12
    nb = max(24, 3 * hop // block + 4)
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))
    tracks = mixed_tracks(rng, (n - 1) // hop + 1, pages, L)
    with em.RenderStream(wL, wR, block, hop, fade, listeners=L, handle=h) as s:
        y = run(s, x, splits(nb, block), tracks, hop)
    assert y.shape == (n, 2, L)
    for l in range(L):
        with em.RenderStream(wL, wR, block, hop, fade, handle=h) as s1:
            y1 = run(s1, x, splits(nb, block), tracks[:, l], hop)
        assert rel(y[:, :, l], y1) < 1e-14, l
        yd = em.binauralDecodeTracked(x, wL, wR, tracks[:, l], hop, fade, handle=h)
        assert rel(y[:, :, l], yd) < 1e-12, l
        if l < 3:
            assert rel(y[:, :, l], tracked_oracle(x, wL, wR, tracks[:, l], hop, fade)) < 1e-9, l


@pytest.mark.parametrize("L", [2, 9])
@pytest.mark.parametrize("order,block,hop,fade", [(0, 256, 480, 480), (1, 480, 480, 480), (4, 128, 37, 0),
                                                  (7, 256, 441, 200)])
def test_sh_listeners_equal_one_listener_sessions(em, h, order, block, hop, fade, L):
    rng = np.random.default_rng(order * 13 + block + hop + L)
    ch = (order + 1) ** 2
    ln, nb = 256, 24
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    nf = (n - 1) // hop + 1
    R = random_rotations(rng, nf * L).reshape(L, nf, 3, 3).transpose(1, 0, 2, 3)
    # listener 1 repeats a frame's rotation bit for bit across a call boundary of splits(): M is exactly Q_c there
    f = (4 * block) // hop
    if f > 0:
        R[f, 1] = R[f - 1, 1]
    with em.ShRenderStream(wL, wR, block, hop, fade, listeners=L, handle=h) as s:
        y = run(s, x, splits(nb, block), R, hop, kw="rotations")
    assert y.shape == (n, 2, L)
    for l in range(L):
        with em.ShRenderStream(wL, wR, block, hop, fade, handle=h) as s1:
            y1 = run(s1, x, splits(nb, block), R[:, l], hop, kw="rotations")
        assert rel(y[:, :, l], y1) < 1e-12, l
        yd = em.binauralDecodeShTracked(x, wL, wR, R[:, l], hop, fade, handle=h)
        assert rel(y[:, :, l], yd) < 1e-12, l
    for l in range(L):
        assert rel(y[:, :, l], sh_oracle(x, wL, wR, R[:, l], hop, fade)) < 1e-9, l


def test_union_of_300_listeners_reaches_the_whole_bank(em, h):
    rng = np.random.default_rng(300)
    L, block, hop, ln, ch, pages, nb = 300, 256, 100, 300, 4, 12, 12
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch, pages)), rng.standard_normal((ln, ch, pages))
    tracks = rng.integers(0, pages, ((n - 1) // hop + 1, L)).astype(np.int32)
    # every block's union is the whole bank
    for b in range(nb):
        f0, f1 = b * block // hop, (b * block + block - 1) // hop
        assert len(np.unique(tracks[f0:f1 + 1])) == pages
    with em.RenderStream(wL, wR, block, hop, listeners=L, handle=h) as s:
        y = run(s, x, splits(nb, block), tracks, hop)
    for l in (0, 1, 57, 150, 298, 299):
        yd = em.binauralDecodeTracked(x, wL, wR, tracks[:, l], hop, handle=h)
        assert rel(y[:, :, l], yd) < 1e-12, l
        with em.RenderStream(wL, wR, block, hop, handle=h) as s1:
            assert rel(y[:, :, l], run(s1, x, splits(nb, block), tracks[:, l], hop)) < 1e-14, l


@pytest.mark.parametrize("kind", ["bank", "sh"])
def test_listeners_are_independent_bit_for_bit(em, h, kind):
    """Permuting the listeners permutes the outputs, and listeners with identical entries get identical bits."""
    rng = np.random.default_rng(23 if kind == "bank" else 29)
    block, hop, nb, L = 256, 300, 16, 7
    n = nb * block
    nf = (n - 1) // hop + 1
    if kind == "bank":
        ch, pages = 4, 9
        wL, wR = rng.standard_normal((400, ch, pages)), rng.standard_normal((400, ch, pages))
        e = mixed_tracks(rng, nf, pages, L)
        e[:, 5] = e[:, 2]
        mk = lambda: em.RenderStream(wL, wR, block, hop, listeners=L, handle=h)   # noqa: E731
        kw = "track"
    else:
        ch = 9
        wL, wR = rng.standard_normal((200, ch)), rng.standard_normal((200, ch))
        e = random_rotations(rng, nf * L).reshape(L, nf, 3, 3).transpose(1, 0, 2, 3).copy()
        e[:, 5] = e[:, 2]
        mk = lambda: em.ShRenderStream(wL, wR, block, hop, listeners=L, handle=h)   # noqa: E731
        kw = "rotations"
    x = rng.standard_normal((n, ch))
    perm = rng.permutation(L)
    with mk() as s:
        y = run(s, x, splits(nb, block), e, hop, kw=kw)
    with mk() as s:
        yp = run(s, x, splits(nb, block), np.ascontiguousarray(e[:, perm]), hop, kw=kw)
    assert np.array_equal(yp, y[:, :, perm])
    assert np.array_equal(y[:, :, 5], y[:, :, 2])


@pytest.mark.parametrize("kind,per_block", [("bank", 5), ("sh", 7)])
def test_launches_per_block_do_not_depend_on_the_listeners(em, h, kind, per_block):
    rng = np.random.default_rng(31)
    block, hop, nb = 256, 200, 10
    n = nb * block
    nf = (n - 1) // hop + 1
    for L in (1, 64):
        if kind == "bank":
            ch, pages = 4, 40
            wL, wR = rng.standard_normal((300, ch, pages)), rng.standard_normal((300, ch, pages))
            e = rng.integers(0, pages, (nf, L)).astype(np.int32)
            s = em.RenderStream(wL, wR, block, hop, listeners=L, handle=h)
            kw = "track"
        else:
            ch = 16
            wL, wR = rng.standard_normal((300, ch)), rng.standard_normal((300, ch))
            e = random_rotations(rng, nf * L).reshape(nf, L, 3, 3)
            s = em.ShRenderStream(wL, wR, block, hop, listeners=L, handle=h)
            kw = "rotations"
        if L == 1:
            e = e[:, 0]
        x = rng.standard_normal((n, ch))
        l0 = h.launches
        run(s, x, splits(nb, block), e, hop, kw=kw)
        assert h.launches - l0 == per_block * nb, L
        s.close()


def _dev_run(h, s, x, sizes, entries, hop, kind, L):
    import torch
    dev = torch.device("cuda", 0)
    outs, t, given = [], 0, 0
    for n in sizes:
        upto = min(len(entries), (t + n - 1) // hop + 1)
        xin = torch.from_numpy(np.ascontiguousarray(x[t:t + n].T)).to(dev)
        out = torch.empty((L, 2, n), dtype=torch.float64, device=dev)
        new = entries[given:max(upto, given)]
        given += len(new)
        nnew = len(new)
        new = np.ascontiguousarray(np.swapaxes(new, 0, 1))          # listener-major
        ptr = new.ctypes.data_as(C.c_void_p)
        trk, rot = (ptr, None) if kind == "bank" else (None, ptr)
        h.check(h.lib.emagls_render_stream_process_dev(s.ptr, C.c_void_p(xin.data_ptr()), n, trk, rot, nnew,
                                                       C.c_void_p(out.data_ptr())))
        torch.cuda.synchronize(dev)
        outs.append(out.cpu().numpy().transpose(2, 1, 0))
        t += n
    return np.concatenate(outs)


@pytest.mark.parametrize("kind", ["bank", "sh"])
def test_dev_and_host_variants_and_entry_spreads_give_identical_bits(em, h, kind):
    rng = np.random.default_rng(37 + len(kind))
    block, hop, nb, L = 480, 300, 20, 6
    n = nb * block
    nf = (n - 1) // hop + 1 + 30
    if kind == "sh":
        ch = 16
        wL, wR = rng.standard_normal((200, ch)), rng.standard_normal((200, ch))
        e = random_rotations(rng, nf * L).reshape(nf, L, 3, 3)
        mk = lambda: em.ShRenderStream(wL, wR, block, hop, listeners=L, handle=h)   # noqa: E731
        kw = "rotations"
    else:
        ch, pages = 6, 5
        wL, wR = rng.standard_normal((700, ch, pages)), rng.standard_normal((700, ch, pages))
        e = mixed_tracks(rng, nf, pages, L)
        mk = lambda: em.RenderStream(wL, wR, block, hop, listeners=L, handle=h)   # noqa: E731
        kw = "track"
    x = rng.standard_normal((n, ch))
    sizes = splits(nb, block)
    with mk() as s:
        yh = run(s, x, sizes, e, hop, kw=kw)
    with mk() as s:
        yd = _dev_run(h, s, x, sizes, e, hop, kind, L)
    assert np.array_equal(yh, yd)
    with mk() as s:
        ahead = run(s, x, sizes, e, hop, lookahead=7, kw=kw)
    with mk() as s:
        parts = [s.process(x[:block], **{kw: e})]
        parts += [s.process(x[t:t + block], **{kw: e[:0]}) for t in range(block, n, block)]
        upfront = np.concatenate(parts)
    assert np.array_equal(yh, ahead)
    assert np.array_equal(yh, upfront)


def test_rejected_calls_change_nothing(em, h):
    rng = np.random.default_rng(41)
    block, hop, pages, ch, L = 256, 480, 6, 3, 4
    nb = 12
    n = nb * block
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((200, ch, pages)), rng.standard_normal((200, ch, pages))
    tracks = rng.integers(0, pages, ((n - 1) // hop + 1, L)).astype(np.int32)
    with em.RenderStream(wL, wR, block, hop, listeners=L, handle=h) as s:
        ref = run(s, x, [block] * nb, tracks, hop)
    lib = h.lib
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    s = em.RenderStream(wL, wR, block, hop, listeners=L, handle=h)
    out = np.zeros((block, 2, L), order="F")
    xa = np.asfortranarray(x[:block])
    good = np.ascontiguousarray(tracks[:1].T)     # [L x 1]: listener-major, one frame each
    bad = good.copy()
    bad[L - 1] = pages                            # the last listener's page is out of range
    neg = good.copy()
    neg[1] = -1
    l0 = h.launches
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(bad), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(neg), None, 1, p(out)) == -1
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, None, None, 0, p(out)) == -1   # no entries
    rot = np.tile(np.eye(3).reshape(1, 9), (L, 1))
    assert lib.emagls_render_stream_process(s.ptr, p(xa), block, p(good), p(rot), 1, p(out)) == -1
    assert h.launches == l0
    got = run(s, x, [block] * nb, tracks, hop)
    s.close()
    assert np.array_equal(got, ref)
    # an SH session: rotations that do not cover the call, a track
    sL, sR = rng.standard_normal((50, 4)), rng.standard_normal((50, 4))
    x4 = rng.standard_normal((n, 4))
    R = random_rotations(rng, ((n - 1) // hop + 1) * L).reshape(-1, L, 3, 3)
    with em.ShRenderStream(sL, sR, block, hop, listeners=L, handle=h) as ss:
        sref = run(ss, x4, [block] * nb, R, hop, kw="rotations")
    with em.ShRenderStream(sL, sR, block, hop, listeners=L, handle=h) as ss:
        xs = np.asfortranarray(x4[:2 * hop // block * block + block])
        l0 = h.launches
        assert lib.emagls_render_stream_process(ss.ptr, p(xs), xs.shape[0], None, p(np.ascontiguousarray(R[:1])), 1,
                                                p(np.zeros((xs.shape[0], 2, L), order="F"))) == -1
        assert lib.emagls_render_stream_process(ss.ptr, p(xs), block, p(good), None, 1, p(out)) == -1
        assert h.launches == l0
        assert np.array_equal(run(ss, x4, [block] * nb, R, hop, kw="rotations"), sref)
    # create: listener counts outside [1, 4096], and more than one listener on a static session
    sp = C.c_void_p()
    wl0 = np.asfortranarray(wL)
    l0 = h.launches
    for nl in (0, -1, 4097):
        assert lib.emagls_render_stream_create_listeners(h.ptr, p(wl0), p(wl0), 200, ch, pages, nl, block, hop, hop,
                                                         C.byref(sp)) == -1
        assert not sp.value
        assert lib.emagls_render_stream_create_sh_listeners(h.ptr, p(wl0), p(wl0), 50, 1, nl, block, hop, hop,
                                                            C.byref(sp)) == -1
        assert not sp.value
    assert lib.emagls_render_stream_create_listeners(h.ptr, p(wl0), p(wl0), 200, ch, 1, 2, block, hop, hop,
                                                     C.byref(sp)) == -1
    assert not sp.value
    # the existing checks apply to the new entry points too
    assert lib.emagls_render_stream_create_listeners(h.ptr, p(wl0), p(wl0), 200, ch, pages, 2, 15, hop, hop,
                                                     C.byref(sp)) == -1
    assert lib.emagls_render_stream_create_sh_listeners(h.ptr, p(wl0), p(wl0), 50, 8, 2, block, hop, hop,
                                                        C.byref(sp)) == -1
    # an SH forward transform of 2^31 samples: 4096 listeners x 64 channels x 2 x 4096
    assert lib.emagls_render_stream_create_sh_listeners(h.ptr, p(wl0), p(wl0), 50, 7, 4096, 4096, hop, hop,
                                                        C.byref(sp)) == -1
    assert not sp.value
    assert h.launches == l0
    with pytest.raises(ValueError):
        with em.RenderStream(wL, wR, block, hop, listeners=L, handle=h) as s:
            s.process(x[:block], tracks[:1, :L - 1])


def test_benchmark_script_runs_at_a_tiny_size(tmp_path):
    out = tmp_path / "listeners.json"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_render_listeners.py"), "--tiny",
                        "--out", str(out)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.loads(out.read_text())
    assert d["device"] and "power_limit_w" in d
    assert d["workloads"] and d["separate_vs_shared"]
    for w in d["workloads"]:
        for key in ("workload", "listeners", "block", "device_ms_per_block", "launches_per_block",
                    "distinct_pages_mean", "distinct_pages_max", "latency_ms_p99", "session_bytes",
                    "realtime_listeners", "max_rel_diff"):
            assert key in w, key
        assert w["max_rel_diff"] < 1e-12
