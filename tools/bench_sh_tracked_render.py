"""Cost of the head-tracked render of SH signals (emagls_binaural_decode_sh_tracked_dev) on one GPU; writes one JSON
file to --out.

A seeded random real SH signal of --seconds at 48 kHz and one random filter pair of --taps taps, both in device memory
(values do not change the cost), at orders 4 (25 channels) and 7 (64 channels).  Three tracks at hop 480 (a 100 Hz
tracker) with fade = hop: a static head (yaw 30 deg, pitch 10 deg), natural head motion (the yaw / pitch formulas of
tools/bench_tracked_render.py, continuous, not snapped to a grid) and a seeded random orientation per frame.  Per
track and order: ms per call (CUDA events around three warmed calls), Msamples/s, the per-class profiler split
(separate call) and the rotation stage (render_stage: the frame-matrix and rotation kernels) with its share of
7.7 TB/s by its byte count, 2 C 8 B per sample.  For comparison in the same process: the static render of the same
signal, and at order 4 the bank render (emagls_binaural_decode_tracked_dev) of a 3600-page bank on the natural track
snapped to synth.orientation_grid().
Correctness at the timed size: the natural and random tracks over the first --check-seconds against an independent
torch reference (the signal rotated with oracle getSHrotMtx matrices, then emagls_binaural_decode_dev); the static
head over the whole signal against emagls_rotate_sh_dev followed by the static render.

    python tools/bench_sh_tracked_render.py --out profiles/r04_sh_tracked_render.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_tracked_render import FS, HBM_PEAK, device_info, natural_track  # noqa: E402


def natural_rotations(frames, hop):
    from emagls_b200 import synth
    t = (np.arange(frames) + 0.5) * hop / FS
    yaw = 60 * np.sin(2 * np.pi * 0.5 * t) + 20 * np.sin(2 * np.pi * 0.13 * t)
    pitch = 20 * np.sin(2 * np.pi * 0.2 * t)
    return np.stack([synth.rotation_yaw_pitch(y, p) for y, p in zip(yaw, pitch)])


def random_rotations(rng, frames):
    q = rng.standard_normal((frames, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(frames, 3, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--orders", default="4,7")
    ap.add_argument("--taps", type=int, default=512)
    ap.add_argument("--hop", type=int, default=480)
    ap.add_argument("--bank-pages", type=int, default=3600)
    ap.add_argument("--check-seconds", type=float, default=30.0, help="reference check length, moving tracks")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()

    import torch
    import emagls_b200 as em
    import oracle
    from emagls_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the render has no CPU path")
    dev = torch.device("cuda", 0)
    h = em.Handle(0)
    st = torch.cuda.ExternalStream(h.stream, device=dev)
    n, ln, hop = int(a.seconds * FS), a.taps, a.hop
    fade = hop
    frames = (n - 1) // hop + 1
    rng = np.random.default_rng(a.seed)
    yaw0, pitch0 = 30.0, 10.0
    tracks = {
        "static_head": np.repeat(synth.rotation_yaw_pitch(yaw0, pitch0)[None], frames, 0),
        "natural": natural_rotations(frames, hop),
        "random": random_rotations(rng, frames),
    }
    rot_d = {k: torch.from_numpy(np.ascontiguousarray(v.reshape(-1, 9))).to(dev) for k, v in tracks.items()}

    def timed(fn, reps=3):
        fn()
        st.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(reps):
            fn()
        e1.record(st)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    def profiled(fn):
        h.profile(True)
        h.profile_read(reset=True)
        fn()
        prof = h.profile_read(reset=True)
        h.profile(False)
        return {k: round(v["ms"], 4) for k, v in prof.items() if v["n"]}

    res = dict(device=device_info(), config=dict(seconds=a.seconds, samples=n, taps=ln, hop=hop, fade=fade, fs=FS,
                                                  seed=a.seed, static_head_yaw_pitch_deg=[yaw0, pitch0]),
               orders={})
    ok = True
    for order in [int(v) for v in a.orders.split(",") if v]:
        Cn = (order + 1) ** 2
        g = torch.Generator(device=dev).manual_seed(a.seed + order)
        # signal [n, C] column-major == [C, n] row-major; filters [len, C] column-major == [C, len] row-major
        x = torch.randn((Cn, n), generator=g, dtype=torch.float64, device=dev)
        wL = torch.randn((Cn, ln), generator=g, dtype=torch.float64, device=dev) / ln
        wR = torch.randn((Cn, ln), generator=g, dtype=torch.float64, device=dev) / ln
        out = torch.empty((2, n), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()        # filled on torch's stream; the library works on the handle's

        def sh_tracked(name, nn=n, y=out, xx=x):
            h.check(h.lib.emagls_binaural_decode_sh_tracked_dev(h.ptr, xx.data_ptr(), nn, order, wL.data_ptr(),
                                                                wR.data_ptr(), ln, rot_d[name].data_ptr(), frames,
                                                                hop, fade, 0, 0, y.data_ptr()))

        def static(nn=n, y=out, xx=x):
            h.check(h.lib.emagls_binaural_decode_dev(h.ptr, xx.data_ptr(), nn, Cn, wL.data_ptr(), wR.data_ptr(), ln, 0,
                                                     y.data_ptr()))

        r = dict(channels=Cn, tracks={})
        rot_bytes = 2 * Cn * 8 * n
        for name in tracks:
            ms = timed(lambda: sh_tracked(name))
            prof = profiled(lambda: sh_tracked(name))
            stage = prof.get("render_stage", 0.0)
            r["tracks"][name] = dict(ms_per_call=round(ms, 3), msamples_per_s=round(n / ms / 1e3, 1), profile_ms=prof,
                                     rotation_stage_ms=stage, rotation_stage_bytes=rot_bytes,
                                     rotation_stage_hbm_fraction=round(rot_bytes / (stage * 1e-3) / HBM_PEAK, 4)
                                     if stage > 0 else None)
            print(order, name, json.dumps(r["tracks"][name]), flush=True)
        r["static_render"] = dict(ms_per_call=round(timed(static), 3), profile_ms=profiled(static))
        print(order, "static", r["static_render"], flush=True)

        # correctness: moving tracks against the torch reference over the first check_seconds
        nn = min(n, int(a.check_seconds * FS))
        nfc = (nn - 1) // hop + 1
        for name in ("natural", "random"):
            R = tracks[name][:nfc]
            Q = torch.from_numpy(np.stack([oracle.getSHrotMtx(Rf, order, "real") for Rf in R])).to(dev)
            same = torch.from_numpy(np.concatenate([[True], [np.array_equal(R[f].view(np.uint64), R[f - 1].view(np.uint64))
                                                             for f in range(1, nfc)]])).to(dev)
            xs = torch.zeros((nfc * hop, Cn), dtype=torch.float64, device=dev)
            xs[:nn] = x[:, :nn].T
            xf = xs.view(nfc, hop, Cn)
            yc = torch.bmm(xf, Q)
            ya = torch.bmm(xf, torch.cat([Q[:1], Q[:-1]]))
            i = torch.arange(hop, device=dev, dtype=torch.float64)
            gg = torch.where(i < fade, (i + 0.5) / max(fade, 1), torch.ones_like(i))[None, :, None]
            blend = (~same)[:, None, None] & (i < fade)[None, :, None]
            xr = torch.where(blend, (1.0 - gg) * ya + gg * yc, yc).reshape(-1, Cn)[:nn].T.contiguous()
            ref = torch.empty((2, nn), dtype=torch.float64, device=dev)
            got = torch.empty((2, nn), dtype=torch.float64, device=dev)
            xn = x[:, :nn].contiguous()
            torch.cuda.synchronize()
            h.check(h.lib.emagls_binaural_decode_dev(h.ptr, xr.data_ptr(), nn, Cn, wL.data_ptr(), wR.data_ptr(), ln, 0,
                                                     ref.data_ptr()))
            sh_tracked(name, nn, got, xn)
            st.synchronize()
            err = float(((got - ref).abs().max() / ref.abs().max()).item())
            r["tracks"][name]["max_rel_diff_vs_reference"] = err
            r["tracks"][name]["reference_check_samples"] = nn
            ok &= err < 1e-12
            print(order, name, "reference check", err, "over", nn, "samples", flush=True)
            del Q, xs, xf, yc, ya, xr, ref, got, xn
        # the static head over the whole signal: emagls_rotate_sh (R = E^T for E = euler2rotationMatrix(-yaw, -pitch,
        # 0, 'zyx')) and the static render
        xr = torch.empty_like(x)
        ref = torch.empty_like(out)
        h.check(h.lib.emagls_rotate_sh_dev(h.ptr, x.data_ptr(), n, order, math.radians(-yaw0), math.radians(-pitch0),
                                           0.0, xr.data_ptr()))
        static(n, ref, xr)
        sh_tracked("static_head")
        st.synchronize()
        err = float(((out - ref).abs().max() / ref.abs().max()).item())
        r["tracks"]["static_head"]["max_rel_diff_vs_reference"] = err
        r["tracks"]["static_head"]["reference_check_samples"] = n
        ok &= err < 1e-12
        print(order, "static_head reference check", err, flush=True)
        del xr, ref

        if order == 4 and a.bank_pages > 0:
            P = a.bank_pages
            bL = torch.randn((P, Cn, ln), generator=g, dtype=torch.float64, device=dev) / ln
            bR = torch.randn((P, Cn, ln), generator=g, dtype=torch.float64, device=dev) / ln
            trk = (natural_track(frames, hop, P) if P >= 3600 else rng.integers(0, P, frames)).astype(np.int32)
            torch.cuda.synchronize()

            def bank():
                h.check(h.lib.emagls_binaural_decode_tracked_dev(h.ptr, x.data_ptr(), n, Cn, bL.data_ptr(),
                                                                 bR.data_ptr(), ln, P, trk.ctypes.data_as(C.c_void_p),
                                                                 trk.size, hop, fade, 0, 0, out.data_ptr()))
            r["bank_render_natural"] = dict(pages=P, bank_bytes=2 * P * Cn * ln * 8, ms_per_call=round(timed(bank), 3),
                                            profile_ms=profiled(bank))
            print(order, "bank", r["bank_render_natural"], flush=True)
            del bL, bR
        res["orders"][str(order)] = r
        del x, wL, wR, out
        torch.cuda.empty_cache()
    res["ok"] = bool(ok)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(dict(out=a.out, ok=ok)))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
