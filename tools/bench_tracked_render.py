"""Cost of the head-tracked render (emagls_binaural_decode_tracked_dev) on one GPU; writes one JSON file to --out.

A seeded random bank of --pages pages (default 3600: the head-orientation grid of synth.orientation_grid(), page =
pitch_row * 360 + yaw_deg) at --taps taps and --ch channels and a --seconds long --ch channel signal at 48 kHz, both
in device memory (filter values do not change the render's cost).  Three tracks at hop 480 (a 100 Hz tracker) with
fade = hop: a static head, natural head motion (yaw 60 sin(2 pi 0.5 t) + 20 sin(2 pi 0.13 t) deg, pitch
20 sin(2 pi 0.2 t) deg, snapped to the grid) and a seeded random page per frame.  Per track: ms per call (CUDA events
around three warmed calls), pages per block, the HBM byte model and the per-class profiler split (separate call).
For reference the static render of the same signal is timed in the same process (default route and the cuFFT route,
EMAGLS_RENDER_FUSED=0), and the FFT sizes in --fft-sizes are timed on the natural track (EMAGLS_TRACK_FFT).
Correctness at the timed size: the tracked output against the same track composed from static renders (one
emagls_binaural_decode_dev per distinct page, mixed on the device with the contract's weights); the full signal for
the natural track, the first 30 s for the random one.

    python tools/bench_tracked_render.py --out profiles/r03_tracked_render.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS = 48000
HBM_PEAK = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU


def natural_track(frames, hop, pages):
    from emagls_b200 import synth
    pitches = np.array([round(float(np.degrees(np.arcsin(-R[2, 0])))) for R in synth.orientation_grid()[::360]])
    t = (np.arange(frames) + 0.5) * hop / FS
    yaw = 60 * np.sin(2 * np.pi * 0.5 * t) + 20 * np.sin(2 * np.pi * 0.13 * t)
    pitch = 20 * np.sin(2 * np.pi * 0.2 * t)
    row = np.abs(pitch[:, None] - pitches[None, :]).argmin(1)
    page = row * 360 + np.mod(np.rint(yaw).astype(np.int64), 360)
    assert page.max() < pages, "the natural track needs the full 3600-page grid"
    return page.astype(np.int32)


def pages_per_block(track, n, hop, fade, L):
    """(block, page) pairs of the render's pair table for blocks of L samples (tracked_render.cu, build_pairs)."""
    nblk = (n + L - 1) // L
    b = np.arange(nblk)
    t_lo, t_hi = b * L, np.minimum((b + 1) * L, n) - 1
    f_lo, f_hi = t_lo // hop, t_hi // hop
    cnt = f_hi - f_lo + 1
    blk = np.repeat(b, cnt)
    fr = np.repeat(f_lo, cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    pg = track[fr].astype(np.int64)
    fade_in = (f_lo > 0) & (fade > 0) & (f_lo * hop + fade - 1 >= t_lo)
    blk = np.concatenate([blk, b[fade_in]])
    pg = np.concatenate([pg, track[f_lo[fade_in] - 1].astype(np.int64)])
    key = np.unique(blk * (int(track.max()) + 1) + pg)
    return np.bincount(key // (int(track.max()) + 1), minlength=nblk)


def modelled_bytes(per_block, ch, N):
    """HBM bytes of the cuFFT route (tracked_render.cu, modelled_bytes): channel spectra per block; per pair the
    filter spectra (2 ch F complex), two ear spectra and two time signals, each written and read once."""
    F = N // 2 + 1
    return per_block.size * ch * F * 16 + per_block.sum() * (2 * ch * F * 16 + 4 * F * 16 + 4 * N * 8)


def chosen_fft(track, n, hop, fade, ch, taps):
    """The FFT size the render picks by default: the candidate with the fewest modelled bytes."""
    ov = (taps + 1) & ~1
    nmin = 16
    while nmin < 2 * taps:
        nmin <<= 1
    best, best_b = nmin, modelled_bytes(pages_per_block(track, n, hop, fade, nmin - ov), ch, nmin)
    nc = 2 * nmin
    while nc <= 4 * nmin and nc // 2 - ov < n:
        b = modelled_bytes(pages_per_block(track, n, hop, fade, nc - ov), ch, nc)
        if b < best_b:
            best, best_b = nc, b
        nc <<= 1
    return best


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, pl, clk = (q.stdout.strip().splitlines()[0].split(", ") + ["", "", ""])[:3] if q.returncode == 0 else ("", "", "")
    import torch
    return dict(name=name or torch.cuda.get_device_name(0), power_limit_w=float(pl) if pl else None,
                max_sm_clock_mhz=float(clk) if clk else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--pages", type=int, default=3600)
    ap.add_argument("--taps", type=int, default=512)
    ap.add_argument("--ch", type=int, default=32)
    ap.add_argument("--hop", type=int, default=480)
    ap.add_argument("--fft-sizes", default="1024,2048,4096")
    ap.add_argument("--check-seconds", type=float, default=30.0, help="composed-static check length, random track")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()

    import torch
    import emagls_b200 as em
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the tracked render has no CPU path")
    dev = torch.device("cuda", 0)
    h = em.Handle(0)
    st = torch.cuda.ExternalStream(h.stream, device=dev)
    n, ch, ln, P, hop = int(a.seconds * FS), a.ch, a.taps, a.pages, a.hop
    fade = hop
    g = torch.Generator(device=dev).manual_seed(a.seed)
    # bank [len, ch, P] column-major == [P, ch, len] row-major; signal [n, ch] column-major == [ch, n] row-major
    wL = torch.randn((P, ch, ln), generator=g, dtype=torch.float64, device=dev) / ln
    wR = torch.randn((P, ch, ln), generator=g, dtype=torch.float64, device=dev) / ln
    x = torch.randn((ch, n), generator=g, dtype=torch.float64, device=dev)
    out = torch.empty((2, n), dtype=torch.float64, device=dev)
    frames = (n - 1) // hop + 1
    rng = np.random.default_rng(a.seed)
    tracks = {
        "static_head": np.full(frames, min(5 * 360, P - 1), np.int32),
        "natural": natural_track(frames, hop, P) if P >= 3600 else rng.integers(0, P, frames).astype(np.int32),
        "worst_case": rng.integers(0, P, frames).astype(np.int32),
    }

    torch.cuda.synchronize()            # the tensors above were filled on torch's stream; the library uses the handle's

    def tracked(trk, nn=n, y=out, xx=x):
        h.check(h.lib.emagls_binaural_decode_tracked_dev(h.ptr, xx.data_ptr(), nn, ch, wL.data_ptr(), wR.data_ptr(), ln,
                                                         P, trk.ctypes.data_as(C.c_void_p), trk.size, hop, fade, 0, 0,
                                                         y.data_ptr()))

    def static(page, nn=n, y=out, xx=x):
        h.check(h.lib.emagls_binaural_decode_dev(h.ptr, xx.data_ptr(), nn, ch, wL[page].data_ptr(), wR[page].data_ptr(),
                                                 ln, 0, y.data_ptr()))

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

    def composed(trk, nn):
        """The contract built from static renders: sum over pages p of w_p(n) * y_p(n)."""
        t = torch.arange(nn, device=dev, dtype=torch.int64)
        f = t // hop
        i = t - f * hop
        td = torch.from_numpy(trk.astype(np.int64)).to(dev)
        c, aa = td[f], td[torch.clamp(f - 1, min=0)]
        gg = torch.where(i < fade, (i.double() + 0.5) / max(fade, 1), torch.ones_like(i, dtype=torch.float64))
        gg = torch.where(aa == c, torch.ones_like(gg), gg)
        xx = x[:, :nn].contiguous()     # [nn, ch] column-major: channel stride nn
        ref = torch.zeros((2, nn), dtype=torch.float64, device=dev)
        ys = torch.empty((2, nn), dtype=torch.float64, device=dev)
        yt = torch.empty((2, nn), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        used = np.unique(np.concatenate([trk[:(nn - 1) // hop + 1], trk[:max((nn - 1) // hop, 0)]]))
        for p in used.tolist():
            with torch.cuda.stream(st):
                static(p, nn, ys, xx)
                w = torch.where(c == p, gg, 0.0) + torch.where(aa == p, 1.0 - gg, 0.0)
                ref += w * ys
        tracked(trk[:(nn - 1) // hop + 1], nn, yt, xx)
        st.synchronize()
        return float(((yt - ref).abs().max() / ref.abs().max()).item()), len(used)

    res = dict(device=device_info(), config=dict(seconds=a.seconds, samples=n, channels=ch, taps=ln, pages=P, hop=hop,
                                                  fade=fade, fs=FS, seed=a.seed, bank_bytes=2 * P * ch * ln * 8),
               tracks={}, static_render={}, fft_sizes_natural={})
    for name, trk in tracks.items():
        N = chosen_fft(trk, n, hop, fade, ch, ln)
        ppb = pages_per_block(trk, n, hop, fade, N - ((ln + 1) & ~1))
        ms = timed(lambda: tracked(trk))
        distinct = int(np.unique(trk).size)
        F = N // 2 + 1
        # algorithmic: input read once, output written once, every referenced page's filters read once
        alg = ch * n * 8 + 2 * n * 8 + distinct * 2 * ch * ln * 8
        model = float(modelled_bytes(ppb, ch, N)) + ch * n * 8 + 2 * n * 8
        r = dict(fft_size=N, ms_per_call=round(ms, 3), msamples_per_s=round(n / ms / 1e3, 1),
                 blocks=int(ppb.size), pages_per_block_mean=round(float(ppb.mean()), 3),
                 pages_per_block_max=int(ppb.max()), distinct_pages=distinct,
                 hbm_bytes_algorithmic=int(alg), hbm_fraction_algorithmic=round(alg / (ms * 1e-3) / HBM_PEAK, 4),
                 hbm_bytes_modelled=int(model), hbm_fraction_modelled=round(model / (ms * 1e-3) / HBM_PEAK, 4),
                 filter_spectrum_bytes_per_pair=2 * ch * F * 16)
        r["profile_ms"] = profiled(lambda: tracked(trk))
        res["tracks"][name] = r
        print(name, json.dumps(r), flush=True)
    for N in [int(v) for v in a.fft_sizes.split(",") if v]:
        os.environ["EMAGLS_TRACK_FFT"] = str(N)
        ms = timed(lambda: tracked(tracks["natural"]))
        ppb = pages_per_block(tracks["natural"], n, hop, fade, N - ((ln + 1) & ~1))
        res["fft_sizes_natural"][str(N)] = dict(ms_per_call=round(ms, 3), pages_per_block_mean=round(float(ppb.mean()), 3),
                                                hbm_bytes_modelled=int(modelled_bytes(ppb, ch, N)))
        print("natural N =", N, res["fft_sizes_natural"][str(N)], flush=True)
    os.environ.pop("EMAGLS_TRACK_FFT", None)
    for key, env in (("default", None), ("cufft", "0")):
        if env is not None:
            os.environ["EMAGLS_RENDER_FUSED"] = env
        res["static_render"][key] = dict(ms_per_call=round(timed(lambda: static(0)), 3),
                                         profile_ms=profiled(lambda: static(0)))
        os.environ.pop("EMAGLS_RENDER_FUSED", None)
        print("static", key, res["static_render"][key], flush=True)
    for name, nn in (("natural", n), ("worst_case", min(n, int(a.check_seconds * FS)))):
        err, used = composed(tracks[name], nn)
        res["tracks"][name]["max_rel_diff_vs_composed_static"] = err
        res["tracks"][name]["composed_check"] = dict(samples=nn, static_renders=used)
        print(name, "composed-static check", err, "over", nn, "samples,", used, "static renders", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    ok = all(res["tracks"][k]["max_rel_diff_vs_composed_static"] < 1e-9 for k in ("natural", "worst_case"))
    print(json.dumps(dict(out=a.out, ok=ok)))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
