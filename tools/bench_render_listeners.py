"""Render sessions for many listeners (emagls_render_stream_create_listeners / _create_sh_listeners) on one GPU; writes
one JSON file to --out.

Workloads, at 48 kHz, hop 480 (a 100 Hz tracker) and fade = hop, every listener hearing the same input:
  bank   the seeded random em32 bank of 3600 pages x 512 taps, blocks --blocks, L in --listeners; listener l follows the
         natural head motion of tools/bench_render_stream.py with a seeded phase and amplitude of its own, snapped to
         the 3600-orientation page grid (synth.orientation_grid());
  sh<N>  SH sessions of orders --orders (512 taps), block --sh-block, L in --sh-listeners, on the same head motions,
         unsnapped.
For each workload:
  device_ms_per_block  CUDA events on the handle's stream around single-block calls of the _dev variant (mean);
  launches_per_block   kernel launches per block (emagls_launch_count);
  distinct_pages_*     pages the bank session's blocks render (the union over the listeners; mean and max);
  latency_ms_*         host clock around single-block calls of the host variant (median, p99);
  session_bytes        device bytes the session allocates (counted from the sizes of its buffers; the pinned host
                       staging is session_pinned_bytes);
  realtime_listeners   L x block duration / device time per block: how many listeners one GPU keeps in real time;
  max_rel_diff         largest relative difference (max-norm) of three listeners' outputs of the _dev calls against the
                       whole-signal render of the same input and entries.
separate_vs_shared: --compare-listeners one-listener bank sessions against one session of that many listeners, at the
first block: the summed device time per block (events around the calls of all sessions for one block) and memory.

    python tools/bench_render_listeners.py --out profiles/r08_render_listeners.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

FS = 48000
GRID_PITCHES = np.array([-45, -35, -25, -15, -5, 5, 15, 25, 35, 45])   # synth.orientation_grid(): 10 rows of 360 yaws


def head_motion(frames, hop, L, rng):
    """[frames, L] yaw and pitch (degrees): bench_render_stream.py's head motion with per-listener phases and an
    amplitude in [0.5, 1.5]"""
    t = ((np.arange(frames) + 0.5) * hop / FS)[:, None]
    ph = rng.uniform(0, 2 * np.pi, (3, L))
    amp = rng.uniform(0.5, 1.5, L)
    yaw = amp * (60 * np.sin(2 * np.pi * 0.5 * t + ph[0]) + 20 * np.sin(2 * np.pi * 0.13 * t + ph[1]))
    pitch = amp * 20 * np.sin(2 * np.pi * 0.2 * t + ph[2])
    return yaw, pitch


def bank_tracks(yaw, pitch, pages):
    if pages >= 3600:
        row = np.abs(pitch[:, :, None] - GRID_PITCHES).argmin(2)
        return (row * 360 + np.mod(np.rint(yaw).astype(np.int64), 360)).astype(np.int32)
    return np.mod(np.rint(yaw).astype(np.int64), pages).astype(np.int32)   # tiny runs: the yaw alone, folded


def rotations(yaw, pitch):
    """[frames, L, 3, 3] = synth.rotation_yaw_pitch for every entry, vectorised"""
    a, b = np.radians(yaw), np.radians(pitch)
    ca, sa, cb, sb = np.cos(a), np.sin(a), np.cos(b), np.sin(b)
    z = np.zeros_like(a)
    return np.stack([ca * cb, -sa, ca * sb, sa * cb, ca, sa * sb, -sb, z, cb], -1).reshape(*a.shape, 3, 3)


def union_sizes(track, nblk, B, hop, fade):
    """Distinct pages per block of a bank session (the rule of run_chunk in stream_render.cu)"""
    out = []
    for b in range(nblk):
        t_lo, t_hi = b * B, b * B + B - 1
        f0, f1 = t_lo // hop, t_hi // hop
        parts = [track[f0:f1 + 1].ravel()]
        for f in range(f0, f1 + 1):
            if f > 0 and fade > 0 and f * hop + fade - 1 >= t_lo:
                parts.append(track[f - 1])
        out.append(len(np.unique(np.concatenate(parts))))
    return np.array(out)


def session_bytes(kind, L, ch, pages, ln, B, hop, order=0):
    """(device, pinned) bytes of a session: the buffers create_session in stream_render.cu allocates"""
    N, F, P = 2 * B, B + 1, -(-ln // B)
    cb = max(1, 16384 // (B * L))
    fr_blk = (B - 1) // hop + 2
    nfr_blk, nfr_chunk = fr_blk + 1, (cb * B - 1) // hop + 3
    pmax = min(pages, fr_blk + 1) if kind == "bank" else 1
    if kind == "bank":
        pcap = 1
        while pcap < min(pages, L * pmax):
            pcap <<= 1
    else:
        pcap = L if kind == "sh" else 1
    xch = L * ch if kind == "sh" else ch
    dev = 16 * (pages * 2 * ch * P * F + P * xch * F + pcap * 2 * F) + 8 * (xch * N + xch * B + pcap * 2 * N)
    dev += 8 * (ch * cb * B + 2 * L * cb * B) + 4
    tab = cb * (2 * L * fr_blk + min(pages, L * pmax)) if kind == "bank" else 1
    dev += 4 * tab
    pinned = 8 * (ch * cb * B + 2 * L * cb * B) + 4 * tab
    if kind == "sh":
        blk = (order + 1) * (4 * (order + 1) ** 2 - 1) // 3
        dev += 8 * (L * nfr_chunk * 9 + L * nfr_blk * blk + xch * B) + 4 * L * nfr_blk
        pinned += 8 * L * nfr_chunk * 9
    return dev, pinned      # plus the cuFFT work area of the per-block plans


def device_info():
    from bench_tracked_render import device_info as info
    return info()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", default="512,128")
    ap.add_argument("--listeners", default="1,8,64,512,4096")
    ap.add_argument("--sh-listeners", default="1,8,64,512")
    ap.add_argument("--sh-block", type=int, default=512)
    ap.add_argument("--orders", default="4,7")
    ap.add_argument("--pages", type=int, default=3600)
    ap.add_argument("--taps", type=int, default=512)
    ap.add_argument("--ch", type=int, default=32)
    ap.add_argument("--hop", type=int, default=480)
    ap.add_argument("--calls", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--dev-calls", type=int, default=200)
    ap.add_argument("--compare-listeners", type=int, default=8)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--tiny", action="store_true", help="a seconds-long smoke run of every code path")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if a.tiny:
        a.blocks, a.listeners, a.sh_listeners, a.sh_block, a.orders = "128", "1,3", "1,3", 128, "1"
        a.pages, a.taps, a.ch, a.calls, a.warmup, a.dev_calls, a.compare_listeners = 16, 64, 4, 20, 3, 10, 3

    import torch
    import emagls_b200 as em
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the render sessions have no CPU path")
    dev = torch.device("cuda", 0)
    h = em.Handle(0)
    lib = h.lib
    st = torch.cuda.ExternalStream(h.stream, device=dev)
    rng = np.random.default_rng(a.seed)
    hop, fade, ln = a.hop, a.hop, a.taps
    p = lambda arr: arr.ctypes.data_as(C.c_void_p)   # noqa: E731
    vp = lambda t: C.c_void_p(t.data_ptr())          # noqa: E731
    n_calls = a.warmup + a.calls + a.dev_calls

    def create(kind, wL, wR, ch, pages, L, B, order):
        s = C.c_void_p()
        if kind == "sh":
            h.check(lib.emagls_render_stream_create_sh_listeners(h.ptr, p(wL), p(wR), ln, order, L, B, hop, fade,
                                                                 C.byref(s)))
        else:
            h.check(lib.emagls_render_stream_create_listeners(h.ptr, p(wL), p(wR), ln, ch, pages, L, B, hop, fade,
                                                              C.byref(s)))
        return s

    def entries(kind, E, t, n, given):
        """(track, rotations, count, new total, keep-alive) of the entries a call over [t, t + n) appends"""
        need = (t + n - 1) // hop + 1
        k = max(need - given, 0)
        new = np.ascontiguousarray(np.swapaxes(E[given:given + k], 0, 1))   # listener-major
        ptr = p(new)
        return (ptr, None, k, given + k, new) if kind == "bank" else (None, ptr, k, given + k, new)

    def dev_block_ms(sessions, xd, B, state):
        """mean device time of one block through every session in `sessions` (events around all their calls)"""
        ods = [torch.empty((2 * L_, B), dtype=torch.float64, device=dev) for (_, _, _, L_) in sessions]
        dms, outs = [], []
        t0 = state["t"]
        for c in range(xd.shape[1] // B):
            xc = xd[:, c * B:(c + 1) * B].contiguous()
            args = []                               # built before the first event: only the calls are timed
            for i, (s, kind, E, _) in enumerate(sessions):
                trk, rot, k, state["given"][i], keep = entries(kind, E, t0 + c * B, B, state["given"][i])
                args.append((s, trk, rot, k, keep))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for i, (s, trk, rot, k, _) in enumerate(args):
                h.check(lib.emagls_render_stream_process_dev(s, vp(xc), B, trk, rot, k, vp(ods[i])))
            e1.record(st)
            e1.synchronize()
            dms.append(e0.elapsed_time(e1))
            outs.append(ods[0].cpu().numpy())
        state["t"] = t0 + xd.shape[1]
        return float(np.mean(dms)), np.concatenate(outs, 1)

    results = []
    plan = [("bank", a.ch, a.pages, None, B, L) for B in (int(b) for b in a.blocks.split(","))
            for L in (int(x) for x in a.listeners.split(","))]
    plan += [(f"sh{o}", (o + 1) ** 2, 1, o, a.sh_block, L) for o in (int(x) for x in a.orders.split(","))
             for L in (int(x) for x in a.sh_listeners.split(","))]
    filters = {}
    for name, ch, pages, order, B, L in plan:
        kind = "sh" if order is not None else "bank"
        if name not in filters:
            frng = np.random.default_rng(a.seed + len(name) + ch)
            filters[name] = (np.asfortranarray(frng.standard_normal((ln, ch, pages)) / ln),
                             np.asfortranarray(frng.standard_normal((ln, ch, pages)) / ln))
        wL, wR = filters[name]
        n = n_calls * B
        frames = (n - 1) // hop + 2
        yaw, pitch = head_motion(frames, hop, L, np.random.default_rng(a.seed + 1))
        E = bank_tracks(yaw, pitch, pages) if kind == "bank" else rotations(yaw, pitch)
        x = rng.standard_normal((ch, n))            # [ch][n]: column-major [n x ch]
        t0 = time.perf_counter()
        s = create(kind, wL, wR, ch, pages, L, B, order)
        create_ms = (time.perf_counter() - t0) * 1e3
        # host variant: one block per call
        lat, given, l0 = [], 0, h.launches
        out = np.zeros((B, 2, L), order="F")
        for c in range(a.warmup + a.calls):
            trk, rot, k, given, keep = entries(kind, E, c * B, B, given)
            xc = np.asfortranarray(x[:, c * B:(c + 1) * B].T)
            t1 = time.perf_counter()
            rc = lib.emagls_render_stream_process(s, p(xc), B, trk, rot, k, p(out))
            t2 = time.perf_counter()
            h.check(rc)
            if c >= a.warmup:
                lat.append((t2 - t1) * 1e3)
        launches = (h.launches - l0) / (a.warmup + a.calls)
        # _dev variant, and the accuracy of its output
        t_dev = (a.warmup + a.calls) * B
        xd = torch.from_numpy(np.ascontiguousarray(x[:, t_dev:])).to(dev)
        state = {"t": t_dev, "given": [given]}
        dms, y_dev = dev_block_ms([(s, kind, E, L)], xd, B, state)
        h.check(lib.emagls_render_stream_destroy(s))
        xw = np.ascontiguousarray(x.T)
        diff = 0.0
        for l in sorted({0, L // 2, L - 1}):
            if kind == "bank":
                yw = em.binauralDecodeTracked(xw, wL, wR, E[:, l], hop, fade, handle=h)
            else:
                yw = em.binauralDecodeShTracked(xw, wL[:, :, 0], wR[:, :, 0], E[:, l], hop, fade, handle=h)
            yl = y_dev[2 * l:2 * l + 2].T
            ref = yw[t_dev:]
            diff = max(diff, float(np.abs(yl - ref).max() / np.abs(ref).max()))
        lat = np.array(lat)
        dev_b, pin_b = session_bytes(kind, L, ch, pages, ln, B, hop, order or 0)
        r = dict(workload=name, listeners=L, channels=ch, pages=pages, taps=ln, hop=hop, fade=fade, block=B,
                 create_ms=create_ms, device_ms_per_block=dms, launches_per_block=launches,
                 latency_ms_median=float(np.median(lat)), latency_ms_p99=float(np.percentile(lat, 99)),
                 block_ms=B / FS * 1e3, realtime_listeners=L * (B / FS * 1e3) / dms,
                 session_bytes=dev_b, session_pinned_bytes=pin_b, max_rel_diff=diff)
        if kind == "bank":
            u = union_sizes(E, n // B, B, hop, fade)
            r.update(distinct_pages_mean=float(u.mean()), distinct_pages_max=int(u.max()))
        else:
            r.update(distinct_pages_mean=1.0, distinct_pages_max=1)
        print(json.dumps(r), flush=True)
        results.append(r)
        del xd
        torch.cuda.empty_cache()

    # L separate one-listener sessions against one L-listener session, first block, bank
    L, B = a.compare_listeners, int(a.blocks.split(",")[0])
    wL, wR = filters["bank"]
    n = (a.warmup + a.dev_calls) * B
    yaw, pitch = head_motion((n - 1) // hop + 2, hop, L, np.random.default_rng(a.seed + 1))
    E = bank_tracks(yaw, pitch, a.pages)
    xd = torch.from_numpy(rng.standard_normal((a.ch, n))).to(dev)
    cmp = dict(listeners=L, block=B)
    for label, sessions in (("separate", [(create("bank", wL, wR, a.ch, a.pages, 1, B, None), "bank",
                                           E[:, l:l + 1], 1) for l in range(L)]),
                            ("shared", [(create("bank", wL, wR, a.ch, a.pages, L, B, None), "bank", E, L)])):
        state = {"t": 0, "given": [0] * len(sessions)}
        dev_block_ms(sessions, xd[:, :a.warmup * B], B, state)
        ms, _ = dev_block_ms(sessions, xd[:, a.warmup * B:], B, state)
        for s, *_ in sessions:
            h.check(lib.emagls_render_stream_destroy(s))
        nl = 1 if label == "separate" else L
        cmp[f"{label}_device_ms_per_block"] = ms
        cmp[f"{label}_session_bytes"] = len(sessions) * session_bytes("bank", nl, a.ch, a.pages, ln, B, hop)[0]
    print(json.dumps(cmp), flush=True)

    info = device_info()
    doc = dict(device=info["name"], power_limit_w=info["power_limit_w"], max_sm_clock_mhz=info["max_sm_clock_mhz"],
               fs=FS, tiny=bool(a.tiny), workloads=results, separate_vs_shared=cmp)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
