"""Latency and throughput of the render sessions (emagls_render_stream_*) on one GPU; writes one JSON file to --out.

Workloads, at 48 kHz, hop 480 (a 100 Hz tracker) and fade = hop: the seeded random em32 bank of 3600 pages x 512 taps
on the natural head motion of tools/bench_tracked_render.py (page grid: synth.orientation_grid()); SH sessions of
orders 4 and 7 (512 taps) on the same head motion, unsnapped; a static 32-channel session (512 taps).  For each
workload and each block in --blocks:
  create_ms          host clock around emagls_render_stream_create (uploads the filters, builds every spectrum);
  latency_ms_*       host clock around --calls warmed calls of the host variant, one block each, with the tracker
                     entries each call needs appended by that call (median, p99, max);
  device_ms_per_block CUDA events on the handle's stream around single-block calls of the _dev variant (mean);
  launches_per_block kernel launches per block (emagls_launch_count);
  realtime_factor    block duration / p99 latency;
  stream_ms, whole_ms, stream_over_whole: --stream-seconds of signal in device memory streamed block by block
                     through the _dev variant (host clock to the last synchronise) against the whole-signal _dev render
                     of the same data;
  max_rel_diff       largest relative difference between those two outputs (max-norm).

    python tools/bench_render_stream.py --out profiles/r05_render_stream.json
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


def head_motion(frames, hop):
    """Yaw and pitch (degrees) of the natural head motion of bench_tracked_render.py at the frame centres."""
    t = (np.arange(frames) + 0.5) * hop / FS
    yaw = 60 * np.sin(2 * np.pi * 0.5 * t) + 20 * np.sin(2 * np.pi * 0.13 * t)
    pitch = 20 * np.sin(2 * np.pi * 0.2 * t)
    return yaw, pitch


def rotations(frames, hop):
    from emagls_b200 import synth
    yaw, pitch = head_motion(frames, hop)
    return np.stack([synth.rotation_yaw_pitch(y, p) for y, p in zip(yaw, pitch)])


def bank_track(frames, hop, pages):
    if pages >= 3600:
        from bench_tracked_render import natural_track
        return natural_track(frames, hop, pages)
    yaw, _ = head_motion(frames, hop)                  # tiny runs: the yaw alone, folded onto the bank
    return np.mod(np.rint(yaw).astype(np.int64), pages).astype(np.int32)


def device_info():
    from bench_tracked_render import device_info as info
    return info()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", default="128,256,512,1024")
    ap.add_argument("--pages", type=int, default=3600)
    ap.add_argument("--taps", type=int, default=512)
    ap.add_argument("--ch", type=int, default=32)
    ap.add_argument("--hop", type=int, default=480)
    ap.add_argument("--orders", default="4,7")
    ap.add_argument("--calls", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--dev-calls", type=int, default=500)
    ap.add_argument("--stream-seconds", type=float, default=60.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--tiny", action="store_true", help="a seconds-long smoke run of every code path")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if a.tiny:
        a.blocks, a.pages, a.taps, a.ch, a.orders = "128,480", 16, 64, 4, "1"
        a.calls, a.warmup, a.dev_calls, a.stream_seconds = 50, 5, 20, 0.5

    import torch
    import emagls_b200 as em
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the render sessions have no CPU path")
    dev = torch.device("cuda", 0)
    h = em.Handle(0)
    lib = h.lib
    st = torch.cuda.ExternalStream(h.stream, device=dev)
    rng = np.random.default_rng(a.seed)
    hop, fade, ln, ch = a.hop, a.hop, a.taps, a.ch
    blocks = [int(b) for b in a.blocks.split(",")]
    n_stream = int(a.stream_seconds * FS)
    max_calls = a.warmup + a.calls + a.dev_calls
    frames = (max(n_stream, max(blocks) * max_calls) - 1) // hop + 2

    workloads = [("bank", ch, a.pages, None), ("static", ch, 1, None)]
    workloads += [(f"sh{o}", (o + 1) ** 2, 1, o) for o in (int(x) for x in a.orders.split(","))]
    track = bank_track(frames, hop, a.pages)
    R = rotations(frames, hop)
    p = lambda arr: arr.ctypes.data_as(C.c_void_p)   # noqa: E731
    results = []
    for name, nch, pages, order in workloads:
        wL = np.asfortranarray(rng.standard_normal((ln, nch, pages)) / ln)
        wR = np.asfortranarray(rng.standard_normal((ln, nch, pages)) / ln)
        x_all = rng.standard_normal((nch, max(n_stream, max(blocks) * max_calls)))   # [ch][n]: column-major [n x ch]
        x_dev = torch.from_numpy(x_all[:, :n_stream].copy()).to(dev)
        kind = "sh" if order is not None else name
        # whole-signal reference on the device
        y_whole = torch.empty((2, n_stream), dtype=torch.float64, device=dev)
        d_wL = torch.from_numpy(np.ascontiguousarray(wL.transpose(2, 1, 0))).to(dev)
        d_wR = torch.from_numpy(np.ascontiguousarray(wR.transpose(2, 1, 0))).to(dev)
        vp = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
        d_R = torch.from_numpy(R.reshape(-1, 9).copy()).to(dev)
        nf_stream = (n_stream - 1) // hop + 1

        def whole():
            if kind == "bank":
                return lib.emagls_binaural_decode_tracked_dev(h.ptr, vp(x_dev), n_stream, nch, vp(d_wL), vp(d_wR), ln,
                                                              pages, p(track), nf_stream, hop, fade, 0, 0, vp(y_whole))
            if kind == "static":
                return lib.emagls_binaural_decode_dev(h.ptr, vp(x_dev), n_stream, nch, vp(d_wL), vp(d_wR), ln, 0,
                                                      vp(y_whole))
            return lib.emagls_binaural_decode_sh_tracked_dev(h.ptr, vp(x_dev), n_stream, order, vp(d_wL), vp(d_wR), ln,
                                                             vp(d_R), nf_stream, hop, fade, 0, 0, vp(y_whole))
        h.check(whole())
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(3):
            h.check(whole())
        torch.cuda.synchronize(dev)
        whole_ms = (time.perf_counter() - t0) / 3 * 1e3
        y_ref = y_whole.clone()

        for B in blocks:
            def create():
                s = C.c_void_p()
                if kind == "sh":
                    h.check(lib.emagls_render_stream_create_sh(h.ptr, p(wL), p(wR), ln, order, B, hop, fade,
                                                               C.byref(s)))
                else:
                    h.check(lib.emagls_render_stream_create(h.ptr, p(wL), p(wR), ln, nch, pages, B, hop, fade,
                                                            C.byref(s)))
                return s

            def entries(t, n, given):
                """(pointer, count) of the entries a call over [t, t + n) appends, and the new total."""
                need = (t + n - 1) // hop + 1
                k = max(need - given, 0)
                if kind == "bank":
                    return C.c_void_p(track.ctypes.data + 4 * given), None, k, given + k
                if kind == "sh":
                    return None, C.c_void_p(R.ctypes.data + 72 * given), k, given + k
                return None, None, 0, given

            t0 = time.perf_counter()
            s = create()
            create_ms = (time.perf_counter() - t0) * 1e3
            # host variant: one block per call, warmed
            xb = np.asfortranarray(x_all[:, :(a.warmup + a.calls) * B].T)
            out = np.zeros((B, 2), order="F")
            lat = []
            given = 0
            l0 = h.launches
            for c in range(a.warmup + a.calls):
                trk, rot, k, given = entries(c * B, B, given)
                xc = np.asfortranarray(xb[c * B:(c + 1) * B])
                t1 = time.perf_counter()
                rc = lib.emagls_render_stream_process(s, p(xc), B, trk, rot, k, p(out))
                t2 = time.perf_counter()
                h.check(rc)
                if c >= a.warmup:
                    lat.append((t2 - t1) * 1e3)
            launches = (h.launches - l0) / (a.warmup + a.calls)
            # _dev variant: events around single-block calls
            t_next = (a.warmup + a.calls) * B
            xd = torch.from_numpy(np.ascontiguousarray(x_all[:, t_next:t_next + a.dev_calls * B])).to(dev)
            od = torch.empty((2, B), dtype=torch.float64, device=dev)
            dms = []
            for c in range(a.dev_calls):
                trk, rot, k, given = entries(t_next + c * B, B, given)
                xc = xd[:, c * B:(c + 1) * B].contiguous()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                h.check(lib.emagls_render_stream_process_dev(s, vp(xc), B, trk, rot, k, vp(od)))
                e1.record(st)
                e1.synchronize()
                dms.append(e0.elapsed_time(e1))
            h.check(lib.emagls_render_stream_destroy(s))
            # the stream of --stream-seconds through the _dev variant, against the whole-signal render
            s = create()
            nb = n_stream // B
            y_s = torch.zeros((2, n_stream), dtype=torch.float64, device=dev)
            xs = [x_dev[:, i * B:(i + 1) * B].contiguous() for i in range(nb)]
            ys = [torch.empty((2, B), dtype=torch.float64, device=dev) for _ in range(nb)]
            torch.cuda.synchronize(dev)
            given = 0
            t0 = time.perf_counter()
            for i in range(nb):
                trk, rot, k, given = entries(i * B, B, given)
                h.check(lib.emagls_render_stream_process_dev(s, vp(xs[i]), B, trk, rot, k, vp(ys[i])))
            torch.cuda.synchronize(dev)
            stream_ms = (time.perf_counter() - t0) * 1e3
            h.check(lib.emagls_render_stream_destroy(s))
            for i in range(nb):
                y_s[:, i * B:(i + 1) * B] = ys[i]
            m = nb * B
            diff = float((y_s[:, :m] - y_ref[:, :m]).abs().max() / y_ref[:, :m].abs().max())
            lat = np.array(lat)
            p99 = float(np.percentile(lat, 99))
            r = dict(workload=name, channels=nch, pages=pages, taps=ln, hop=hop, fade=fade, block=B,
                     partitions=-(-ln // B), create_ms=create_ms, calls=len(lat),
                     latency_ms_median=float(np.median(lat)), latency_ms_p99=p99, latency_ms_max=float(lat.max()),
                     device_ms_per_block=float(np.mean(dms)), launches_per_block=launches,
                     block_ms=B / FS * 1e3, realtime_factor=(B / FS * 1e3) / p99,
                     stream_seconds=m / FS, stream_ms=stream_ms, whole_ms=whole_ms,
                     stream_over_whole=stream_ms / whole_ms, max_rel_diff=diff)
            print(json.dumps(r), flush=True)
            results.append(r)
        del x_dev, y_whole, d_wL, d_wR, y_ref
        torch.cuda.empty_cache()

    info = device_info()
    doc = dict(device=info["name"], power_limit_w=info["power_limit_w"], max_sm_clock_mhz=info["max_sm_clock_mhz"],
               fs=FS, tiny=bool(a.tiny), workloads=results)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
