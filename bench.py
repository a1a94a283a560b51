#!/usr/bin/env python
"""Benchmark of the eMagLS hot path on B200: eMagLS2 filter sets / s (em32, N=4, 512 taps).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the reference algorithm on host cores

A "step" designs one batch of head-orientation filter sets (BASELINE config 2: the 3600-orientation
head-tracking grid, one HRTF set per rank -> weak scaling, no data-path collective).  Rank 0 prints
ONE JSON line.  `value` is device-resident throughput (inputs already in HBM, CUDA events on the
library's stream, max over ranks); `e2e` goes through the public host API (pinned host buffers,
H2D + D2H inside the timed region, plus the NCCL gather of the banks onto rank 0 for N > 1).

`--dump-outputs DIR` writes what the last timed step designed on rank 0, so that two builds can be compared output
for output: DIR/wL.npy and DIR/wR.npy, float64 [orientation, microphone, tap], the filters of a fixed sample of
DUMP_SETS orientations of the batch (every orientation when the batch is that small; indices in ascending order,
drawn with seed DUMP_SEED).  The inputs are synthetic and seeded, so equal arguments give equal inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "emagls2_filter_sets_per_sec"
UNIT = "filter sets/s"
ORDER, LEN = 4, 512
# SURVEY.md 8(d): direct formulation, per filter set (512 bins): 22.3 GFLOP
ALGO_GFLOP_PER_SET = 22.3
# 128 filter-set pairs of 2 x 32 x 512 doubles: 32 MiB on disk
DUMP_SETS, DUMP_SEED = 128, 0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--orient", type=int, default=3600, help="orientations per rank per step")
    ap.add_argument("--render-seconds", type=float, default=600.0,
                    help="length of the rendered 32-channel signal (SURVEY.md 8-d: 10 min)")
    ap.add_argument("--no-render", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spot-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the filters the last timed step designed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def problem(rank: int, n_orient: int):
    from emagls_b200 import synth
    g = synth.load_grids()
    az, ze = g["hrirGridAziRad"], g["hrirGridZenRad"]
    # one HRTF set per rank (SURVEY.md 8-d: seed = 20261017 + set index, randomised head)
    rng = np.random.default_rng(20261017 + rank)
    a = 0.0875 if rank == 0 else float(rng.uniform(0.075, 0.10))
    ear = 90.0 if rank == 0 else float(rng.uniform(85.0, 100.0))
    hL, hR = synth.synth_hrirs(az, ze, head_radius=a, ear_azi_deg=ear, seed=20261017 + rank)
    R = synth.orientation_grid()
    if n_orient <= R.shape[0]:
        R = R[:: max(1, R.shape[0] // n_orient)][:n_orient]
    else:
        R = np.concatenate([R] * (n_orient // R.shape[0] + 1))[:n_orient]
    return dict(g=g, az=az, ze=ze, hL=hL, hR=hR, R=np.ascontiguousarray(R), r=g["micRadius"],
                maz=g["micGridAziRad"], mze=g["micGridZenRad"], fs=g["fs"])


class ClockSampler:
    """SM clock / power / throttle reasons during the timed region (B200_PROFILING.md recipe), sampled every 0.2 s
    through NVML (nvidia_ml_py) in a background thread; falls back to spawning nvidia-smi when NVML is not importable.
    NVML queries do not take the driver lock a whole `nvidia-smi` process start does, so they do not stall the
    kernel launches of the step being timed."""

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._dev = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self._nvml = None

    @staticmethod
    def _physical_index(index: int) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                return int(ids[index])
        return index

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def _sample_nvml(self):
        n, d = self._nvml, self._dev
        sm = n.nvmlDeviceGetClockInfo(d, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(d, n.NVML_CLOCK_SM)
        try:
            pw = n.nvmlDeviceGetPowerUsage(d) / 1000.0
        except Exception:
            pw = 0.0
        r = n.nvmlDeviceGetCurrentClocksEventReasons(d) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(d)
        def flag(suffix):
            bit = getattr(n, "nvmlClocksEventReason" + suffix, None) or getattr(n, "nvmlClocksThrottleReason" + suffix, 0)
            return "Active" if r & bit else "Not Active"
        return [str(sm), str(mx), f"{pw:.1f}", flag("HwSlowdown"), flag("HwThermalSlowdown"), flag("SwThermalSlowdown"),
                flag("SwPowerCap")]

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                    if out.returncode == 0 and out.stdout.strip():
                        self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "source": "nvml" if self._nvml is not None else "nvidia-smi"}


def cpu_port_round(pr, first, workers):
    """One round of the NumPy restatement on the host cores: `workers` filter sets (orientations
    first..first+workers-1) designed concurrently, one thread each with single-threaded BLAS/LAPACK
    inside (the per-bin 2702 x 32 SVDs do not scale inside one call; NumPy releases the GIL in
    BLAS/LAPACK).  Overrides the OMP_NUM_THREADS=1 torchrun exports.  Returns seconds."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    from threadpoolctl import threadpool_limits
    from emagls_b200 import synth

    def one(i):
        raz, rze = synth.rotate_grid(pr["az"], pr["ze"], pr["R"][i % len(pr["R"])])
        oracle.getEMagLs2Filters(pr["hL"], pr["hR"], raz, rze, pr["r"], pr["maz"], pr["mze"], ORDER, pr["fs"], LEN)

    t0 = time.perf_counter()
    with threadpool_limits(limits=1):
        with ThreadPoolExecutor(max_workers=workers) as ex:
            list(ex.map(one, range(first, first + workers)))
    return time.perf_counter() - t0


def cpu_workers():
    return max(1, min(os.cpu_count() or 1, 32))


def run_reference(args, rank, world):
    """The reference's own algorithm on the box's host cores.  The reference is MATLAB, which this
    image cannot run, so this is the NumPy restatement (oracle/), labelled kind = "port"."""
    if rank != 0:
        return
    pr = problem(0, args.orient)
    workers = cpu_workers()
    sample = (f"{workers} filter sets (orientations) of the 3600-orientation batch per step, one host thread each "
              f"({os.cpu_count()} logical cores)")
    for i in range(args.warmup):
        cpu_port_round(pr, i * workers, workers)
    dt = 0.0
    for i in range(args.steps):
        dt += cpu_port_round(pr, (args.warmup + i) * workers, workers)
    v = args.steps * workers / dt
    ncores = workers
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": "eMagLS2 em32 order 4, 512 taps, 2702-dir grid; bounded sample of the "
                                   "3600-orientation batch", "sample_sets_per_step": workers},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes as C
    import torch
    import emagls_b200 as em
    from emagls_b200 import dist as emdist

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    emdist.init("nccl")
    dev = torch.device("cuda", local_rank)
    h = em.Handle(local_rank)
    cfg = h.default_config()
    stream = torch.cuda.ExternalStream(h.stream, device=dev)
    pr = problem(rank, args.orient)
    B, M, D, T = args.orient, pr["maz"].size, pr["az"].size, pr["hL"].shape[0]

    def dt64(x):
        return torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64))).to(dev)

    # ---------------- device-resident inputs ([T, D] column-major == [D, T] row-major)
    d_hL, d_hR = dt64(pr["hL"].T), dt64(pr["hR"].T)
    d_az, d_ze, d_maz, d_mze, d_R = dt64(pr["az"]), dt64(pr["ze"]), dt64(pr["maz"]), dt64(pr["mze"]), dt64(pr["R"])
    d_wL = torch.empty((B, M, LEN), dtype=torch.float64, device=dev)   # [len, M, B] column-major
    d_wR = torch.empty_like(d_wL)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_dev():
        rc = h.lib.emagls_design_emagls2_dev(
            h.ptr, C.byref(cfg), d_hL.data_ptr(), d_hR.data_ptr(), T, D, d_az.data_ptr(), d_ze.data_ptr(),
            float(pr["r"]), d_maz.data_ptr(), d_mze.data_ptr(), M, ORDER, float(pr["fs"]), LEN, 1, B,
            d_R.data_ptr(), d_wL.data_ptr(), d_wR.data_ptr(), None)
        h.check(rc)

    def l2_flush():
        with torch.cuda.stream(stream):
            flush.fill_(1)

    for _ in range(max(args.warmup, 3)):
        l2_flush()
        step_dev()
    torch.cuda.synchronize()
    h.profile(True)
    h.profile_read()
    h.stats_read()
    launches0 = h.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    emdist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local_rank) as clk:
        for i in range(args.steps):
            l2_flush()
            ev[i][0].record(stream)
            step_dev()
            ev[i][1].record(stream)
        torch.cuda.synchronize()
    emdist.barrier()
    if args.dump_outputs and rank == 0:     # before the steps below write the banks again
        os.makedirs(args.dump_outputs, exist_ok=True)
        pick = np.sort(np.random.default_rng(DUMP_SEED).choice(B, size=min(B, DUMP_SETS), replace=False))
        pick = torch.from_numpy(pick).to(dev)
        for name, bank in (("wL", d_wL), ("wR", d_wR)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), bank.index_select(0, pick).cpu().numpy())
    ms_local = sum(a.elapsed_time(b) for a, b in ev)
    ms = emdist.max_over_ranks(ms_local, dev)
    prof = h.profile_read()
    h.profile(False)
    stats = h.stats_read()
    launches = h.launches - launches0
    value = world * B * args.steps / (ms * 1e-3)
    # secondary: what the profiler's event pairs (about two timing events per launch on the stream, inside the timed
    # region above) cost: the same step alternately without and with them, each timed on its own
    evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2 * args.steps)]
    torch.cuda.synchronize()
    for i in range(2 * args.steps):
        h.profile(bool(i & 1))
        l2_flush()
        evp[i][0].record(stream)
        step_dev()
        evp[i][1].record(stream)
    torch.cuda.synchronize()
    h.profile_read()
    h.profile(False)
    ms_unprofiled = sum(evp[i][0].elapsed_time(evp[i][1]) for i in range(0, 2 * args.steps, 2)) / args.steps
    ms_reprofiled = sum(evp[i][0].elapsed_time(evp[i][1]) for i in range(1, 2 * args.steps, 2)) / args.steps

    # ---------------- end to end (pinned host buffers -> H2D -> design -> NCCL gather of the banks into rank 0's
    # device bank -> D2H of every rank's shard), through the package's sharded designer (emagls_b200/dist.py).
    # Weak scaling: rank r holds HRTF set r and the whole orientation grid, so the job is world x B filter sets.
    sd = emdist.ShardedDesigner(h, pr["hL"], pr["hR"], pr["az"], pr["ze"], pr["r"], pr["maz"], pr["mze"], ORDER,
                                pr["fs"], LEN, np.tile(pr["R"].reshape(-1, 9), (world, 1)), config=cfg)
    assert sd.n_local == B
    h2d, d2h = sd.h2d_bytes, sd.d2h_bytes

    def timed_e2e(designer, nsteps):
        designer.step()
        designer.wait()
        emdist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(nsteps):
            designer.step()          # returns when the design is enqueued; the D2H + gather of this step run on the
        designer.wait()              # transfer stream while the next step is designed into the other bank buffer
        torch.cuda.synchronize()     # every host shard (and rank 0's gathered device banks) is complete here
        return emdist.max_over_ranks(time.perf_counter() - t0, dev)

    e2e_steps = args.steps
    e2e_s = timed_e2e(sd, e2e_steps)
    e2e_value = world * B * e2e_steps / e2e_s
    # the e2e path and the device-resident path must have produced the same banks (same inputs)
    e2e_same = float(max((sd.bank[0] - d_wL).abs().max() / d_wL.abs().max(),
                         (sd.bank[1] - d_wR).abs().max() / d_wR.abs().max()))
    # and, through the reference-facing host call of the C ABI (one call, host buffers in and out; N = 1 only)
    host_api = None
    if world == 1:
        wLh = np.zeros((LEN, M, B), order="F")
        wRh = np.zeros((LEN, M, B), order="F")
        t0 = time.perf_counter()
        em.getEMagLs2Filters(pr["hL"], pr["hR"], pr["az"], pr["ze"], pr["r"], pr["maz"], pr["mze"], ORDER, pr["fs"], LEN,
                             rotations=pr["R"], handle=h, out=(wLh, wRh))
        host_api = {"value": B / (time.perf_counter() - t0), "unit": UNIT, "steps": 1,
                    "call": "emagls_design_emagls2 (host pointers, pageable memory)"}
        del wLh, wRh
    del sd

    # ---------------- the north-star batch: 3600 orientations of ONE HRTF set in total, sharded over the ranks
    # (strong scaling: 3600 / world per GPU); time to solution for the whole bank on rank 0.
    strong = None
    if world > 1:
        pr0 = problem(0, args.orient)
        ss = emdist.ShardedDesigner(h, pr0["hL"], pr0["hR"], pr0["az"], pr0["ze"], pr0["r"], pr0["maz"], pr0["mze"],
                                    ORDER, pr0["fs"], LEN, pr0["R"], config=cfg)
        s_steps = args.steps
        s_s = timed_e2e(ss, s_steps)
        strong = {"orientations_total": int(ss.n_total), "orientations_per_gpu": int(ss.n_local),
                  "ms_per_batch": s_s / s_steps * 1e3, "value": ss.n_total * s_steps / s_s, "unit": UNIT,
                  "steps": s_steps, "scaling": "strong",
                  "includes": "H2D of the inputs, design, NCCL gather into rank 0's bank, D2H of every shard"}
        del ss

    # ---------------- parity spot check of the timed batch (outside the timed regions): three random orientations and the last one of the
    # bank the device-resident steps produced against the oracle (NumPy restatement of the reference), rank 0
    spot = None
    if rank == 0 and not args.no_spot_check:
        import oracle
        from concurrent.futures import ThreadPoolExecutor
        from emagls_b200 import synth
        rng = np.random.default_rng(12345)
        idx = sorted(int(i) for i in rng.choice(B, size=min(3, B), replace=False))
        if B - 1 not in idx:
            idx.append(B - 1)   # the end of the batch: the part the Jacobi launch cuts into bin ranges (launch_svdclip)

        def ref(i):
            raz, rze = synth.rotate_grid(pr["az"], pr["ze"], pr["R"][i])
            return oracle.getEMagLs2Filters(pr["hL"], pr["hR"], raz, rze, pr["r"], pr["maz"], pr["mze"], ORDER, pr["fs"], LEN)
        with ThreadPoolExecutor(max_workers=len(idx)) as ex:
            refs = list(ex.map(ref, idx))
        errs = []
        for i, (rl, rr) in zip(idx, refs):
            gl, gr = d_wL[i].cpu().numpy().T, d_wR[i].cpu().numpy().T       # [len, M]
            sc = max(np.abs(rl).max(), np.abs(rr).max())
            errs.append(float(max(np.abs(gl - rl).max(), np.abs(gr - rr).max()) / sc))
        spot = {"orientations": idx, "max_rel_err_vs_oracle": max(errs), "per_orientation": errs,
                "bound": 5e-9, "ok": bool(max(errs) <= 5e-9),
                "note": "whole-filter max-norm error relative to the oracle; 5e-9 is the floor of two FP64 "
                        "implementations on bins 1-7 (tests/test_gpu_design.py), north-star 1e-10 is per bin >= 16"}

    # ---------------- roofline of the dominant tensor kernel
    # The two direction-grid contractions run on the int8 tensor cores (tcgen05.mma kind::i8, FP64
    # accuracy through T = 6 error-free base-256 slices: T (T + 1) / 2 = 21 int8 GEMMs per product).  The roofline
    # counts the int8 operations the kernel EXECUTES against the int8 tensor peak; the FP64-equivalent
    # rate and the DGEMM (DMMA) peak of this GPU are reported next to it.
    S = (19 + 1) ** 2
    use_oz = os.environ.get("EMAGLS_GEMM", "") != "dmma"
    oz_T = int(os.environ.get("EMAGLS_OZAKI_SLICES", "6"))
    pairs = oz_T * (oz_T + 1) // 2
    KpS, KpD = (S + 31) // 32 * 32, (D + 31) // 32 * 32
    dgemm_peak = i8_peak = None
    i8_src = None
    if rank == 0:
        def best_ms(fn, n=5):
            fn()
            best = 1e9
            for _ in range(n):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            return best
        a = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
        b = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
        dgemm_peak = 2 * 8192 ** 3 / (best_ms(lambda: torch.matmul(a, b)) * 1e-3) / 1e12
        del a, b
        try:   # library int8 GEMM (cuBLASLt) as the measured int8 tensor peak
            ai = torch.randint(-64, 64, (8192, 8192), dtype=torch.int8, device=dev)
            bi = torch.randint(-64, 64, (8192, 8192), dtype=torch.int8, device=dev).t()
            i8_peak = 2 * 8192 ** 3 / (best_ms(lambda: torch._int_mm(ai, bi)) * 1e-3) / 1e12
            i8_src = "live torch._int_mm (cuBLASLt int8) 8192^3, best of 5"
            del ai, bi
        except Exception as ex:  # noqa: BLE001
            i8_peak = None
            i8_src = f"torch._int_mm unavailable ({type(ex).__name__})"
        try:
            mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            alt = 2.0 * float(mp["bf16_tflops"])
            if i8_peak is None or i8_peak < alt:
                i8_peak, i8_src = alt, ("2 x MEASURED_PEAKS.json bf16_tflops (burst): tcgen05 kind::i8 runs at twice "
                                        "the bf16 rate; " + (i8_src or ""))
        except Exception:
            if i8_peak is None:
                i8_peak, i8_src = 4500.0, "nominal dense int8 (B200_PROFILING.md fallback)"
    fp64_flops = {"gemm_fwd": 2.0 * D * 4 * B * S, "gemm_bwd": 2.0 * 4 * B * S * D}
    i8_ops = {"gemm_fwd": 2.0 * D * 4 * B * KpS * pairs, "gemm_bwd": 2.0 * 4 * B * S * KpD * pairs}
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    shares = {k: round(v["ms"] / tot_ms, 4) for k, v in prof.items() if v["n"]}
    dom = max(("gemm_fwd", "gemm_bwd"), key=lambda k: prof[k]["ms"])
    avg_ms = prof[dom]["ms"] / max(prof[dom]["n"], 1)
    fp64_equiv = fp64_flops[dom] / (avg_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_oz_traffic.json" if use_oz else "r01_gemm_traffic.json")))
        want = ("EpiPhase" if dom == "gemm_fwd" else "EpiStore")
        if B == 3600:
            traffic = next(x["traffic_bytes"] for x in tj["launches"] if want in x["kernel"])
            traffic_src = ("profiles/" + ("r02_oz_traffic.json" if use_oz else "r01_gemm_traffic.json") +
                           " (dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full launch)")
    except Exception:
        pass
    # ---------------- one roofline entry per kernel class of the step (work models: DESIGN.md section 5).
    # FP64 CUDA-core classes are measured against the live cuBLAS DGEMM figure (the FP64 pipe of this part;
    # MEASURED_PEAKS.json has no FP64 entry), HBM classes against MEASURED_PEAKS.json hbm_gbs.
    hbm_peak = 6650.0
    try:
        hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    st = stats            # (problem, bin) counts of the timed steps, from the library
    nblk = (S + 31) // 32
    per_step = lambda k: prof[k]["ms"] / args.steps if prof.get(k, {}).get("n") else None   # noqa: E731
    classes = {}

    def add(name, kernel, bound, work, unit_scale, peak, unit, note):
        ms_c = per_step(name)
        if not ms_c or not work:
            return
        ach = work / (ms_c * 1e-3) / unit_scale
        classes[name] = {"kernel": kernel, "ms_per_step": ms_c, "share": shares.get(name), "bound": bound,
                         "achieved": ach, "peak": peak, "unit": unit, "frac": (ach / peak) if peak else None, "note": note}
    tsqr_pb = st["tsqr_problem_bins"] / args.steps
    gram_pb = st["gram_problem_bins"] / args.steps
    jac_p = st["jacobi_problems"] / args.steps
    jac_sw = st["jacobi_sweeps"] / args.steps
    new_path = bool(prof.get("jacobi", {}).get("n"))
    if new_path:
        add("factor", "tsqr_sep_kernel (register-resident Householder TSQR, warp per (orientation, bin))", "fp64",
            8.0 * (S * M * M - M ** 3 / 3.0) * tsqr_pb, 1e12, dgemm_peak, "TFLOP/s (FP64, algorithmic)",
            f"8 (S M^2 - M^3/3) flops x {tsqr_pb:.0f} (orientation, bin) problems per step (algorithmic: all {nblk} row "
            f"blocks); the kernel skips row blocks whose modal coefficients are below 2^-60 of the largest and folds the "
            f"last 16 Householder steps of a block onto all 32 lanes (12 k instead of 16 k FP64 lane-FMAs per block)")
        add("jacobi", "svdclip_kernel (one-sided Jacobi, block round-robin, warm starts)", "fp64",
            1800.0 * M * (M - 1) / 2 * jac_sw + 8.0 * M ** 3 * jac_p, 1e12, dgemm_peak, "TFLOP/s (FP64, algorithmic)",
            f"1800 flops per rotated column pair x M (M - 1) / 2 pairs x {jac_sw / max(jac_p, 1):.2f} sweeps (measured mean) "
            f"+ 8 M^3 for the projector, {jac_p:.0f} problems per step")
    else:
        add("factor", "factor_kernel (shared-memory TSQR + one-sided Jacobi, round-1 kernel)", "fp64",
            (8.0 * (S * M * M - M ** 3 / 3.0) + 8 * 1800.0 * M * (M - 1) / 2 + 8.0 * M ** 3) * tsqr_pb, 1e12, dgemm_peak,
            "TFLOP/s (FP64, algorithmic)", "QR + 8 Jacobi sweeps + projector per (orientation, bin) problem")
    if use_oz:
        for nm, lab in (("gemm_fwd", "forward y = Y_h c with fused phase continuation + digit slicing"),
                        ("gemm_bwd", "backward t Y_h / t Q")):
            n_l = max(prof[nm]["n"], 1) / args.steps
            add(nm, f"ozaki_gemm_kernel<{oz_T}> ({lab}; tcgen05.mma kind::i8, TMEM accumulators, TMA operands)", "tensor",
                i8_ops[nm] * n_l, 1e12, i8_peak, "TOP/s (int8, executed)",
                f"{pairs} digit products per FP64 product; FP64-equivalent "
                f"{fp64_flops[nm] * n_l / (per_step(nm) * 1e-3) / 1e12:.1f} TFLOP/s")
    else:
        for nm in ("gemm_fwd", "gemm_bwd"):
            n_l = max(prof[nm]["n"], 1) / args.steps
            add(nm, "gemm_f64_kernel (DMMA.8x8x4)", "tensor", fp64_flops[nm] * n_l, 1e12, dgemm_peak, "TFLOP/s (FP64)", "")
    # backward small kernels: Gram bins read Y_o (Mc x S doubles), Pb, z, write digits; TSQR bins read the reflectors
    bytes_bwd = gram_pb * (M * S * 8 + M * M * 16 + 4 * S * 8 + oz_T * 4 * KpS) + tsqr_pb * (S * 32 * 16 + M * M * 16 + 4 * S * 8)
    add("chain_bwd", "bwd_fused_kernel (Gram bins: Y_o staged once in shared memory by cp.async.bulk) + chain_bwd_sep_kernel "
        "(TSQR bins: 32-row reflector tiles)", "hbm",
        bytes_bwd, 1e9, hbm_peak, "GB/s (algorithmic)", "operator bytes per (orientation, bin): Y_o 102 KB + Pb 16 KB + "
        "right-hand sides 13 KB + digits 10 KB (Gram route) or reflectors 205 KB + Pb 16 KB (TSQR route, all row blocks)")
    ne = M * (M + 1) // 2
    add("gram", "gemm_f64_kernel (DMMA assembly of G_k from the F blocks) + gram_sweep_kernel (in-register inversion)", "fp64",
        gram_pb * (2.0 * ne * S + 8.0 * M ** 3 / 2), 1e12, dgemm_peak, "TFLOP/s (FP64, algorithmic)",
        "2 ne S flops of assembly + 4 M^3 of Hermitian inversion per (orientation, bin)")
    dom_cls = max(classes, key=lambda k: classes[k]["ms_per_step"]) if classes else None
    if use_oz:
        achieved = i8_ops[dom] / (avg_ms * 1e-3) / 1e12
        gemm_roof = {"kernel": f"ozaki_gemm_kernel<{oz_T}> ({dom}: tcgen05.mma kind::i8, TMEM accumulators, TMA operands)",
                     "bound": "tensor", "achieved": achieved, "peak": i8_peak, "unit": "TOP/s (int8, executed)",
                     "frac": (achieved / i8_peak) if i8_peak else None, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": i8_src, "int8_ops_per_launch": i8_ops[dom], "slice_pairs": pairs,
                     "fp64_equivalent_tflops": fp64_equiv, "fp64_flops_per_launch": fp64_flops[dom],
                     "dgemm_peak_tflops": dgemm_peak,
                     "fp64_equivalent_vs_dgemm_peak": (fp64_equiv / dgemm_peak) if dgemm_peak else None, "avg_launch_ms": avg_ms}
    else:
        gemm_roof = {"kernel": f"gemm_f64_kernel ({dom}, DMMA.8x8x4)", "bound": "tensor", "achieved": fp64_equiv,
                     "peak": dgemm_peak, "unit": "TFLOP/s", "frac": (fp64_equiv / dgemm_peak) if dgemm_peak else None,
                     "traffic": traffic, "traffic_source": traffic_src, "flops_per_launch": fp64_flops[dom],
                     "avg_launch_ms": avg_ms}
    # headline roofline = the class that takes the largest share of the step; the tensor-core GEMM beside it
    if dom_cls in ("gemm_fwd", "gemm_bwd") or dom_cls is None:
        roofline = dict(gemm_roof)
    else:
        c = classes[dom_cls]
        roofline = {"kernel": c["kernel"], "bound": "tensor" if c["bound"] in ("tensor", "fp64") else "hbm",
                    "pipe": c["bound"], "achieved": c["achieved"], "peak": c["peak"], "unit": c["unit"], "frac": c["frac"],
                    "traffic": None, "note": c["note"], "ms_per_step": c["ms_per_step"], "share": c["share"]}
    roofline["peak_source"] = ("int8: " + str(i8_src) + "; FP64: live cuBLAS DGEMM 8192^3, best of 5 (MEASURED_PEAKS.json "
                               "has no FP64 entry); HBM: MEASURED_PEAKS.json hbm_gbs")
    roofline["dominant_class"] = dom_cls
    roofline["class_time_share"] = shares
    roofline["classes"] = classes
    roofline["tensor_gemm"] = gemm_roof
    roofline["algorithmic_tflops_whole_job"] = value / world * ALGO_GFLOP_PER_SET / 1e3
    roofline["jacobi_mean_sweeps"] = (jac_sw / jac_p) if jac_p else None
    roofline["profiler_cost_check"] = {"ms_per_step_without_events": round(ms_unprofiled, 3),
                                       "ms_per_step_with_events": round(ms_reprofiled, 3),
                                       "note": "alternating steps after the timed region, each timed on its own"}

    # ---------------- render (secondary metric: Msamples/s of the 32 -> 2 channel, 512-tap FIR)
    render = None
    if not args.no_render and rank == 0:
        n = int(args.render_seconds * 48000)
        x = torch.randn((32, n), dtype=torch.float64, device=dev)           # [n, 32] column-major
        y = torch.empty((2, n), dtype=torch.float64, device=dev)
        wl, wr = d_wL[0].contiguous(), d_wR[0].contiguous()                 # [M, LEN] == [len, M] col-major

        def rstep():
            h.check(h.lib.emagls_binaural_decode_dev(h.ptr, x.data_ptr(), n, 32, wl.data_ptr(), wr.data_ptr(), LEN, 0,
                                                     y.data_ptr()))
        for _ in range(2):
            rstep()
        torch.cuda.synchronize()
        h.profile(True)
        h.profile_read()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record(stream)
        for _ in range(3):
            rstep()
        r1.record(stream)
        torch.cuda.synchronize()
        rp = h.profile_read()
        h.profile(False)
        rms = r0.elapsed_time(r1) / 3
        hbm = None
        try:
            hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        except Exception:
            pass
        hbm = hbm or 6650.0
        algo_bytes = n * 272.0                                              # SURVEY.md 8(d): 272 B / frame
        render = {"metric": "render_msamples_per_sec", "value": n / (rms * 1e-3) / 1e6, "unit": "Msamples/s",
                  "frames": n, "channels": 32, "taps": LEN, "ms": rms,
                  "kernel": "fused_render16_kernel (overlap-save block per CTA: radix 16 x 16 x 8 Stockham passes in "
                            "registers / shared memory, multiply-accumulate over the channels, inverse transform; the "
                            "channel spectra never reach HBM)",
                  "roofline": {"bound": "hbm", "achieved": algo_bytes / (rms * 1e-3) / 1e9, "peak": hbm,
                               "unit": "GB/s", "frac": algo_bytes / (rms * 1e-3) / 1e9 / hbm,
                               "class_ms": {k: v["ms"] / 3 for k, v in rp.items() if v["n"]}}}
        del x, y

    # ---------------- render end to end: the 10-minute signal sharded by time blocks with a (taps - 1)-frame halo over
    # all ranks (SURVEY.md 8-e), pinned host blocks -> H2D -> decode -> D2H of the block's two output channels
    render_e2e = None
    if not args.no_render:
        n_all = int(args.render_seconds * 48000)
        r_lo, r_hi, r_halo = emdist.render_shard(n_all, LEN, rank, world)
        blk = np.random.default_rng(777 + rank).standard_normal((r_hi - r_lo + r_halo, 32))
        wl_h, wr_h = d_wL[0].cpu().numpy().T, d_wR[0].cpu().numpy().T          # [len, M]
        sr = emdist.ShardedRenderer(h, blk, wl_h, wr_h, r_halo)
        del blk
        sr.step(); sr.wait()
        emdist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            sr.step()
            sr.wait()
        r_s = emdist.max_over_ranks(time.perf_counter() - t0, dev) / 3
        render_e2e = {"value": n_all / r_s / 1e6, "unit": "Msamples/s", "ms": r_s * 1e3, "frames_total": n_all,
                      "frames_per_gpu": r_hi - r_lo, "halo_frames": LEN - 1, "h2d_bytes_per_step": sr.h2d_bytes * world,
                      "d2h_bytes_per_step": sr.d2h_bytes * world,
                      "path": "emagls_b200.dist.ShardedRenderer (time blocks, no exchange between ranks)"}
        del sr
        if render is not None:
            render["e2e"] = render_e2e

    # ---------------- BASELINE config 3 (secondary line): getEMagLsFiltersFromAtf on the measured glasses-on-HATS
    # ATF set (1625 directions x 8 microphones), batched over the 3600-orientation grid, + the 10-minute 8-channel
    # render that consumes one of the filter sets.  Rank 0, device-resident, CUDA events on the library's stream.
    config3 = None
    atf_path = os.path.join(ROOT, "tests", "golden", "atf_full.npz")
    if not args.no_render and rank == 0 and world == 1 and os.path.exists(atf_path):
        ad = np.load(atf_path)
        atf = np.ascontiguousarray(ad["atfIrs"].astype(np.float64).transpose(2, 1, 0))     # [Da, M, Ta] = col-major [Ta, M, Da]
        agd = np.deg2rad(ad["atfGridAziEleDeg"].astype(np.float64))
        ag = np.stack([agd[:, 0], np.pi / 2 - agd[:, 1]], 0)                               # [2, Da] = col-major [Da, 2]
        Da, M3, Ta = atf.shape
        L3 = 256
        d_atf, d_ag = dt64(atf), dt64(ag)
        d_hg = dt64(np.stack([pr["az"], pr["ze"]], 0))
        w3L = torch.empty((B, M3, L3), dtype=torch.float64, device=dev)
        w3R = torch.empty_like(w3L)

        def c3step():
            h.check(h.lib.emagls_design_from_atf_batch_dev(
                h.ptr, C.byref(cfg), d_hL.data_ptr(), d_hR.data_ptr(), T, D, d_hg.data_ptr(), d_atf.data_ptr(), Ta, M3, Da,
                d_ag.data_ptr(), float(pr["fs"]), L3, 2000.0, B, d_R.data_ptr(), w3L.data_ptr(), w3R.data_ptr(), None))
        for _ in range(2):
            c3step()
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(3):
            l2_flush()
            c3step()
        c1.record(stream)
        torch.cuda.synchronize()
        c3ms = c0.elapsed_time(c1) / 3
        n3 = int(args.render_seconds * 48000)
        x3 = torch.randn((M3, n3), dtype=torch.float64, device=dev)
        y3 = torch.empty((2, n3), dtype=torch.float64, device=dev)
        f3l, f3r = w3L[0].contiguous(), w3R[0].contiguous()

        def r3step():
            h.check(h.lib.emagls_binaural_decode_dev(h.ptr, x3.data_ptr(), n3, M3, f3l.data_ptr(), f3r.data_ptr(), L3, 0,
                                                     y3.data_ptr()))
        for _ in range(2):
            r3step()
        torch.cuda.synchronize()
        c0.record(stream)
        for _ in range(3):
            r3step()
        c1.record(stream)
        torch.cuda.synchronize()
        r3ms = c0.elapsed_time(c1) / 3
        config3 = {"workload": "BASELINE config 3: getEMagLsFiltersFromAtf, glasses-on-HATS ATFs (1625 x 8, 192 taps), "
                               "2702-direction HRIRs, filterLen 256, fTrans 2 kHz, 3600-orientation batch",
                   "filter_sets_per_sec": B / (c3ms * 1e-3), "ms_per_batch": c3ms, "orientations": B,
                   "render": {"frames": n3, "channels": M3, "taps": L3, "ms": r3ms,
                              "msamples_per_sec": n3 / (r3ms * 1e-3) / 1e6,
                              "hbm_frac": n3 * (M3 * 8 + 16.0) / (r3ms * 1e-3) / 1e9 / hbm_peak},
                   "data": "measured ATF set (float32 copy of the reference's resource, tests/golden/atf_full.npz), "
                           "synthetic rigid-sphere HRIRs"}
        del x3, y3, d_atf

    # ---------------- CPU baseline (the reference algorithm restated, on this box's host cores)
    cpu = None
    if not args.no_cpu_baseline and rank == 0 and world == 1:
        workers = cpu_workers()
        dtc = cpu_port_round(pr, 0, workers)
        cpu = {"value": workers / dtc, "unit": UNIT, "cores": workers, "kind": "port",
               "sample": f"{workers} of the {B} filter sets of one step, designed concurrently with one host thread each "
                         f"(NumPy restatement of the MATLAB reference; {os.cpu_count()} logical cores)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "BASELINE config 2: eMagLS2, em32 (32 mics, r=4.2 cm), SH order 4, 512 taps, "
                                       "2702-direction HRIR grid @48 kHz, head-orientation batch",
                           "orientations_per_gpu_per_step": B, "hrtf_sets_per_gpu": 1, "parallelism": f"shard{world}",
                           "l2": "flushed between steps (256 MiB write); per-step working set is several GB"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                        "steps": e2e_steps, "includes_nccl_gather": world > 1,
                        "path": "emagls_b200.dist.ShardedDesigner: pinned host inputs -> H2D -> emagls_design_emagls2_dev "
                                "-> D2H of every shard (pinned) and NCCL send/recv of the shards into rank 0's device bank on a "
                                "transfer stream, double-buffered banks: the transfers of step i overlap the design of step "
                                "i + 1; the timed region ends when the last step's transfers have finished",
                        "max_rel_diff_vs_device_resident_banks": e2e_same, "host_api_call": host_api},
                "strong_scaling": strong, "parity_spot_check": spot, "config3": config3,
                "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roofline,
                "cpu_baseline": cpu, "render": render if render is not None else ({"e2e": render_e2e} if render_e2e else None)}
        print(json.dumps(line), flush=True)
    emdist.barrier()


if __name__ == "__main__":
    main()
