"""Handles on a second device and in concurrent host threads (include/emagls_cuda.h: handles live on a device, and
different handles may be used from different host threads at once).  The launchers keep per-device state (the
opt-in to more than 48 KB of dynamic shared memory, the SM count), so the same call on device 1 after device 0 must
launch every kernel with the shared memory it asks for.  The library has no floating-point atomics and two B200s get
the same launch geometry, so results are compared bit for bit."""
import threading

import numpy as np
import pytest

from emagls_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def n_devices():
    import torch
    return torch.cuda.device_count()


def _dense_grid():
    # more than 6136 directions: the Householder steps (8 (D + 8) bytes) and the generic chain kernel
    # (16 (D + 2 Mc) bytes) then need more than 48 KB of shared memory
    az, ze = synth.fibonacci_sphere(6400)
    hL, hR = synth.synth_hrirs(az, ze, taps=64, delay=20)
    return az, ze, hL, hR


def _cases(em, grids):
    """name -> (environment, call taking a handle).  Together they reach every kernel launched with more than 48 KB
    of dynamic shared memory; the sizes keep each orientation chunk plan independent of free memory."""
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    maz, mze, r, fs = grids["micGridAziRad"], grids["micGridZenRad"], grids["micRadius"], grids["fs"]
    R = np.stack([np.eye(3), synth.rotation_yaw_pitch(40.0, 10.0), synth.rotation_yaw_pitch(-75.0, -20.0)])
    daz, dze, dL, dR = _dense_grid()
    h5L, h5R = synth.synth_hrirs(az, ze, fs=96000.0, taps=128, delay=40)
    m5az, m5ze = synth.fibonacci_sphere(64)
    ring = 2 * np.pi * np.arange(13) / 13
    rng = np.random.default_rng(3)
    x = rng.standard_normal((30000, 32))
    wl, wr = rng.standard_normal((512, 32)), rng.standard_normal((512, 32))
    return {
        # Gram and TSQR routes, both int8 products, the DMMA GEMM, CholeskyQR2
        "emagls2": ({}, lambda h: em.getEMagLs2Filters(hL, hR, az, ze, r, maz, mze, 4, fs, 256, rotations=R,
                                                       handle=h)),
        # Householder QR of the grid basis (hh_factor_step, hh_formq_step)
        "emagls2_householder": ({"EMAGLS_QR_HOUSEHOLDER": "1"},
                                lambda h: em.getEMagLs2Filters(dL, dR, daz, dze, r, maz, mze, 4, fs, 128,
                                                               rotations=R[:2], handle=h)),
        # BASELINE config-5 shape: 64 channels (factor_kernel<64, 128>, gram_chol_kernel, bwd_small_kernel,
        # chain_bwd_kernel, build_F_kernel)
        "config5": ({}, lambda h: em.getEMagLs2Filters(h5L, h5R, az, ze, 0.042, m5az, m5ze, 7, 96000.0, 128,
                                                       handle=h)),
        # generic path: factor_kernel<32, 96>, form_q_kernel, generic_chain_kernel
        "magls": ({}, lambda h: em.getMagLsFilters(dL, dR, daz, dze, 4, fs, 128, handle=h)),
        # ema_sh_rows_kernel (order 6: 49 harmonics)
        "ema_sh": ({}, lambda h: em.getEMagLsFiltersEMAinSH(hL, hR, az, ze, 0.042, ring, 6, 48000, 512, handle=h)),
        # fused render route (fused_render16_kernel)
        "render": ({}, lambda h: (em.binauralDecode(x, 48000, wl, wr, 48000, handle=h),)),
    }


def test_second_device_gives_identical_results(em, grids, n_devices, monkeypatch):
    if n_devices < 2:
        pytest.skip("needs two visible GPUs")
    h0, h1 = em.Handle(0), em.Handle(1)
    for name, (env, call) in _cases(em, grids).items():
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            a = call(h0)
            b = call(h1)
        for i, (x, y) in enumerate(zip(a, b)):
            assert np.array_equal(x, y), (name, i)


def test_handles_in_concurrent_threads(em, grids, n_devices):
    """Two handles each run a different-sized design in its own host thread (ctypes releases the GIL during the
    call); the results equal those of the same calls made one after the other."""
    hs = [em.Handle(0), em.Handle(1 if n_devices >= 2 else 0)]
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    maz, mze, r, fs = grids["micGridAziRad"], grids["micGridZenRad"], grids["micRadius"], grids["fs"]
    hL, hR = synth.synth_hrirs(az, ze)
    h2L, h2R = synth.synth_hrirs(az[::2], ze[::2], taps=64, delay=20)
    R = np.stack([np.eye(3), synth.rotation_yaw_pitch(40.0, 10.0), synth.rotation_yaw_pitch(-75.0, -20.0)])
    calls = [
        # em32: 400 simulation harmonics
        lambda h: em.getEMagLs2Filters(hL, hR, az, ze, r, maz, mze, 4, fs, 256, rotations=R, handle=h),
        # a 6 cm array on every second direction: 784 simulation harmonics, other shared-memory sizes
        lambda h: em.getEMagLs2Filters(h2L, h2R, az[::2], ze[::2], 0.06, maz, mze, 4, fs, 128, rotations=R[:2],
                                       handle=h),
    ]
    got, errors = [None, None], []

    def run(i):
        try:
            got[i] = calls[i](hs[i])
        except BaseException as e:  # re-raised in the main thread
            errors.append(e)

    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    ref = [call(h) for call, h in zip(calls, hs)]
    for i in range(2):
        for j, (x, y) in enumerate(zip(ref[i], got[i])):
            assert np.array_equal(x, y), (i, j)
