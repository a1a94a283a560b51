"""Which em32 bins take the Gram route (B200 only).

The clip of lib/getEMagLs2Filters.m:88 is active in bins 1..66 (numbered from 0 = DC) of the em32 / order-4 / 512-tap
design (cond_2(G_k) > 1/c^2 = 1e4 there, tests/test_gram_certificate_cpu.py); every other bin has cond_2(G_k) <= 9.6e3
and the condition
certificate of the Gram route accepts it, so exactly the clipped bins go through TSQR + Jacobi.  The per-bin parity of
the Gram bins against the oracle is checked with the same protocol as tests/test_gpu_design.py.
"""
import numpy as np
import pytest

import oracle
from emagls_b200 import synth

pytestmark = pytest.mark.gpu


def test_em32_gram_route_takes_every_unclipped_bin(grids):
    import emagls_b200 as em
    h = em.Handle(0)
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    args = (az, ze, grids["micRadius"], grids["micGridAziRad"], grids["micGridZenRad"], 4, grids["fs"], 512)
    R = np.stack([np.eye(3), synth.rotation_yaw_pitch(90.0, 5.0)])
    h.stats_read()
    _, _, sp = em.getEMagLs2Filters(hL, hR, *args, rotations=R, handle=h, return_spectra=True)
    st = h.stats_read()
    assert st["tsqr_problem_bins"] == 66 * 2, st
    assert st["gram_problem_bins"] == 446 * 2, st
    # bins 67..76 moved from the TSQR to the Gram route: same acceptance as every other well-conditioned bin
    _, _, osp = oracle.getEMagLs2Filters(hL, hR, *args, return_spectra=True)
    for ear, key in ((0, "W_l"), (1, "W_r")):
        err = np.abs(sp[:, :, 0, ear] - osp[key]).max(1) / np.abs(osp[key]).max(1)
        assert err[67:77].max() <= 1e-10, err[67:77].max()
