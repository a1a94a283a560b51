"""Parity of the full eMagLS2 design path against the oracle and the reference goldens (B200 only).

Acceptance protocol (SURVEY.md 8-c; measured floors in DESIGN.md):
* per bin, FP64: |W_cuda - W_oracle|_inf / |W_oracle|_inf <= 1e-10 for every bin whose steering
  matrix has sigma_min/sigma_max >= 1e-6 (em32: bins >= 16, i.e. >= 750 Hz);
* ill-conditioned bins (< 750 Hz): bounded by the reference algorithm's own 1-ulp sensitivity
  (1e-7 at bin 1 falling to 1e-12 at bin 8), asserted at 2e-6 / 1e-8;
* whole filter: max-norm relative error <= 5e-9 (the measured floor is ~1e-9).
"""
import numpy as np
import pytest

import oracle
from emagls_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def h(em):
    return em.Handle(0)


@pytest.fixture(scope="module")
def c1(grids):
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    return dict(az=az, ze=ze, hL=hL, hR=hR, r=grids["micRadius"], maz=grids["micGridAziRad"],
                mze=grids["micGridZenRad"], fs=grids["fs"])


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def check_bins(W, Wo, first_good=16):
    err = np.abs(W - Wo).max(1) / np.abs(Wo).max(1)
    assert err[first_good:].max() <= 1e-10, err[first_good:].max()
    assert err[8:first_good].max() <= 1e-8, err[8:first_good].max()
    assert err[:8].max() <= 2e-6, err[:8].max()


@pytest.fixture(scope="module")
def oracle_c1(c1):
    return oracle.getEMagLs2Filters(c1["hL"], c1["hR"], c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4,
                                    c1["fs"], 512, return_spectra=True)


def test_emagls2_single_reference_call(em, h, c1, oracle_c1):
    wL, wR, sp = em.getEMagLs2Filters(c1["hL"], c1["hR"], c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4,
                                      c1["fs"], 512, handle=h, return_spectra=True)
    oL, oR, osp = oracle_c1
    assert wL.shape == (512, 32) and wL.dtype == np.float64
    check_bins(sp[:, :, 0], osp["W_l"])
    check_bins(sp[:, :, 1], osp["W_r"])
    assert rel(wL, oL) < 5e-9 and rel(wR, oR) < 5e-9
    assert np.all(wL[0] == 0) and np.all(wL[-1] == 0)                 # fade window end points
    assert np.all(sp[0].imag == 0)                                    # DC bin := real(bin 2)
    # deterministic: a second call is bit-identical
    wL2, wR2 = em.getEMagLs2Filters(c1["hL"], c1["hR"], c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4,
                                    c1["fs"], 512, handle=h)
    assert np.array_equal(wL, wL2) and np.array_equal(wR, wR2)


def test_emagls2_rotation_batch_equals_reference_calls_on_rotated_grids(em, h, c1, oracle_c1):
    Rm = np.stack([synth.rotation_yaw_pitch(33.0, 15.0), np.eye(3), synth.rotation_yaw_pitch(-120.0, -35.0)])
    wL, wR, sp = em.getEMagLs2Filters(c1["hL"], c1["hR"], c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4,
                                      c1["fs"], 512, rotations=Rm, handle=h, return_spectra=True)
    assert wL.shape == (512, 32, 3)
    for o in (0, 1):
        if o == 1:
            oL, oR, osp = oracle_c1
        else:
            raz, rze = synth.rotate_grid(c1["az"], c1["ze"], Rm[o])
            oL, oR, osp = oracle.getEMagLs2Filters(c1["hL"], c1["hR"], raz, rze, c1["r"], c1["maz"], c1["mze"],
                                                   4, c1["fs"], 512, return_spectra=True)
        check_bins(sp[:, :, o, 0], osp["W_l"])
        check_bins(sp[:, :, o, 1], osp["W_r"])
        assert rel(wL[:, :, o], oL) < 5e-9 and rel(wR[:, :, o], oR) < 5e-9


def test_emagls2_hrtf_set_batch_and_orientation_independence(em, h, c1):
    """Two HRTF sets x two orientations in one call == the four single calls (bit for bit on the
    shared operators, to rounding on the rest)."""
    hL2, hR2 = synth.synth_hrirs(c1["az"], c1["ze"], head_radius=0.08, ear_azi_deg=95.0, seed=20261018)
    HL = np.stack([c1["hL"], hL2], 2)
    HR = np.stack([c1["hR"], hR2], 2)
    Rm = np.stack([np.eye(3), synth.rotation_yaw_pitch(90.0, 5.0)])
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"], 512)
    wL, wR = em.getEMagLs2Filters(HL, HR, *args, rotations=Rm, handle=h)
    assert wL.shape == (512, 32, 4)
    for s, (a, b) in enumerate(((c1["hL"], c1["hR"]), (hL2, hR2))):
        sL, sR = em.getEMagLs2Filters(a, b, *args, rotations=Rm, handle=h)
        assert rel(wL[:, :, 2 * s:2 * s + 2], sL) < 1e-12
        assert rel(wR[:, :, 2 * s:2 * s + 2], sR) < 1e-12


def test_emagls2_left_right_symmetry_property(em, h, c1):
    """Size-independent property: swapping the ears of the HRIR set swaps the outputs."""
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"], 512)
    wL, wR = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, handle=h)
    xL, xR = em.getEMagLs2Filters(c1["hR"], c1["hL"], *args, handle=h)
    # the right ear carries the inter-aural delay difference, so compare magnitudes of the spectra
    A, Bq = np.abs(np.fft.rfft(wL, axis=0)), np.abs(np.fft.rfft(xR, axis=0))
    assert np.abs(A - Bq).max() / A.max() < 2e-2


def test_emagls2_orientation_batch_full_size_properties(em, h, c1):
    """BASELINE config 2 shape at reduced batch: identity orientation inside a batch equals the single
    call; filters are finite; a 360-degree yaw returns to the start."""
    R = synth.orientation_grid()[::100]               # 36 orientations of the 3600 grid
    R = np.concatenate([R, np.eye(3)[None], synth.rotation_yaw_pitch(360.0, 0.0)[None]])
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"], 512)
    wL, wR = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, rotations=R, handle=h)
    assert np.all(np.isfinite(wL)) and np.all(np.isfinite(wR))
    sL, sR = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, handle=h)
    assert rel(wL[:, :, -2], sL) < 5e-9 and rel(wL[:, :, -1], sL) < 5e-9


def test_last_partial_round_of_the_jacobi_launch_matches_a_small_batch(em, h, c1):
    """A batch larger than the number of resident Jacobi CTAs (4 per SM: 592 on a B200): the orientations of the
    last partial round are cut into bin ranges (launch_svdclip, tsqr_kernels.cu).  Their filters must equal those
    of the same orientations designed as a small batch of their own (no split there); the only difference allowed
    is the rounding of cold against warm Jacobi starts (lib/getEMagLs2Filters.m:86-89 is the same SVD either way)."""
    Rall = synth.orientation_grid()
    R = Rall[np.arange(603) * 5 % Rall.shape[0]]      # 603 orientations: 11 of them in the last round of 592
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"], 512)
    wL, wR = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, rotations=R, handle=h)
    tail = slice(603 - 12, 603)                        # the split orientations and one before them
    sL, sR = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, rotations=R[tail], handle=h)
    assert np.all(np.isfinite(wL)) and np.all(np.isfinite(wR))
    assert rel(wL[:, :, tail], sL) < 5e-9 and rel(wR[:, :, tail], sR) < 5e-9
    head = slice(0, 4)
    s2L, _ = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, rotations=R[head], handle=h)
    assert rel(wL[:, :, head], s2L) < 5e-9


def test_emagls2_through_cabi_matches_reference_golden_conventions(em, h, goldens):
    """Golden pin (3) through the CUDA path: order-4 surrogate HRIRs from the LS golden reproduce the
    eMagLS2 golden's low bins to a few percent (any convention error gives O(1))."""
    G = goldens
    az, ze = G["hrirGridAziRad"], G["hrirGridZenRad"]
    Y4 = oracle.getSH(4, np.stack([az, ze], 1), "real")
    h4L, h4R = G["real_LS_wLsL"] @ Y4.T, G["real_LS_wLsR"] @ Y4.T
    wL, wR = em.getEMagLs2Filters(h4L, h4R, az, ze, float(G["micRadius"]), G["micGridAziRad"],
                                  G["micGridZenRad"], 4, 48000, 512, handle=h)
    A = np.fft.fft(wL, 1024, axis=0)
    Bq = np.fft.fft(G["real_eMagLS2_woDC_wEMls2L"], 1024, axis=0)
    for lo, hi, tol in ((1, 10, 0.06), (10, 20, 0.12)):
        assert np.abs(A[lo:hi] - Bq[lo:hi]).max() / np.abs(Bq[lo:hi]).max() < tol
    assert np.all(wL[0] == 0) and np.all(wL[-1] == 0)
    assert 250 <= int(np.argmax(np.abs(wL).max(1))) <= 280


def test_error_behaviour_mirrors_reference_asserts(em, h, c1):
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"])
    with pytest.raises(em.EmaglsError, match="len too short"):        # lib/getEMagLs2Filters.m:42
        em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, 64, handle=h)
    with pytest.raises(ValueError):
        em.getEMagLs2Filters(c1["hL"], c1["hR"][:, :100], *args, 512, handle=h)
    # a custom shFunction is evaluated on the host (SURVEY.md H8): one that returns the wrong shape is refused
    with pytest.raises(ValueError, match="shFunction must return"):
        em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, 512, "real", lambda n, d, k: np.zeros((3, 3)), handle=h)
    # designers without the basis pass-through still refuse a non-default handle explicitly
    with pytest.raises(NotImplementedError):
        em.getMagLsFilters(c1["hL"], c1["hR"], c1["az"], c1["ze"], 4, c1["fs"], 512, "real", lambda *a: None, handle=h)


def test_other_filter_lengths_and_rates(em, h, grids):
    """Ragged sizes: short HRIRs, a filter length that is not a power of two, another rate."""
    az, ze = grids["hrirGridAziRad"][::2], grids["hrirGridZenRad"][::2]       # 1351 directions
    hL, hR = synth.synth_hrirs(az, ze, fs=32000.0, taps=48, delay=10)
    args = (az, ze, 0.042, grids["micGridAziRad"], grids["micGridZenRad"], 3, 32000.0, 96)
    wL, wR, sp = em.getEMagLs2Filters(hL, hR, *args, handle=h, return_spectra=True)
    oL, oR, osp = oracle.getEMagLs2Filters(hL, hR, *args, return_spectra=True)
    assert wL.shape == (96, 32)
    err = np.abs(sp[:, :, 0] - osp["W_l"]).max(1) / np.abs(osp["W_l"]).max(1)
    assert err[6:].max() < 1e-9 and rel(wL, oL) < 1e-7 and rel(wR, oR) < 1e-7


def test_stress_config_shape_at_reduced_length(em, h, grids):
    """BASELINE config 5 shape (64-microphone Fibonacci sphere, SH order 7, 96 kHz: simulation order 37,
    1444 harmonics) at a filter length the oracle finishes in seconds."""
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze, fs=96000.0, taps=128, delay=40)
    maz, mze = synth.fibonacci_sphere(64)
    args = (az, ze, 0.042, maz, mze, 7, 96000.0, 128)
    wL, wR, sp = em.getEMagLs2Filters(hL, hR, *args, handle=h, return_spectra=True)
    oL, oR, osp = oracle.getEMagLs2Filters(hL, hR, *args, return_spectra=True)
    assert wL.shape == (128, 64)
    for e, Wo in enumerate((osp["W_l"], osp["W_r"])):
        err = np.abs(sp[:, :, e] - Wo).max(1) / np.abs(Wo).max(1)
        assert err[8:].max() <= 1e-8, err[8:].max()      # 750 Hz bins: same conditioning classes as config 1
        assert err[1:8].max() <= 2e-6, err[1:8].max()
    assert rel(wL, oL) < 5e-8 and rel(wR, oR) < 5e-8
    # SH-domain variant of the same array (64 channels)
    wL, wR = em.getEMagLsFilters(hL, hR, *args, handle=h)
    oL, oR = oracle.getEMagLsFilters(hL, hR, *args)
    assert wL.shape == (128, 64) and rel(wL, oL) < 1e-8 and rel(wR, oR) < 1e-8


def test_stress_config_full_length_properties(em, h, grids):
    """BASELINE config 5 at its full size for one (HRTF set, two orientations): 4096 taps at 96 kHz need
    NFFT_MAX_LEN lifted to 8192 (SURVEY.md H5; K = 4097 bins).  The oracle would need minutes, so the
    checks are size-independent properties: LS bins of single reference-style solves, zero end taps,
    identity orientation inside a batch equals the single call."""
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze, fs=96000.0, taps=256, delay=60)
    maz, mze = synth.fibonacci_sphere(64)
    cfg = h.default_config()
    cfg.nfft_max_len = 8192
    args = (az, ze, 0.042, maz, mze, 7, 96000.0, 4096)
    R = np.stack([synth.rotation_yaw_pitch(33.0, 15.0), np.eye(3)])
    wL, wR, sp = em.getEMagLs2Filters(hL, hR, *args, rotations=R, handle=h, config=cfg, return_spectra=True)
    assert wL.shape == (4096, 64, 2) and np.all(np.isfinite(wL)) and np.all(np.isfinite(wR))
    assert np.all(wL[0] == 0) and np.all(wL[-1] == 0)
    sL, sR = em.getEMagLs2Filters(hL, hR, *args, handle=h, config=cfg)
    assert rel(wL[:, :, 1], sL) < 1e-8 and rel(wR[:, :, 1], sR) < 1e-8
    # LS bins (below k_cut = 299) against the oracle's per-bin solve (lib/getEMagLs2Filters.m:86-92)
    nfft, K = 8192, 4097
    f = np.linspace(0, 48000.0, K)
    Ymic = oracle.getSH(37, np.stack([maz, mze], 1), "real")                   # [64, 1444]
    Yc = oracle.getSH(37, np.stack([az, ze], 1), "real").T                     # [1444, 2702]
    hp = np.zeros((nfft, az.size))
    hp[:256] = hL
    grp = float(np.median(oracle.grpdelay(hp.sum(1), f, 96000.0)))
    HL = np.fft.fft(oracle.applySubsampleDelay(hp, -grp), axis=0)
    for k in (150, 220, 290):   # cond(pwGrid) <= 3e5 there; lower bins sit on the 1e-7 noise floor (DESIGN.md 2)
        bn = -oracle.sphModalCoeffs(37, np.array([2 * np.pi * f[k] / 343.0 * 0.042]))[0]
        pw = (Ymic * oracle.sh_repToOrder(bn[:, None])[:, 0][None, :]) @ Yc
        Wo = HL[k] @ oracle.regularized_inverse(pw)
        assert np.abs(sp[k, :, 1, 0] - Wo).max() <= 1e-8 * np.abs(Wo).max(), k


def test_optional_fp32_contraction_path(em, h, c1, oracle_c1):
    """north_star's optional reduced-precision path (config.precision = FP32: 4 instead of 6 int8 slices in the
    two direction-grid contractions): within 1e-4 relative / 0.05 dB of the reference on the bins FP32 can
    represent (sigma_min / sigma_max >= 1e-3: bins >= 16 for em32), and much closer in practice."""
    cfg = h.default_config()
    cfg.precision = 1
    args = (c1["az"], c1["ze"], c1["r"], c1["maz"], c1["mze"], 4, c1["fs"], 512)
    wL, wR, sp = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, handle=h, config=cfg, return_spectra=True)
    oL, oR, osp = oracle_c1
    for e, Wo in enumerate((osp["W_l"], osp["W_r"])):
        err = np.abs(sp[:, :, e] - Wo).max(1) / np.abs(Wo).max(1)
        assert err[16:].max() <= 1e-4, err[16:].max()
        # magnitude response towards the grid directions is not needed here: per-bin coefficient error of 1e-4
        # bounds the level error by 20 log10(1 + 1e-4) = 9e-4 dB << 0.05 dB
    assert rel(wL, oL) < 1e-4 and rel(wR, oR) < 1e-4
    # the switch really changes the arithmetic (different rounding than the FP64 path) and stays close to it
    w64, _ = em.getEMagLs2Filters(c1["hL"], c1["hR"], *args, handle=h)
    d = rel(wL, w64)
    assert 0 < d < 1e-5, d


_FWD_VARIANT_SNIPPET = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
import emagls_b200 as em
from emagls_b200 import synth
g = synth.load_grids()
az, ze = g["hrirGridAziRad"][::3], g["hrirGridZenRad"][::3]
hL, hR = synth.synth_hrirs(az, ze, taps=64, delay=20)
R = np.stack([np.eye(3), synth.rotation_yaw_pitch(40.0, 10.0), synth.rotation_yaw_pitch(-75.0, -20.0)])
wL, wR = em.getEMagLs2Filters(hL, hR, az, ze, g["micRadius"], g["micGridAziRad"], g["micGridZenRad"], 4, g["fs"], 128,
                              rotations=R, handle=em.Handle(0))
np.savez({out!r}, wL=wL, wR=wR)
"""


def test_forward_functor_variants_agree(tmp_path):
    """The forward tensor-core product's two epilogue functors for six digits must give the same filters
    (lib/getEMagLs2Filters.m:95-103, t = |H_k| y / |y|): the FP64-free one (default) and the FP64 one it is checked
    against (EMAGLS_OZ_FWD=raw: may differ by one unit of the last base-256 digit, 2^-46 of a row maximum).  The switch
    is read once per process, hence the subprocesses."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for name, env in (("default", {}), ("raw", {"EMAGLS_OZ_FWD": "raw"})):
        out = str(tmp_path / f"{name}.npz")
        e = dict(os.environ)
        e.update(env)
        subprocess.run([sys.executable, "-c", _FWD_VARIANT_SNIPPET.format(root=root, out=out)], check=True, env=e,
                       timeout=600)
        res[name] = np.load(out)
    for k in ("wL", "wR"):
        assert rel(res["default"][k], res["raw"][k]) <= 2e-10, (k, rel(res["default"][k], res["raw"][k]))
