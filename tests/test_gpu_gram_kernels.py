"""The Gram route's kernels (emagls_b200/csrc/gram_kernels.cu), launch by launch, against high-precision references
(B200 only).

tests/csrc/gram_harness.cu includes the library's translation units, so the inversion + certificate pair
(`launch_gram_chol`) runs on matrices whose spectra the test chooses, and each backward kernel runs directly as well as
through `launch_bwd_small`'s own choice:

* inversion at every code path of the channel count: `gram_sweep_kernel` with identity padding (Mc < 32) and without
  (Mc = 32), `gram_chol_kernel` with 4 warps per CTA (33 <= Mc <= 59) and 3 (Mc >= 60); complex and real (Gim = 0)
  matrices against the exact inverse (mpmath, 40 digits); the Gim diagonal and the packing gap are never read;
* the route decision: the shifted-Cholesky certificate at its boundary lambda_max ||G^-1||_F = tau (1 - delta), the
  Frobenius classification outside the band, refusals of indefinite and non-finite matrices, the per-bin `fail[]`
  counts against the NumPy mirror `route_ok` (tests/test_gram_certificate_cpu.py);
* production-size launches (128 bins x 3600 orientations at Mc = 32 and 64): a bad candidate in any round of
  `gram_certify_kernel`'s strided loop refuses exactly its own bin;
* the backward step W_k = (Y_o (conj(b_k) .* z)) Pb of `bwd_fused_kernel` and `bwd_small_kernel` against an extended-
  precision reference, their fused forward tails against the unfused `launch_fwd_small` + `launch_slice_rows`.
"""
import math

import mpmath
import numpy as np
import pytest

from oracle.gram_harness import Harness, compile_harness
from test_gram_certificate_cpu import DELTA, em32_spectrum, hermitian, route_ok

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
INVALID = 1                       # cudaErrorInvalidValue
GUARD = 64
ALL_ONES = np.uint64(0xFFFFFFFFFFFFFFFF)   # the FP64 sentinel of the harness (every byte 0xFF)
# Mc -> the inversion kernel that runs: identity-padded sweep, full sweep, Cholesky with 4 or 3 warps per CTA
INV_MC = [1, 2, 7, 16, 25, 31, 32, 33, 47, 59, 60, 64]


def inv_path(Mc):
    if Mc < 32:
        return f"Mc{Mc}-sweep_padded"
    if Mc == 32:
        return f"Mc{Mc}-sweep"
    return f"Mc{Mc}-chol_{4 if Mc <= 59 else 3}warps"


@pytest.fixture(scope="session")
def gh(tmp_path_factory):
    return Harness(compile_harness(str(tmp_path_factory.mktemp("gram_harness"))))


def bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


def real_symmetric(lam, rng):
    M = len(lam)
    Q, _ = np.linalg.qr(rng.standard_normal((M, M)))
    G = (Q * lam) @ Q.T
    return ((G + G.T) / 2).astype(complex)


def pack(mats, ne_ld, poison=False):
    """Packed lower triangles (entry e = m(m+1)/2 + m' holds G[m][m'], m >= m') of the matrices, [n, ne_ld] each.
    poison: NaN in the Gim diagonal and in the packing gap ne .. ne_ld of both arrays (entries the kernels never read)."""
    M = mats[0].shape[0]
    ne = M * (M + 1) // 2
    rows, cols = np.tril_indices(M)                 # row-major order of the lower triangle = e order
    Gre, Gim = np.zeros((len(mats), ne_ld)), np.zeros((len(mats), ne_ld))
    for i, G in enumerate(mats):
        Gre[i, :ne], Gim[i, :ne] = G[rows, cols].real, G[rows, cols].imag
    Gim[:, np.flatnonzero(rows == cols)] = 0.0
    if poison:
        Gim[:, np.flatnonzero(rows == cols)] = np.nan
        Gre[:, ne:] = Gim[:, ne:] = np.nan
    return Gre, Gim


def exact_inverse(G, dps=40):
    with mpmath.workdps(dps):
        X = mpmath.matrix(G.tolist()) ** -1
        return np.array(X.tolist(), dtype=complex)


def refined_inverse(G):
    """FP64 inverse plus one step of refinement with the residual in extended precision (well-conditioned G only)"""
    X = np.linalg.inv(G)
    Gl, Xl = G.astype(np.clongdouble), X.astype(np.clongdouble)
    R = np.eye(G.shape[0], dtype=np.clongdouble) - Gl @ Xl
    return (Xl + Xl @ R).astype(complex)


def guard_intact(a, n):
    return bool((bits(a[n:]) == ALL_ONES).all())


def cert_ratio(G, tau):
    """r = lambda_max ||G^-1||_F / tau of the FP64 matrix"""
    ev = np.linalg.eigvalsh(G)
    return ev[-1] * math.sqrt((ev ** -2.0).sum()) / tau


def spectrum_at_ratio(Mc, r, tau, rng):
    """em32-like spectrum (8 eigenvalues near the top, the largest 1, so ||G||_F ~ 2.8 and condF > tau) whose smallest
    eigenvalue puts lambda_max ||G^-1||_F at r tau"""
    lam = em32_spectrum(tau, rng, M=Mc)[:-1]
    rest = (lam ** -2.0).sum()
    return np.concatenate([lam, [1.0 / math.sqrt((r * tau) ** 2 - rest)]])


# ------------------------------------------------------------------------------------------------- inversion
@pytest.mark.parametrize("kind", ["complex", "real"])
@pytest.mark.parametrize("Mc", INV_MC, ids=inv_path)
def test_inverse_against_the_exact_inverse(gh, Mc, kind, capsys):
    """Pb[m][i] = conj(Ginv[m][i]) within 8 Mc u cond_2(G) (max norm) of the exact inverse; the Gim diagonal and the
    packing gap (NaN) are never read; nothing is written past Pb, sig and fail."""
    rng = np.random.default_rng(1000 + Mc + (kind == "real"))
    make = hermitian if kind == "complex" else real_symmetric
    conds = [30.0, 1e4]
    mats = []
    for c in conds:
        lam = np.exp(rng.uniform(0.0, math.log(c), Mc)) / c
        lam[0] = 1.0
        if Mc > 1:
            lam[-1] = 1.0 / c
        mats.append(make(lam, rng))
    ne = Mc * (Mc + 1) // 2
    ne_ld = ne + 3
    thr = 1e4
    err, Pb, sig, fail = gh.gram_chol(*pack(mats, ne_ld), Mc, len(mats), thr, guard=GUARD)
    assert err == 0
    errp, Pbp, sigp, failp = gh.gram_chol(*pack(mats, ne_ld, poison=True), Mc, len(mats), thr, guard=GUARD)
    assert errp == 0
    assert (bits(Pbp) == bits(Pb)).all() and (bits(sigp) == bits(sig)).all() and (failp == fail).all()
    n = len(mats) * Mc * Mc
    assert guard_intact(Pb.view(np.float64), 2 * n) and guard_intact(sig, len(mats))
    assert (fail[2:] == -1).all()                    # one bin: fail[0], fail[1], then the guard
    for i, G in enumerate(mats):
        X = exact_inverse(G.real if kind == "real" else G) if conds[i] > 100 else refined_inverse(G)
        got = Pb[i * Mc * Mc:(i + 1) * Mc * Mc].reshape(Mc, Mc)
        c2 = np.linalg.cond(G)
        e = np.abs(got - X.conj()).max() / np.abs(X).max()
        with capsys.disabled():
            print(f"\ninverse {inv_path(Mc)} {kind} cond {c2:8.2e}: err {e:8.2e} = {e / (Mc * U * c2):6.3f} Mc u cond")
        assert e <= 8 * Mc * U * c2, (Mc, kind, c2, e)


# ------------------------------------------------------------------------------------------------- certificate
BOUNDARY = [1 - 3e-6, 1 - 2e-6, 1 - 5e-7, 1 + 1e-3, 1.5]


@pytest.mark.parametrize("tau", [1e4, 2500.0])
@pytest.mark.parametrize("Mc", [16, 25, 32, 33, 60, 64], ids=inv_path)
def test_certificate_boundary_on_device(gh, Mc, tau, capsys):
    """lambda_max ||G^-1||_F = r tau with r at both sides of 1 - delta: every matrix is a candidate (sig > 0); accepted
    at and below r = 1 - 2e-6, refused from r = 1 - 5e-7 on (the margin GRAM_CERT_DELTA = 1e-6), as the mirror does;
    sig = tau (1 - delta) / ||G^-1||_F."""
    rng = np.random.default_rng(int(tau) + Mc)
    reps = 3
    mats, ratios = [], []
    for r in BOUNDARY:
        for _ in range(reps):
            mats.append(hermitian(spectrum_at_ratio(Mc, r, tau, rng), rng))
            ratios.append(r)
    ne = Mc * (Mc + 1) // 2
    err, _, sig, fail = gh.gram_chol(*pack(mats, (ne + 1) & ~1), Mc, 1, tau, copy_pb=False, guard=GUARD)
    assert err == 0
    nb = len(mats)
    assert fail[0] == fail[1:1 + nb].sum()
    worst = 0.0
    for b, (G, r) in enumerate(zip(mats, ratios)):
        assert abs(cert_ratio(G, tau) / r - 1) < 1e-9, (b, r)
        assert sig[b] > 0, (b, r, sig[b])
        accepted = fail[1 + b] == 0
        assert accepted == (r <= 1 - 2e-6), (Mc, tau, r)
        assert accepted == route_ok(G, tau), (Mc, tau, r)
        X = np.linalg.inv(G)
        ref = tau * (1 - DELTA) / np.linalg.norm(X, "fro")
        worst = max(worst, abs(sig[b] / ref - 1))
    with capsys.disabled():
        print(f"\ncertificate Mc {Mc} tau {tau:g}: sig vs mirror worst rel {worst:.2e}")
    assert worst <= 1e-12


@pytest.mark.parametrize("tau", [1e4, 2500.0])
def test_certificate_never_accepts_above_tau(gh, tau):
    """Random spectra around and above tau at every channel count: a matrix with cond_2 >= tau is never accepted, and
    the device decides as the mirror wherever the mirror is not within rounding of one of its thresholds."""
    rng = np.random.default_rng(17 + int(tau))
    for Mc in INV_MC[2:]:
        mats = []
        for trial in range(16):
            factor = [1 + 1e-3, 1 - 1e-3, rng.uniform(1.0, 4.0 * Mc), rng.uniform(0.05, 1.0)][trial % 4]
            cond = tau * factor
            lam = np.exp(rng.uniform(0.0, math.log(cond), Mc))
            lam[0], lam[1] = 1.0, cond
            mats.append(hermitian(lam / cond, rng))
        ne = Mc * (Mc + 1) // 2
        err, _, sig, fail = gh.gram_chol(*pack(mats, (ne + 1) & ~1), Mc, 1, tau, copy_pb=False)
        assert err == 0
        for b, G in enumerate(mats):
            accepted = fail[1 + b] == 0
            if np.linalg.cond(G) >= tau:
                assert not accepted, (Mc, b)
            X = np.linalg.inv(G)
            condF = np.linalg.norm(G, "fro") * np.linalg.norm(X, "fro")
            r = cert_ratio(G, tau)
            near = (abs(condF / tau - 1) < 1e-9 or abs(condF / (Mc * tau) - 1) < 1e-9 or
                    abs(r / (1 - DELTA) - 1) < 1e-9)
            if not near:
                assert accepted == route_ok(G, tau), (Mc, b, r)


@pytest.mark.parametrize("Mc", [2, 16, 32, 33, 64], ids=inv_path)
def test_classification_outside_the_band(gh, Mc):
    """condF <= tau: accepted without a certificate; condF > Mc tau: refused without one (sig = 0 for both);
    an indefinite matrix and one with a NaN or an Inf entry (diagonal or off-diagonal) are refused."""
    tau = 1e4
    rng = np.random.default_rng(Mc)
    good = hermitian(np.linspace(1.0, 2.0, Mc), rng)
    bad = hermitian(np.logspace(0, -6, Mc), rng)
    indef = hermitian(np.concatenate([[-1e-3], np.linspace(1.0, 2.0, Mc - 1)]), rng)
    mats = [good, bad, indef]
    assert np.linalg.norm(good) * np.linalg.norm(np.linalg.inv(good)) <= tau
    assert np.linalg.norm(bad) * np.linalg.norm(np.linalg.inv(bad)) > Mc * tau
    ne = Mc * (Mc + 1) // 2
    Gre, Gim = pack(mats + [good] * 4, ne)
    last_off = ne - 2                                # entry (Mc-1, Mc-2)
    Gre[3, last_off] = np.nan
    Gim[4, last_off] = np.inf
    Gre[5, ne - 1] = np.nan                          # last diagonal entry
    Gre[6, 0] = np.inf                               # first diagonal entry
    err, _, sig, fail = gh.gram_chol(Gre, Gim, Mc, 1, tau, copy_pb=False)
    assert err == 0
    assert list(fail[1:8]) == [0, 1, 1, 1, 1, 1, 1] and fail[0] == 6
    assert sig[0] == 0.0 and sig[1] == 0.0
    assert (sig[2:7] == 0.0).all()


def test_more_than_64_channels_is_refused(gh):
    Mc = 65
    ne = Mc * (Mc + 1) // 2
    err, _, _, _ = gh.gram_chol(np.eye(1, ne), np.zeros((1, ne)), Mc, 1, 1e4, copy_pb=False)
    assert err == INVALID


@pytest.mark.parametrize("Mc", [16, 32, 48], ids=inv_path)
def test_fail_counts_against_the_mirror(gh, Mc):
    """fail[0] = sum of the bins; a bin's count is zero iff the mirror accepts all of its matrices; it is at least the
    number of refusals of the inversion stage (indefinite, condF > Mc tau) and at most the mirror's refusals (the
    certificate skips the candidates of a bin that is refused already)."""
    tau = 1e4
    rng = np.random.default_rng(5 + Mc)
    P, nbins = 8, 12
    mats, stage1, mirror = [], [], []
    for b in range(nbins):
        for o in range(P):
            kind = rng.choice(["easy", "easy", "cand_good", "cand_bad", "far", "indef"], p=None if b % 3 else
                              [0.5, 0.3, 0.2, 0.0, 0.0, 0.0])
            if kind == "easy":
                G = hermitian(np.linspace(1.0, 2.0, Mc), rng)
            elif kind == "cand_good":
                G = hermitian(spectrum_at_ratio(Mc, 0.97, tau, rng), rng)
            elif kind == "cand_bad":
                G = hermitian(spectrum_at_ratio(Mc, 1.2, tau, rng), rng)
            elif kind == "far":
                G = hermitian(np.logspace(0, -6, Mc), rng)
            else:
                G = hermitian(np.concatenate([[-0.5], np.linspace(1.0, 2.0, Mc - 1)]), rng)
            mats.append(G)
            stage1.append(kind in ("far", "indef"))
            mirror.append(not route_ok(G, tau) if kind != "indef" else True)
    ne = Mc * (Mc + 1) // 2
    err, _, _, fail = gh.gram_chol(*pack(mats, ne + 1), Mc, P, tau, copy_pb=False)
    assert err == 0
    assert fail[0] == fail[1:1 + nbins].sum()
    st1 = np.array(stage1).reshape(nbins, P).sum(1)
    mir = np.array(mirror).reshape(nbins, P).sum(1)
    for b in range(nbins):
        assert (fail[1 + b] == 0) == (mir[b] == 0), (b, fail[1 + b], mir[b])
        assert st1[b] <= fail[1 + b] <= mir[b], (b, fail[1 + b], st1[b], mir[b])
    assert (mir == 0).sum() >= 2 and (mir > 0).sum() >= 2


# ------------------------------------------------------------------------------------------------- production size
def certify_warps(Mc, nmat, sms):
    """Warps of gram_certify_kernel's grid, as launch_gram_chol sizes it: one round covers 32 x this many ids"""
    per_warp = (Mc * (Mc + 1) + (Mc + 1) // 2) * 16
    wpc = 4
    while wpc > 1 and per_warp * wpc > 227 * 1024:
        wpc -= 1
    smem = per_warp * wpc
    resident = sms * max(1, (228 * 1024) // (smem + 1024))
    chunks = (nmat + 31) // 32
    return min((chunks + wpc - 1) // wpc, resident) * wpc


@pytest.mark.parametrize("Mc", [32, 64], ids=["Mc32-sweep_4warps_3ctas", "Mc64-chol_3warps_1cta"])
def test_production_size_certificate_rounds(gh, Mc, capsys):
    """128 bins x 3600 orientations, as the design launches them: single bad candidates (r = 1 + 1e-3) at the first and
    last lanes of round 0, inside round 2, inside the last round and at the last id each refuse exactly their own bin;
    a bin full of good candidates (r = 0.97) is accepted, and one bad candidate among them refuses it."""
    import torch
    tau, P, nbins = 1e4, 3600, 128
    nmat = P * nbins
    dev = torch.device("cuda")
    rng = np.random.default_rng(Mc)
    ne = Mc * (Mc + 1) // 2
    ne_ld = (ne + 1) & ~1
    easy = [hermitian(np.exp(rng.uniform(0.0, math.log(50.0), Mc)) / 50.0, rng) for _ in range(96)]
    good = [hermitian(spectrum_at_ratio(Mc, 0.97, tau, rng), rng) for _ in range(4)]
    bad = hermitian(spectrum_at_ratio(Mc, 1 + 1e-3, tau, rng), rng)
    assert all(route_ok(G, tau) for G in easy[:4] + good) and not route_ok(bad, tau)

    def dev_pack(mats):
        re, im = pack(mats, ne_ld)
        return torch.from_numpy(re).to(dev), torch.from_numpy(im).to(dev)

    ere, eim = dev_pack(easy)
    idx = torch.arange(nmat, device=dev) % len(easy)
    Gre, Gim = ere[idx].contiguous(), eim[idx].contiguous()
    del idx
    gre, gim = dev_pack(good)
    bre, bim = dev_pack([bad])
    Pb = torch.empty(nmat * Mc * Mc, dtype=torch.complex128, device=dev)
    sig = torch.empty(nmat, dtype=torch.float64, device=dev)
    fail = torch.empty(1 + nbins, dtype=torch.int32, device=dev)

    def run():
        assert gh.gram_chol_device(Gre, Gim, Mc, P, tau, Pb, sig, fail) == 0
        return fail.cpu().numpy()

    f = run()
    assert (f == 0).all() and float(sig.max()) == 0.0
    nw = certify_warps(Mc, nmat, gh.sm_count())
    rnd = 32 * nw
    nrounds = (nmat + rnd - 1) // rnd
    assert nrounds >= 4, nrounds
    last0 = (nrounds - 1) * rnd
    plants = {"round 0, warp 0, lane 0": 0, "round 0, warp 0, lane 31": 31 * nw,
              "round 0, last warp, lane 31": rnd - 1, "inside round 2": 2 * rnd + rnd // 3 + 7,
              "inside the last round": last0 + (nmat - last0) // 2, "last id": nmat - 1}
    with capsys.disabled():
        print(f"\nproduction launch Mc {Mc}: {nw} certify warps, {nrounds} rounds of {rnd} ids")
    for name, i in plants.items():
        Gre[i], Gim[i] = bre[0], bim[0]
        f = run()
        expect = np.zeros(1 + nbins, np.int32)
        expect[0], expect[1 + i // P] = 1, 1
        assert (f == expect).all(), (name, i, np.flatnonzero(f[1:]), f[0])
        assert float(sig[i]) > 0.0
        Gre[i], Gim[i] = ere[i % len(easy)], eim[i % len(easy)]
    # a bin that straddles a round boundary, full of good candidates, then one bad candidate at its end
    b = rnd // P
    ids = torch.arange(b * P, (b + 1) * P, device=dev)
    Gre[ids], Gim[ids] = gre[ids % len(good)], gim[ids % len(good)]
    f = run()
    assert (f == 0).all(), np.flatnonzero(f)
    assert int((sig[b * P:(b + 1) * P] > 0).sum()) == P
    i = (b + 1) * P - 1
    Gre[i], Gim[i] = bre[0], bim[0]
    f = run()
    expect = np.zeros(1 + nbins, np.int32)
    expect[0], expect[1 + b] = 1, 1
    assert (f == expect).all(), (np.flatnonzero(f[1:]), f[0])
    del Gre, Gim, Pb, sig, fail
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------- backward step
def fused_fits(Mc, S, T):
    """launch_bwd_small's choice of bwd_fused_kernel (N < 40 always here)"""
    smem = ((Mc * S + 1) & ~1) * 8 + (8 * 64 + 64 + 64 + 80) * 16 + (4 * 8 + 4) * 8
    kps = (S + 31) & ~31
    return Mc <= 32 and S <= 512 and (Mc * S) % 2 == 0 and smem <= 113 * 1024 and (T == 0 or kps <= 512)


def bwd_id(shape):
    Mc, S = shape
    why = []
    if Mc > 32:
        why.append("Mc_gt_32")
    if S > 512:
        why.append("S_gt_512")
    if (Mc * S) % 2:
        why.append("odd_McS")
    return f"Mc{Mc}_S{S}-" + ("fused" if not why else "small_" + "_".join(why))


BWD_SHAPES = [(4, 289), (4, 400), (4, 529), (19, 289), (19, 400), (19, 529), (32, 289), (32, 400), (32, 529),
              (48, 400), (64, 289)]
# (nsplit, z_shared, k): split-K partials, per-set shared right-hand sides (LS bins), k = 1 with the DC fix
BWD_VARIANTS = [(1, 0, 1), (3, 1, 1), (6, 0, 2), (6, 1, 3)]
SENT = np.uint64(0x7FF8DEADBEEF0001)


def bwd_case(Mc, S, nsplit, z_shared, k, rng):
    N = int(round(math.sqrt(S))) - 1
    assert (N + 1) ** 2 == S
    oc, sets, o0, num_orient, K = 3, 2, 2, 6, 5
    num_prob = sets * oc
    roword = np.repeat(np.arange(N + 1), 2 * np.arange(N + 1) + 1).astype(np.int32)
    cz = lambda *s: rng.standard_normal(s) + 1j * rng.standard_normal(s)
    c = dict(Mc=Mc, S=S, N=N, oc=oc, o0=o0, num_orient=num_orient, num_prob=num_prob, K=K, k=k, dc_fix=1,
             nsplit=nsplit, z_shared=z_shared, roword=roword, KpS=(S + 31) & ~31)
    c["Y"] = rng.standard_normal((oc, Mc, S))
    c["Pb"] = cz(oc, Mc, Mc)
    c["bk"], c["bk_next"] = cz(N + 1), cz(N + 1)
    if z_shared:
        c["z_ear_stride"] = 2 * S + 5
        c["z_set_stride"] = 2 * c["z_ear_stride"] + 7
        c["split_stride"] = sets * c["z_set_stride"] + 3
    else:
        c["z_ear_stride"] = c["z_set_stride"] = 0
        c["split_stride"] = num_prob * 4 * S
    c["z"] = rng.standard_normal(nsplit * c["split_stride"] + 4 * S)
    per_ear = sets * num_orient * Mc * K
    c["w_ear_stride"] = per_ear + 11
    c["nW"] = 2 * c["w_ear_stride"]
    return c


def z_rows(c, j, e):
    """the nsplit partials of problem j, ear e: [nsplit][2][S] (re, im)"""
    S = c["S"]
    if c["z_shared"]:
        base = (j // c["oc"]) * c["z_set_stride"] + e * c["z_ear_stride"]
    else:
        base = (j * 2 + e) * 2 * S
    return np.stack([c["z"][q * c["split_stride"] + base:q * c["split_stride"] + base + 2 * S].reshape(2, S)
                     for q in range(c["nsplit"])])


def w_index(c, j, e, m, k):
    p = (j // c["oc"]) * c["num_orient"] + c["o0"] + j % c["oc"]
    return e * c["w_ear_stride"] + (p * c["Mc"] + m) * c["K"] + k


def bwd_reference(c):
    """W_k[j][e][m] in extended precision and the magnitude bound (|Y_o| |zb|) |Pb| of each entry"""
    Mc, S = c["Mc"], c["S"]
    ld = np.longdouble
    W = np.zeros((c["num_prob"], 2, Mc), np.clongdouble)
    mag = np.zeros((c["num_prob"], 2, Mc), ld)
    bconj = np.conj(c["bk"][c["roword"]]).astype(np.clongdouble)
    for j in range(c["num_prob"]):
        ol = j % c["oc"]
        Y = c["Y"][ol].astype(ld)
        Pb = c["Pb"][ol].astype(np.clongdouble)
        for e in range(2):
            zr = z_rows(c, j, e).astype(ld)
            zc = zr[:, 0].sum(0) + 1j * zr[:, 1].sum(0)
            zb = bconj * zc
            v = Y @ zb
            W[j, e] = v @ Pb
            zmag = np.abs(bconj) * np.abs(zr).sum(axis=(0, 1))
            mag[j, e] = (np.abs(Y) @ zmag) @ np.abs(Pb)
    return W, mag


def fwd_reference(c, W):
    """u = b_{k+1} .* (Y_o^T W_k) rows (j*2+e)*2 + {re, im} in extended precision, and |b| |Y_o|^T |W_k|"""
    S = c["S"]
    u = np.zeros((4 * c["num_prob"], S), np.longdouble)
    mag = np.zeros_like(u)
    b = c["bk_next"][c["roword"]].astype(np.clongdouble)
    for j in range(c["num_prob"]):
        Y = c["Y"][j % c["oc"]].astype(np.longdouble)
        for e in range(2):
            w = W[j, e].astype(np.clongdouble)
            x = b * (Y.T @ w)
            u[(j * 2 + e) * 2], u[(j * 2 + e) * 2 + 1] = x.real, x.imag
            m = np.abs(b) * (np.abs(Y).T @ np.abs(w))
            mag[(j * 2 + e) * 2] = mag[(j * 2 + e) * 2 + 1] = m
    return u, mag


def read_w(c, Wout, k):
    Mc = c["Mc"]
    return np.array([[[Wout[w_index(c, j, e, m, k)] for m in range(Mc)] for e in range(2)]
                     for j in range(c["num_prob"])])


def digits_value(q, sc, T, rows, KpS):
    d = q[:T * rows * KpS].reshape(T, rows, KpS).astype(np.float64)
    w = 256.0 ** -np.arange(T)
    return np.einsum("t,trs->rs", w, d) * sc[:rows, None], d


@pytest.mark.parametrize("shape", BWD_SHAPES, ids=bwd_id)
def test_backward_step_and_fused_tail(gh, shape, capsys):
    """W_k within 4 (Mc + S + nsplit) u of the extended-precision reference (relative to |Y_o| |zb| |Pb|) through both
    kernels and launch_bwd_small (bitwise the kernel it picks); W_{k-1} = real(W_k) at k = 1 (DC fix), every other
    entry of Wsp untouched.  Fused tails: bwd_small_kernel's digits and scales bitwise those of launch_fwd_small +
    launch_slice_rows of its W_k; bwd_fused_kernel's digits reconstruct u within the T-digit bound, with the scales of
    launch_row_scale's rule."""
    Mc, S = shape
    rng = np.random.default_rng(Mc * 1000 + S)
    fits = {T: fused_fits(Mc, S, T) for T in (0, 4, 6)}
    worst = 0.0
    for nsplit, z_shared, k in BWD_VARIANTS:
        c = bwd_case(Mc, S, nsplit, z_shared, k, rng)
        rows, KpS = 4 * c["num_prob"], c["KpS"]
        Wref, mag = bwd_reference(c)
        Wsent = np.full(2 * c["nW"], SENT, np.uint64).view(np.complex128)
        written = {w_index(c, j, e, m, k) for j in range(c["num_prob"]) for e in range(2) for m in range(Mc)}
        dc = {w_index(c, j, e, m, k - 1) for j in range(c["num_prob"]) for e in range(2) for m in range(Mc)} \
            if k == 1 else set()
        untouched = np.ones(c["nW"], bool)
        untouched[list(written | dc)] = False
        tol = 4 * (Mc + S + nsplit) * U
        outs = {}
        for T in (0, 4, 6):
            for mode in (1, 2, 0):
                if mode == 1 and not fits[T]:
                    err, *_ = gh.bwd(mode, T, c, Wsent)
                    assert err == INVALID
                    continue
                err, Wout, q, sc = gh.bwd(mode, T, c, Wsent)
                assert err == 0, (mode, T)
                outs[mode, T] = (Wout, q, sc)
                assert (bits(Wout.view(np.float64)).reshape(-1, 2)[untouched] == SENT).all(), (mode, T)
                W = read_w(c, Wout, k)
                e = np.abs(W - Wref) / mag
                worst = max(worst, float(e.max()) / ((Mc + S + nsplit) * U))
                assert (e <= tol).all(), (mode, T, float(e.max()))
                if k == 1:
                    W0 = read_w(c, Wout, 0)
                    assert (bits(W0.real) == bits(W.real)).all() and (W0.imag == 0).all()
                if T:
                    assert (q[T * rows * KpS:] == 0x5A).all() and guard_intact(sc, rows), (mode, T)
            # launch_bwd_small runs the kernel it picks, bit for bit
            pick = 1 if fits[T] else 2
            for a, b in zip(outs[0, T], outs[pick, T]):
                assert (a is None and b is None) or (bits(a) == bits(b)).all(), (T, pick)
            if T == 0:
                continue
            # bwd_small_kernel's tail: bitwise launch_fwd_small + launch_slice_rows of the same W_k
            Wout, q, sc = outs[2, T]
            err, cv, q2, sc2 = gh.fwd_slice(T, c, Wout, k)
            assert err == 0
            assert (q == q2).all() and (bits(sc) == bits(sc2)).all(), T
            if not fits[T]:
                continue
            # bwd_fused_kernel's tail: digits x scales reconstruct u of its own W_k
            Wout, q, sc = outs[1, T]
            u_ref, umag = fwd_reference(c, read_w(c, Wout, k))
            val, d = digits_value(q, sc, T, rows, KpS)
            assert (d[:, :, S:] == 0).all() and (np.abs(d[0]) <= 64).all()
            bound = sc[:rows, None] * 0.5 * 256.0 ** -(T - 1) * (1 + 1e-12) + 4 * Mc * U * umag
            assert (np.abs(val[:, :S] - u_ref) <= bound).all(), T
            mx = np.abs(u_ref).max(1).astype(np.float64)
            e_ref = np.frexp(mx)[1]
            e_dev = np.log2(sc[:rows]).astype(int) + 6
            near = np.abs(mx - np.ldexp(1.0, np.round(np.log2(mx)).astype(int))) <= 4 * Mc * U * umag.max(1)
            assert ((e_dev == e_ref) | (near & (np.abs(e_dev - e_ref) == 1))).all(), T
    with capsys.disabled():
        print(f"\nbackward {bwd_id(shape)}: worst |W - W_ref| = {worst:.3f} (Mc + S + nsplit) u |Y||zb||Pb|")
