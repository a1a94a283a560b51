"""The int8 tensor-core GEMM (emagls_b200/csrc/ozaki.cuh, ozaki_kernels.cu), instance by instance, against its
bit-exact NumPy model (oracle/ozaki_model.py).

tests/csrc/ozaki_harness.cu includes the library's translation unit, so every one of the ten `ozaki_gemm_kernel`
instances runs directly as well as through `launch_oz_bwd` / `launch_oz_fwd`:

* slicing (`launch_slice_rows`, `launch_row_scale`): digits, scales and zero padding bitwise, both stride layouts;
* backward (`EpiStoreF64` x tile widths 64 / 80 / 48 x T = 4, 6): bitwise equal to the model at edge shapes (N not a
  multiple of 16, odd ldc, half k-tiles, more tiles than SMs in both tile orders, the production shapes, the longest
  contraction `contraction_fits` admits with the int32 accumulators near their limit), accurate against the exact
  product, nothing written outside the output, every element written, the cost rule's choice, the refusals;
* forward (`EpiPhaseSliceRaw<4>`, `<6>`, `EpiPhaseSliceFix<6>` on 128 x 64 and 128 x 80 tiles): the digits of
  Z = rn(t 2^24 256^(T-4)) within 0.6 units of the exact value on hardware (the real MUFU.RSQ seed), digit ranges,
  Nyquist rows, output scales, stores masked at D not a multiple of 4, HRTF-set boundaries inside a tile, and the range
  of the integer functor's 64-bit drain at the longest contractions.
"""
import numpy as np
import pytest

from oracle import ozaki_model as om
from oracle.ozaki_harness import BWD_WIDTH, FWD_NAMES, Harness, compile_harness

pytestmark = pytest.mark.gpu

INVALID = 1            # cudaErrorInvalidValue
GUARD = 256
NAN_BITS = np.uint64(0xFFFFFFFFFFFFFFFF)   # the FP64 sentinel (every byte 0xFF)
WORST = {}             # functor -> worst |Z_dev - Z_exact| seen (units of the last digit)


@pytest.fixture(scope="session")
def oh(tmp_path_factory):
    h = Harness(compile_harness(str(tmp_path_factory.mktemp("ozaki_harness"))))
    yield h
    for k, w in sorted(WORST.items()):
        print(f"\nforward functor {k}: worst |Z_dev - Z_exact| = {w:.4f} units of the last digit")


def bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


def rand_digits(rng, T, R, K, Kpad):
    """valid digit planes: |q_0| <= 64, q_s in [-128, 127]; columns K..Kpad-1 zero"""
    q = np.zeros((T, R, Kpad), np.int8)
    q[0, :, :K] = rng.integers(-64, 65, (R, K), dtype=np.int8)
    q[1:, :, :K] = rng.integers(-128, 128, (T - 1, R, K), dtype=np.int8)
    return q


def rand_scales(rng, R):
    return np.ldexp(1.0, rng.integers(-30, 30, R))


# ----------------------------------------------------------------------------------------------------- slicing
def _slice_source(rng, R, K):
    X = rng.standard_normal((R, K)) * np.ldexp(1.0, rng.integers(-60, 60, R))[:, None]
    X[0] = 0.0                                           # zero row: e = 0
    if R > 2:
        X[1] = np.ldexp(1.0, -1000) * rng.standard_normal(K)   # tiny row (inside the supported range)
        X[2, : K // 2] = 1e290                           # huge row, constant half
    return X


@pytest.mark.parametrize("T", [4, 6])
@pytest.mark.parametrize("R,K,Kpad", [(1, 1, 32), (37, 400, 416), (300, 2702, 2720), (9, 64, 64)])
@pytest.mark.parametrize("layout", ["rows_contiguous", "cols_contiguous"])
def test_slice_rows_matches_the_model_bitwise(oh, T, R, K, Kpad, layout):
    rng = np.random.default_rng(R * 7 + T)
    X = _slice_source(rng, R, K)
    if layout == "rows_contiguous":                      # x(r, k) = src[r ld + k], ld > K
        ld = K + 3
        src = np.zeros((R, ld))
        src[:, :K] = X
        rs, cs = ld, 1
    else:                                                # x(r, k) = src[r + k R] (the direction rows of Y_h)
        src = np.ascontiguousarray(X.T)
        rs, cs = 1, R
    err, out, sc = oh.slice_rows(src.ravel(), rs, cs, R, K, Kpad, T, guard=GUARD, fill=0x5A)
    assert err == 0
    q_ref, s_ref = om.slice_rows(X, T, Kpad)
    n = T * R * Kpad
    assert np.array_equal(out[:n].reshape(T, R, Kpad), q_ref)
    assert (out[n:] == 0x5A).all(), "digits written past the output"
    assert np.array_equal(bits(sc[:R]), bits(s_ref))
    assert (bits(sc[R:]) == NAN_BITS).all(), "scales written past the output"


def test_slice_rows_refuses_other_digit_counts(oh):
    X = np.ones((4, 32))
    err, out, sc = oh.slice_rows(X.ravel(), 32, 1, 4, 32, 32, 5, Tbuf=6, guard=GUARD, fill=0x5A)
    assert err == INVALID
    assert (out == 0x5A).all() and (bits(sc) == NAN_BITS).all()


@pytest.mark.parametrize("rows,D", [(1, 1), (13, 131), (78, 2702)])
def test_row_scale_matches_the_model_bitwise(oh, rows, D):
    rng = np.random.default_rng(rows)
    x = np.abs(rng.standard_normal((rows, D))) * np.ldexp(1.0, rng.integers(-40, 40, rows))[:, None]
    x[0] = 0.0
    err, up, sc = oh.row_scale(x, guard=GUARD)
    assert err == 0
    up_ref, sc_ref = om.row_scale(x)
    assert np.array_equal(bits(up[:rows]), bits(up_ref)) and np.array_equal(bits(sc[:rows]), bits(sc_ref))
    assert (bits(up[rows:]) == NAN_BITS).all() and (bits(sc[rows:]) == NAN_BITS).all()


# ----------------------------------------------------------------------------------------------------- backward
def run_bwd(oh, inst, qA, sA, qB, sB, T):
    M, N = qA.shape[1], qB.shape[1]
    err, out = oh.bwd(inst, qA, sA, qB, sB, T, guard=GUARD)
    assert err == 0, f"instance {inst}: error {err}"
    assert (bits(out[M * N:]) == NAN_BITS).all(), f"instance {inst}: written past the output"
    C = out[: M * N].reshape(M, N)
    assert not np.isnan(C).any(), f"instance {inst}: {np.isnan(C).sum()} elements not written"
    return C


def check_bwd(oh, qA, sA, qB, sB, T, sample=None):
    """every backward instance and launch_oz_bwd: bitwise the model (on `sample` rows) and bitwise one another"""
    M = qA.shape[1]
    rows = np.arange(M) if sample is None else sample
    ref = om.gemm_f64(qA[:, rows], sA[rows], qB, sB, T)
    first = None
    for inst in (0, 1, 2, 3):
        C = run_bwd(oh, inst, qA, sA, qB, sB, T)
        bad = bits(C[rows]) != bits(ref)
        assert not bad.any(), (f"instance {inst}: {bad.sum()} elements differ from the model, first at "
                               f"{np.argwhere(bad)[0]}")
        if first is None:
            first = C
        else:
            assert np.array_equal(bits(C), bits(first)), f"instance {inst} differs from instance 0"
    return first


@pytest.mark.parametrize("T", [4, 6])
@pytest.mark.parametrize("M,N,K,Kpad", [
    (1, 1, 1, 32),                      # one element
    (129, 17, 90, 96),                  # N not a multiple of 16, odd ldc; Kpad = 1.5 k-tiles
    (129, 25, 96, 96),
    (129, 401, 70, 96),
    (300, 100, 400, 416),               # the em32 harmonic count: 6.5 k-tiles
    (2 * 148 * 128 + 1, 48, 32, 32),    # more tiles than SMs, one column tile (consecutive tiles share A rows)
    (128, 300 * 80, 32, 32),            # more tiles than SMs, one row tile (consecutive tiles share B rows)
])
def test_backward_instances_match_the_model_bitwise(oh, T, M, N, K, Kpad):
    rng = np.random.default_rng(M + N + K + T)
    qA, qB = rand_digits(rng, T, M, K, Kpad), rand_digits(rng, T, N, K, Kpad)
    check_bwd(oh, qA, rand_scales(rng, M), qB, rand_scales(rng, N), T)


@pytest.mark.parametrize("T", [4, 6])
@pytest.mark.parametrize("rows", [14400, 1800])
def test_backward_production_shapes(oh, T, rows):
    """4P x S x KpD of the 3600- and 450-orientation batches: the model on a sample of rows that includes the
    first and the last row tile, the instances bitwise equal everywhere"""
    S, D, KpD = 400, 2702, 2720
    rng = np.random.default_rng(rows + T)
    qA, qB = rand_digits(rng, T, rows, D, KpD), rand_digits(rng, T, S, D, KpD)
    sample = np.unique(np.r_[np.arange(0, 128, 5), np.arange(rows - 128, rows, 5), rows - 1,
                             rng.choice(rows, 64, replace=False)])
    check_bwd(oh, qA, rand_scales(rng, rows), qB, rand_scales(rng, S), T, sample)


@pytest.mark.parametrize("T,Kpad", [(6, 21824), (4, 32736)])
def test_backward_longest_contraction(oh, T, Kpad):
    """the largest Kpad contraction_fits admits, with constant rows of extreme digits: (64, -128, -128, ...) (the
    digits of a row at 63.5 of its scale) and (-64, -128, ...), which bring the int32 accumulators to 0.74 - 0.83 of
    2^31"""
    assert oh.contraction_fits(Kpad, T) and not oh.contraction_fits(Kpad + 32, T)
    rng = np.random.default_rng(Kpad)
    M, N = 130, 70
    qA, qB = rand_digits(rng, T, M, Kpad, Kpad), rand_digits(rng, T, N, Kpad, Kpad)
    for q in (qA, qB):
        q[:, :3] = -128
        q[0, 0], q[0, 1], q[0, 2] = 64, -64, -64
    sA, sB = rand_scales(rng, M), rand_scales(rng, N)
    acc = om.diagonals(qA[:, :3], qB[:, :3], T)
    assert max(np.abs(a).max() for a in acc) >= 0.74 * 2.0 ** 31
    check_bwd(oh, qA, sA, qB, sB, T, sample=np.r_[0:8, M - 8:M])


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="long double without a 64-bit significand")
@pytest.mark.parametrize("T", [4, 6])
def test_backward_accuracy_against_the_exact_product(oh, T):
    """|C - A B^T| <= 2^-(8T-4) max|a_row| max|b_row| K (T = 6: the 2^-44 of test_sliced_product_error_and_int32_range)
    with A, B sliced by the model from real data of widely varying row scales"""
    M, N, K, Kpad = 129, 60, 2702, 2720
    rng = np.random.default_rng(T)
    A = rng.standard_normal((M, K)) * np.ldexp(1.0, rng.integers(-20, 20, M))[:, None]
    B = rng.standard_normal((N, K)) * np.ldexp(1.0, rng.integers(-20, 20, N))[:, None]
    qA, sA = om.slice_rows(A, T, Kpad)
    qB, sB = om.slice_rows(B, T, Kpad)
    C = run_bwd(oh, 0, qA, sA, qB, sB, T)
    exact = A.astype(np.longdouble) @ B.T.astype(np.longdouble)
    bound = 2.0 ** -(8 * T - 4) * np.abs(A).max(1)[:, None] * np.abs(B).max(1)[None, :] * K
    ratio = (np.abs(C.astype(np.longdouble) - exact) / bound).max()
    assert ratio <= 1.0, ratio


def test_backward_cost_rule_picks_each_width(oh):
    """launch_oz_bwd equals the instance its cost rule names; at 148 SMs the three shapes take each width once"""
    sms, S, D, KpD, T = oh.sm_count(), 400, 2702, 2720, 6
    picked = set()
    for rows in (14400, 1800, 2688):
        m_tiles = (rows + 127) // 128
        cost = {nt: om.cost_rounds(m_tiles, S, nt, sms) for nt in (64, 80, 48)}
        nt = 80 if cost[80] <= cost[64] else 64
        if cost[48] < cost[nt]:
            nt = 48
        picked.add(nt)
        rng = np.random.default_rng(rows)
        qA, qB = rand_digits(rng, T, rows, D, KpD), rand_digits(rng, T, S, D, KpD)
        sA, sB = rand_scales(rng, rows), rand_scales(rng, S)
        inst = {64: 0, 80: 1, 48: 2}[nt]
        assert BWD_WIDTH[inst] == nt
        C = run_bwd(oh, 3, qA, sA, qB, sB, T)
        assert np.array_equal(bits(C), bits(run_bwd(oh, inst, qA, sA, qB, sB, T)))
    if sms == 148:
        assert picked == {48, 64, 80}


@pytest.mark.parametrize("inst", [0, 1, 2, 3])
@pytest.mark.parametrize("T,Kpad", [(6, 48), (6, 21856), (4, 32768), (5, 32)])
def test_backward_refusals(oh, inst, T, Kpad):
    """Kpad not a multiple of 32, Kpad over the int32 limit, T not in {4, 6}: cudaErrorInvalidValue, nothing written"""
    q = np.ones((6, 2, Kpad), np.int8)
    err, out = oh.bwd(inst, q, np.ones(2), q, np.ones(2), T, guard=GUARD)
    assert err == INVALID
    assert (bits(out) == NAN_BITS).all()


# ----------------------------------------------------------------------------------------------------- forward
_CASES = {}


def fwd_case(D, S, KpS, P, T, flat=False, orient_per_set=3):
    """Y_h [D][S] and c [4P][S] sliced by the model, |H| of one bin of a [set][ear][bin][D] array, the exact y and
    the unrounded Z of every output row.  Problem 1 has y = 0 (zero rows of c); the re / im rows of a problem are up to
    2^40 apart in scale; some |H| are 2^-30 of their row maximum.  `flat`: every row of Y_h and c constant just below
    a power of two, the largest |y| the digit ranges allow."""
    key = (D, S, KpS, P, T, flat, orient_per_set)
    if key in _CASES:
        return _CASES[key]
    rng = np.random.default_rng(D * 31 + S + P + T)
    rows = 4 * P
    Y = rng.standard_normal((D, S)) * np.ldexp(1.0, rng.integers(-3, 4, D))[:, None]
    Cm = rng.standard_normal((rows, S))
    sh = rng.integers(-20, 21, 2 * P)
    Cm[0::2] *= np.ldexp(1.0, sh)[:, None]
    Cm[1::2] *= np.ldexp(1.0, -sh)[:, None]
    if P > 1:
        Cm[4:8] = 0.0
    if flat:
        Y[:] = 1.0 - 2.0 ** -30
        Cm[:] = 1.0 - 2.0 ** -30
    qY, sY = om.slice_rows(Y, T, KpS)
    qC, sC = om.slice_rows(Cm, T, KpS)
    nsets, Kb, kb = -(-P // orient_per_set), 3, 1
    absH = np.abs(rng.standard_normal((nsets, 2, Kb, D))) + 0.01
    absH[0, 1, kb, : D // 2] *= 2.0 ** -30
    up, sc = om.row_scale(absH.reshape(-1, D))
    v = om.exact_values(om.diagonals(qY, qC, T), T)
    Z = om.phase_reference(v, sC, absH[:, :, kb, :], up.reshape(nsets, 2, Kb)[:, :, kb], T, orient_per_set, False)
    prob = np.arange(rows) >> 2
    c = dict(qY=qY, sY=sY, qC=qC, sC=sC, D=D, KpS=KpS, KpD=(D + 31) // 32 * 32, rows=rows, T=T, v=v, Z=Z,
             absH_bin=np.ascontiguousarray(absH.ravel()[kb * D:]), abs_set_stride=2 * Kb * D, abs_ear_stride=Kb * D,
             up_bin=np.ascontiguousarray(up[kb:]), sc_bin=np.ascontiguousarray(sc[kb:]), scale_stride=Kb,
             orient_per_set=orient_per_set,
             sT=sc[kb + ((prob // orient_per_set) * 2 + ((np.arange(rows) >> 1) & 1)) * Kb])
    _CASES[key] = c
    return c


def run_fwd(oh, inst, c, nyquist, fill):
    T, rows, KpD, D = c["T"], c["rows"], c["KpD"], c["D"]
    err, out, sT = oh.fwd(inst, c, T, nyquist, fill, guard=GUARD)
    assert err == 0, f"{FWD_NAMES[inst]}: error {err}"
    n = T * rows * KpD
    assert (out[n:] == np.int8(fill)).all(), f"{FWD_NAMES[inst]}: digits written past the output"
    assert (bits(sT[rows:]) == NAN_BITS).all(), f"{FWD_NAMES[inst]}: scales written past the output"
    q = out[:n].reshape(T, rows, KpD)
    # the integer functor's 4-byte stores may put zeros into the padding up to the next multiple of 4, no further
    D4 = (D + 3) // 4 * 4
    assert (q[:, :, D4:] == np.int8(fill)).all(), f"{FWD_NAMES[inst]}: padding written"
    pad = q[:, :, D:D4]
    assert ((pad == np.int8(fill)) | (pad == 0)).all()
    return q[:, :, :D], sT[:rows]


def check_fwd(oh, inst, c, nyquist, name):
    T = c["T"]
    q, sT = run_fwd(oh, inst, c, nyquist, 0x7F)
    q2, sT2 = run_fwd(oh, inst, c, nyquist, -0x80)
    assert np.array_equal(q, q2) and np.array_equal(bits(sT), bits(sT2)), "bytes of rows < D left unwritten"
    assert np.abs(q[0].astype(int)).max() <= 64, "leading digit out of range"
    assert np.array_equal(bits(sT), bits(c["sT"])), "output row scales"
    Z = c["Z"].copy()
    if nyquist:
        Z[1::2] = 0
        assert not q[:, 1::2].any(), "imaginary rows of the Nyquist bin not zero"
    dz = float(np.abs(om.digits_value(q).astype(np.longdouble) - Z).max())
    WORST[name] = max(WORST.get(name, 0.0), dz)
    assert dz <= 0.6, f"{FWD_NAMES[inst]}: |Z - exact| = {dz:.4f} units of the last digit"
    return q, sT


_FWD_T = {0: 4, 1: 6, 2: 6, 3: 6}
_FUNCTOR = {0: "EpiPhaseSliceRaw<4>", 1: "EpiPhaseSliceRaw<6>", 2: "EpiPhaseSliceFix<6>", 3: "EpiPhaseSliceFix<6>"}


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="long double without a 64-bit significand")
@pytest.mark.parametrize("nyquist", [0, 1])
@pytest.mark.parametrize("D", [1, 5, 131, 2702])
@pytest.mark.parametrize("S,KpS", [(25, 32), (400, 416)])
@pytest.mark.parametrize("inst", [0, 1, 2, 3])
def test_forward_instances_against_the_exact_phase(oh, inst, S, KpS, D, nyquist):
    """37 problems (148 rows = 4 mod 8), 3 orientations per HRTF set (set boundaries inside tiles and inside 8-column
    chunks)"""
    c = fwd_case(D, S, KpS, 37, _FWD_T[inst])
    check_fwd(oh, inst, c, nyquist, _FUNCTOR[inst])


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="long double without a 64-bit significand")
@pytest.mark.parametrize("P", [16, 450])
def test_forward_cost_rule(oh, P):
    """launch_oz_fwd equals the instance its cost rule names (at 148 SMs: 128 x 64 tiles for 64 rows, 128 x 80 tiles
    with 20 epilogue warps for 1800 rows); four digits take the FP64 functor"""
    sms, D = oh.sm_count(), 2702
    c = fwd_case(D, 400, 416, P, 6)
    m_tiles = (D + 127) // 128
    inst = 3 if om.cost_rounds(m_tiles, c["rows"], 80, sms) < om.cost_rounds(m_tiles, c["rows"], 64, sms) else 2
    if sms == 148:
        assert inst == {16: 2, 450: 3}[P]
    q, sT = check_fwd(oh, 4, c, 0, _FUNCTOR[inst])
    q_i, sT_i = run_fwd(oh, inst, c, 0, 0x7F)
    assert np.array_equal(q, q_i) and np.array_equal(bits(sT), bits(sT_i))
    c4 = fwd_case(131, 400, 416, 5, 4)
    q, sT = check_fwd(oh, 4, c4, 1, _FUNCTOR[0])
    q_i, sT_i = run_fwd(oh, 0, c4, 1, 0x7F)
    assert np.array_equal(q, q_i) and np.array_equal(bits(sT), bits(sT_i))


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="long double without a 64-bit significand")
def test_forward_integer_drain_range(oh):
    """The integer functor's drain holds |y| < 2^63 only up to KpS = 2016 (oz::drain_i64_fits).  At KpS = 2016 flat
    rows stay below 2^63 and both six-digit functors are exact; at KpS = 2080 (S = 2049, simulation order 44) the same
    rows give |y| > 2^63, and launch_oz_fwd must still deliver the exact phase."""
    assert oh.drain_i64_fits(2016, 6) and not oh.drain_i64_fits(2048, 6) and oh.drain_i64_fits(32736, 4)
    c = fwd_case(131, 2016, 2016, 3, 6, flat=True)
    vmax = max(abs(int(x)) for x in c["v"].ravel())
    assert 2 ** 62 < vmax < 2 ** 63
    for inst in (1, 2, 3, 4):
        check_fwd(oh, inst, c, 0, _FUNCTOR[inst] if inst < 4 else "EpiPhaseSliceFix<6>")
    c = fwd_case(131, 2049, 2080, 3, 6, flat=True)
    vmax = max(abs(int(x)) for x in c["v"].ravel())
    assert vmax > 2 ** 63
    check_fwd(oh, 4, c, 0, "launch_oz_fwd KpS 2080")
    check_fwd(oh, 1, c, 1, _FUNCTOR[1])


@pytest.mark.parametrize("what", ["rows_not_4", "T5", "kpad_over_limit"])
def test_forward_refusals(oh, what):
    """six digits with a row count that is not a multiple of 4, T not in {4, 6}, KpS over the int32 limit:
    cudaErrorInvalidValue, nothing written"""
    D, P = 5, 2
    c = dict(fwd_case(D, 25, 32, P, 6))
    T = 6
    if what == "rows_not_4":
        c["qC"] = c["qC"][:, :6]
        c["sC"] = c["sC"][:6]
    elif what == "T5":
        T = 5
    else:
        c["KpS"] = 21856
        c["qY"] = np.zeros((6, D, 21856), np.int8)
        c["qC"] = np.zeros((6, 4 * P, 21856), np.int8)
    err, out, sT = oh.fwd(4, c, T, 0, 0x7F, guard=GUARD)
    assert err == INVALID
    assert (out == 0x7F).all() and (bits(sT) == NAN_BITS).all()
