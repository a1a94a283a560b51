"""CPU mirrors of two warp-level data-flow patterns of the CUDA path (no GPU needed): the lanes of a warp are the
rows of a NumPy array, `__shfl_xor_sync(x, m)` is `x[lane ^ m]`, `__byte_perm` is restated below.

* `EpiPhaseSliceFix<T>::apply` (emagls_b200/csrc/ozaki_kernels.cu): the digit bytes of four columns, packed per
  digit plane, are transposed across groups of four lanes with two shuffles and two byte permutes, so that lane l
  holds rows l & ~3 .. (l & ~3) + 3 of column l & 3 and stores one 4-byte word.
* `wsum2c` (emagls_b200/csrc/reflect.cuh): the warp sums of two complex values by reduce-scatter over the first two
  butterfly stages, three stages on the remaining scalar and an all-gather; every lane must end up with the same
  bits, because the applied-reflector chain (`chain_bwd_sep_kernel`, `apply_qc`) branches on them lane by lane.
"""
import numpy as np

LANES = np.arange(32)


def byte_perm(a, b, sel):
    """__byte_perm(a, b, sel): byte i of the result is byte (sel >> 4 i) & 7 of the 8-byte pool {a: 0-3, b: 4-7}."""
    a, b, sel = np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64), np.asarray(sel, dtype=np.int64)
    sh = 8 * np.arange(4, dtype=np.int64)
    pool = np.concatenate([(a[:, None] >> sh) & 0xFF, (b[:, None] >> sh) & 0xFF], 1)
    out = np.zeros_like(a)
    for i in range(4):
        idx = (sel >> (4 * i)) & 7
        out |= pool[np.arange(a.size), idx] << (8 * i)
    return out


def test_four_lane_byte_transpose_matches_the_store_layout():
    rng = np.random.default_rng(5)
    # byte c of lane l's word = digit of (row l, column c)
    B = rng.integers(0, 256, size=(32, 4), dtype=np.int64)
    x = (B << (8 * np.arange(4, dtype=np.int64))).sum(1)
    sel_a = np.where(LANES & 2, 0x3276, 0x5410)
    sel_b = np.where(LANES & 1, 0x3715, 0x6240)
    x = byte_perm(x, x[LANES ^ 2], sel_a)
    x = byte_perm(x, x[LANES ^ 1], sel_b)
    for lane in range(32):
        g, base = lane & 3, lane & ~3
        want = sum(int(B[base + k, g]) << (8 * k) for k in range(4))
        assert int(x[lane]) == want, lane


def test_transpose4x3_packs_digit_planes():
    """oz::transpose4x3: words r0, r1, r2 hold byte 0, 1, 2 of the four inputs (one digit plane each)."""
    rng = np.random.default_rng(6)
    a, b, c, d = (rng.integers(0, 1 << 24, size=8, dtype=np.int64) for _ in range(4))
    ab_lo, cd_lo = byte_perm(a, b, np.full(8, 0x5140)), byte_perm(c, d, np.full(8, 0x5140))
    ab_hi, cd_hi = byte_perm(a, b, np.full(8, 0x7362)), byte_perm(c, d, np.full(8, 0x7362))
    r0 = byte_perm(ab_lo, cd_lo, np.full(8, 0x5410))
    r1 = byte_perm(ab_lo, cd_lo, np.full(8, 0x7632))
    r2 = byte_perm(ab_hi, cd_hi, np.full(8, 0x5410))
    for j, r in enumerate((r0, r1, r2)):
        for k, src in enumerate((a, b, c, d)):
            assert np.array_equal((r >> (8 * k)) & 0xFF, (src >> (8 * j)) & 0xFF)


def wsum2c(a, b):
    """The data flow of wsum2c() on arrays indexed by lane (complex128 in, complex128 out)."""
    hi16, hi8 = (LANES & 16) != 0, (LANES & 8) != 0
    keep = np.where(hi16, b, a)
    send = np.where(hi16, a, b)
    keep = keep + send[LANES ^ 16]                 # re and im are added separately on the device, as here
    k = np.where(hi8, keep.imag, keep.real)
    s = np.where(hi8, keep.real, keep.imag)
    k = k + s[LANES ^ 8]
    for m in (4, 2, 1):
        k = k + k[LANES ^ m]
    o = k[LANES ^ 8]
    c = np.where(hi8, o, k) + 1j * np.where(hi8, k, o)
    d = c[LANES ^ 16]
    return np.where(hi16, d, c), np.where(hi16, c, d)


def test_fused_two_value_warp_sum():
    rng = np.random.default_rng(7)
    for scale in (1.0, 1e-9, 1e12):
        a = (rng.standard_normal(32) + 1j * rng.standard_normal(32)) * scale
        b = (rng.standard_normal(32) + 1j * rng.standard_normal(32)) * scale * rng.uniform(1e-6, 1e6, 32)
        sa, sb = wsum2c(a, b)
        assert np.all(sa == sa[0]) and np.all(sb == sb[0])      # identical bits in every lane
        assert abs(sa[0] - a.sum()) <= 64 * np.finfo(float).eps * np.abs(a).sum()
        assert abs(sb[0] - b.sum()) <= 64 * np.finfo(float).eps * np.abs(b).sum()
