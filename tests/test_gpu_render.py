"""Parity of the binaural render (dependencies/binauralDecode.m) through the C ABI (B200 only).
Tolerance: 1e-9 relative max-norm (north_star); measured ~1e-15."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def h(em):
    return em.Handle(0)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.mark.parametrize("n,ch,ln,comp", [(5000, 32, 512, False), (70000, 32, 512, True), (1000, 25, 512, False),
                                            (300, 4, 64, True), (513, 3, 512, False), (100, 2, 512, False),
                                            (1, 1, 2, False), (360290, 32, 512, False), (40000, 8, 256, True),
                                            (3000, 5, 100, False)])
def test_binaural_decode_matches_oracle(em, h, n, ch, ln, comp):
    rng = np.random.default_rng(n + ch)
    x = rng.standard_normal((n, ch))
    wl, wr = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    y = em.binauralDecode(x, 48000, wl, wr, 48000, comp, handle=h)
    yo = oracle.binauralDecode(x, 48000, wl, wr, 48000, comp)
    assert y.shape == yo.shape
    assert rel(y, yo) < 1e-9


def test_chunk_boundaries(em, h, monkeypatch):
    rng = np.random.default_rng(11)
    x = rng.standard_normal((512 * 70 + 17, 6))
    wl, wr = rng.standard_normal((512, 6)), rng.standard_normal((512, 6))
    yo = oracle.binauralDecode(x, 48000, wl, wr, 48000)
    for chunk in ("1", "7", "64"):
        monkeypatch.setenv("EMAGLS_RENDER_CHUNK", chunk)
        assert rel(em.binauralDecode(x, 48000, wl, wr, 48000, handle=h), yo) < 1e-9


@pytest.mark.parametrize("direct", ["0", "1"])
@pytest.mark.parametrize("fft", ["1024", "2048", "4096", "16384"])
def test_overlap_save_geometries(em, h, monkeypatch, direct, fft):
    """Every FFT size / hop and both forward routes (input transformed in place vs. staged) give the
    reference convolution; even and odd signal lengths (odd lengths always take the staged route)."""
    monkeypatch.setenv("EMAGLS_RENDER_DIRECT", direct)
    monkeypatch.setenv("EMAGLS_RENDER_FFT", fft)
    rng = np.random.default_rng(21)
    wl, wr = rng.standard_normal((512, 5)), rng.standard_normal((512, 5))
    for n in (40000, 40001, 3584 * 4, 3584 * 4 + 512, 700):
        x = rng.standard_normal((n, 5))
        yo = oracle.binauralDecode(x, 48000, wl, wr, 48000)
        assert rel(em.binauralDecode(x, 48000, wl, wr, 48000, handle=h), yo) < 1e-9
    for chunk in ("1", "3"):
        monkeypatch.setenv("EMAGLS_RENDER_CHUNK", chunk)
        x = rng.standard_normal((30000, 5))
        yo = oracle.binauralDecode(x, 48000, wl, wr, 48000, True)
        assert rel(em.binauralDecode(x, 48000, wl, wr, 48000, True, handle=h), yo) < 1e-9


def test_linearity_and_impulse_properties_at_full_size(em, h):
    """Size-independent properties on a 10 s, 32-channel signal: linearity and the impulse response."""
    rng = np.random.default_rng(12)
    n, ch, ln = 480000, 32, 512
    wl, wr = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    a, b = rng.standard_normal((n, ch)), rng.standard_normal((n, ch))
    ya = em.binauralDecode(a, 48000, wl, wr, 48000, handle=h)
    yb = em.binauralDecode(b, 48000, wl, wr, 48000, handle=h)
    yab = em.binauralDecode(2.0 * a - 3.0 * b, 48000, wl, wr, 48000, handle=h)
    assert rel(yab, 2.0 * ya - 3.0 * yb) < 1e-11
    imp = np.zeros((n, ch))
    imp[1000, 5] = 1.0
    yi = em.binauralDecode(imp, 48000, wl, wr, 48000, handle=h)
    assert np.abs(yi[1000:1000 + ln, 0] - wl[:, 5]).max() < 1e-12
    assert np.abs(yi[1000:1000 + ln, 1] - wr[:, 5]).max() < 1e-12
    assert np.abs(yi[:1000]).max() < 1e-12 and np.abs(yi[1000 + ln:]).max() < 1e-12


def test_render_with_designed_filters_end_to_end(em, h, grids):
    """The consumer path: design eMagLS2 filters on the device, render a 32-channel signal with them."""
    from emagls_b200 import synth
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    wL, wR = em.getEMagLs2Filters(hL, hR, az, ze, grids["micRadius"], grids["micGridAziRad"],
                                  grids["micGridZenRad"], 4, grids["fs"], 512, handle=h)
    x = np.random.default_rng(13).standard_normal((20000, 32))
    y = em.binauralDecode(x, 48000, wL, wR, 48000, True, handle=h)
    yo = oracle.binauralDecode(x, 48000, wL, wR, 48000, True)
    assert y.shape == (20000 - 255, 2) and rel(y, yo) < 1e-9


def test_errors(em, h):
    x = np.zeros((10, 3))
    with pytest.raises(ValueError):
        em.binauralDecode(x, 48000, np.zeros((4, 2)), np.zeros((4, 2)), 48000, handle=h)
    with pytest.raises(NotImplementedError):
        em.binauralDecode(x, 48000, np.zeros((4, 3)), np.zeros((4, 3)), 44100, handle=h)


@pytest.mark.parametrize("n,ch,ln,comp,fft", [(30000, 32, 512, False, 0), (9000, 25, 512, True, 0), (20000, 7, 128, False, 4096),
                                              (5000, 1, 64, True, 4096), (12288, 4, 512, False, 0)])
def test_fused_radix16_route_matches_oracle(em, h, monkeypatch, n, ch, ln, comp, fft):
    """The register-resident single-kernel route (default for 4096-sample blocks: radix-16 x 16 x 8 Stockham passes,
    four channels at a time) against the oracle's convolution, 1e-9 relative as for the cuFFT route; channel counts
    that are not multiples of four, signals shorter than a block and the compensated delay included."""
    if fft:
        monkeypatch.setenv("EMAGLS_RENDER_FFT", str(fft))
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    y = em.binauralDecode(x, 48000, wL, wR, 48000, comp, handle=h)
    yo = oracle.binauralDecode(x, 48000, wL, wR, 48000, comp)
    assert y.shape == yo.shape
    assert np.abs(y - yo).max() / np.abs(yo).max() < 1e-9


def test_complex_basis_chain_keeps_the_real_part_of_the_complex_products(em, h, grids):
    """shDefinition = 'complex': encodeSH and the designers return complex arrays; binauralDecode must render
    real(sum_ch x * w) as the reference does (binauralDecode.m:39-42,59-64), not real(x) * real(w)."""
    from emagls_b200 import synth
    rng = np.random.default_rng(5)
    maz, mze = grids["micGridAziRad"], grids["micGridZenRad"]
    sig = rng.standard_normal((6000, maz.size))
    x = em.encodeSH(sig, maz, mze, 4, "complex", handle=h)
    assert np.iscomplexobj(x) and np.abs(x.imag).max() > 0
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    hL, hR = synth.synth_hrirs(az, ze)
    wl, wr = em.getMagLsFilters(hL, hR, az, ze, 4, grids["fs"], 512, "complex", handle=h)
    assert np.iscomplexobj(wl) and np.abs(wl.imag).max() > 0
    for comp in (False, True):
        y = em.binauralDecode(x, 48000, wl, wr, 48000, comp, handle=h)
        yo = oracle.binauralDecode(x, 48000, wl, wr, 48000, comp)
        assert y.shape == yo.shape and not np.iscomplexobj(y)
        assert rel(y, yo) < 1e-9
        # and it is not what dropping the imaginary parts gives
        assert rel(em.binauralDecode(x.real, 48000, wl.real, wr.real, 48000, comp, handle=h), yo) > 1e-3
    with pytest.raises(ValueError):
        em.encodeSH(sig + 1j, maz, mze, 4, handle=h)


def test_time_block_sharded_render_with_halo(em, h):
    """emagls_b200.dist.ShardedRenderer: every rank renders a time block with a (taps - 1)-frame input halo
    (SURVEY.md 8-e); the concatenated blocks equal the unsharded oracle render."""
    from emagls_b200 import dist as emdist
    rng = np.random.default_rng(8)
    n, taps, ch, world = 50000, 512, 32, 4
    x = rng.standard_normal((n, ch))
    wl, wr = rng.standard_normal((taps, ch)), rng.standard_normal((taps, ch))
    ref = oracle.binauralDecode(x, 48000, wl, wr, 48000)
    parts = []
    for r in range(world):
        lo, hi, halo = emdist.render_shard(n, taps, r, world)
        sr = emdist.ShardedRenderer(h, x[lo - halo:hi], wl, wr, halo)
        sr.step()
        parts.append(sr.wait().copy())
    got = np.concatenate(parts, 0)
    assert got.shape == ref.shape and rel(got, ref) < 1e-9


@pytest.mark.parametrize("n,ch,ln,comp", [(30000, 32, 512, False), (9000, 5, 400, True)])
def test_cufft_route_matches_oracle_for_4096_sample_blocks(em, h, monkeypatch, n, ch, ln, comp):
    """The cuFFT + multiply-accumulate route (EMAGLS_RENDER_FUSED=0) on the block size the fused kernel takes by default."""
    monkeypatch.setenv("EMAGLS_RENDER_FUSED", "0")
    rng = np.random.default_rng(n + 1)
    x = rng.standard_normal((n, ch))
    wL, wR = rng.standard_normal((ln, ch)), rng.standard_normal((ln, ch))
    y = em.binauralDecode(x, 48000, wL, wR, 48000, comp, handle=h)
    yo = oracle.binauralDecode(x, 48000, wL, wR, 48000, comp)
    assert np.abs(y - yo).max() / np.abs(yo).max() < 1e-9
