"""Posterior quantiles and marginal histograms on the device (ParticlePDF.quantile / histogram / histogram2d).

Every result is compared with oracle/summaries.py bit for bit: the masses are fixed-point integers, so the device
and the oracle sum the same integers, and a quantile is always one particle's coordinate."""
import ctypes as C
import warnings

import numpy as np
import pytest

from oracle import summaries as orc

pytestmark = pytest.mark.gpu

LEVELS = [(0.5,), (0.0, 1.0), (0.025, 0.5, 0.975), tuple(np.linspace(0.0, 1.0, 16)), (1e-300, 0.3, 1 - 2 ** -53)]


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _check_all(pdf, levels=(0.025, 0.5, 0.975), bins=64, bins2d=(16, 24)):
    x, w = pdf.particles, pdf.particle_weights
    wq = orc.quantised(w)
    d = x.shape[0]
    got = pdf.quantile(levels)
    want = orc.quantiles(x, w, levels)
    np.testing.assert_array_equal(_bits(got), _bits(want))
    mass, edges, counts = pdf.histogram(bins, return_counts=True)
    for r in range(d):
        lo, hi = orc.auto_range(x[r], wq)
        e = np.histogram_bin_edges(np.empty(0), bins, range=(lo, hi))
        np.testing.assert_array_equal(_bits(edges[r]), _bits(e))
        raw, cnt = orc.histogram(x[r], wq, e)
        np.testing.assert_array_equal(_bits(mass[r]), _bits(orc.mass(raw)))
        np.testing.assert_array_equal(counts[r], cnt)
    i, j = 0, d - 1
    m2, xe, ye, c2 = pdf.histogram2d(i, j, bins2d, return_counts=True)
    xe_w = np.histogram_bin_edges(np.empty(0), bins2d[0], range=orc.auto_range(x[i], wq))
    ye_w = np.histogram_bin_edges(np.empty(0), bins2d[1], range=orc.auto_range(x[j], wq))
    np.testing.assert_array_equal(_bits(xe), _bits(xe_w))
    np.testing.assert_array_equal(_bits(ye), _bits(ye_w))
    raw2, cnt2 = orc.histogram2d(x[i], x[j], wq, xe_w, ye_w)
    np.testing.assert_array_equal(_bits(m2), _bits(orc.mass(raw2)))
    np.testing.assert_array_equal(c2, cnt2)
    return got


def _cloud(n, d, seed):
    g = np.random.default_rng(seed)
    cols = [g.normal(3.0, 0.5, n), g.uniform(-2000, -400, n), g.normal(5e4, 1e3, n), g.standard_cauchy(n)]
    return np.array(cols[:d])


@pytest.mark.parametrize('n', [1, 2, 3, 2047, 2049, 4097, 100_003, 1_000_000, 10_000_001])
@pytest.mark.parametrize('kind', ['explicit', 'uniform', 'masked'])
def test_matches_oracle(obe, n, kind):
    d = 1 + n % 4
    pdf = obe.ParticlePDF(_cloud(n, d, n), seed=3)
    g = np.random.default_rng(n + 1)
    if kind == 'explicit':
        w = g.exponential(size=n) ** 3
        pdf.particle_weights = w / w.sum()
    elif kind == 'uniform':
        pdf.resample()                                     # systematic: the weights are implicit afterwards
        assert pdf._buf.stats[62].item() > 0
    else:
        pdf.particles = pdf.particles - np.median(pdf.particles[0]) * np.eye(d, 1)
        if n > 1:
            pdf._refresh(mask_le=1, renormalise=1)       # weight <- 0 where x_0 <= 0, as a constraint mask does
            pdf._weights_lazy = True
            pdf._invalidate()
            assert np.count_nonzero(pdf.particle_weights == 0) > 0
    for levels in LEVELS:
        _check_all(pdf, levels)


@pytest.mark.parametrize('d', [1, 2, 3, 4])
def test_dimensions_and_param_subsets(obe, d):
    n = 300_001
    pdf = obe.ParticlePDF(_cloud(n, d, d), seed=1)
    w = np.random.default_rng(d).random(n)
    pdf.particle_weights = w / w.sum()
    levels = (0.1, 0.5, 0.9)
    full = pdf.quantile(levels)
    assert full.shape == (d, 3)
    for r in range(d):
        np.testing.assert_array_equal(_bits(pdf.quantile(levels, params=r)), _bits(full[r:r + 1]))
        np.testing.assert_array_equal(_bits(pdf.quantile(levels, params=[r, 0])), _bits(full[[r, 0]]))
    assert pdf.quantile(0.5).shape == (d, 1)
    m, e = pdf.histogram(4096, range=(-1.0, 6.0), params=[0])
    raw, _ = orc.histogram(pdf.particles[0], orc.quantised(pdf.particle_weights), e[0])
    np.testing.assert_array_equal(_bits(m[0]), _bits(orc.mass(raw)))
    if d >= 2:                                             # 65536 bins: several shared-memory windows
        m2, xe, ye, c2 = pdf.histogram2d(1, 0, (256, 256), range=[[-2100, -300], [0, 6]], return_counts=True)
        raw2, cnt2 = orc.histogram2d(pdf.particles[1], pdf.particles[0], orc.quantised(pdf.particle_weights), xe, ye)
        np.testing.assert_array_equal(_bits(m2), _bits(orc.mass(raw2)))
        np.testing.assert_array_equal(c2, cnt2)


def _lorentz_engine(obe, n, seed=11, **kw):
    g = np.random.default_rng(3)
    prior = np.array([g.uniform(2, 4, n), g.uniform(-2000, -400, n), g.normal(50000, 1000, n)])
    return obe.OptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 400),), prior, (0.1,), scale=False,
                            default_noise_std=500.0, seed=seed, **kw)


def _measure(x, meas):
    return 50400.0 - 1200.0 / (((x[0] - 3.14) / 0.1) ** 2 + 1) + 500.0 * meas.standard_normal()


def test_broad_and_peaked_cloud(obe):
    eng = _lorentz_engine(obe, 1_000_000)
    _check_all(eng)                                        # broad prior
    meas = np.random.default_rng(9)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(30):
            x = eng.opt_setting()
            eng.pdf_update((x, _measure(x, meas), 500.0))
    q = _check_all(eng, levels=(0.025, 0.5, 0.975))       # sharply peaked
    assert q[0, 2] - q[0, 0] < 1.0


def test_ties_beyond_the_gather_cap(obe):
    n = 200_000
    g = np.random.default_rng(4)
    x = g.normal(0.0, 1.0, (2, n))
    x[0, :50_000] = 0.25                                   # 50k particles share one value (cap is 4096)
    x[1, ::3] = -0.0
    x[1, 1::3] = 0.0
    pdf = obe.ParticlePDF(x, seed=2)
    w = g.random(n)
    pdf.particle_weights = w / w.sum()
    levels = np.linspace(0, 1, 16)
    got = _check_all(pdf, levels)
    assert np.any(got[0] == 0.25)
    assert np.any((got[1] == 0.0) & ~np.signbit(got[1]))
    one = obe.ParticlePDF(np.full((1, 10_000), 1.5), seed=2)   # all particles at one value
    np.testing.assert_array_equal(one.quantile(levels), np.full((1, 16), 1.5))
    m, e = one.histogram(10)
    np.testing.assert_array_equal(e[0], np.histogram_bin_edges([1.5], 10))
    assert m[0, 5] == orc.mass(orc.quantised(one.particle_weights).sum(dtype=np.uint64).reshape(1))[0]


def test_repeatable_and_read_only(obe):
    eng = _lorentz_engine(obe, 2_000_001)
    w = np.random.default_rng(1).random(eng.n_particles)
    eng.particle_weights = w / w.sum()
    before = (eng.particles.copy(), eng.particle_weights.copy(), eng._buf.stats.cpu().numpy().copy(),
              eng._buf.weights.cpu().numpy().copy(), eng.rng.bit_generator.state)
    a = (eng.quantile((0.1, 0.5)), eng.histogram(256), eng.histogram2d(0, 2, 128))
    b = (eng.quantile((0.1, 0.5)), eng.histogram(256), eng.histogram2d(0, 2, 128))
    np.testing.assert_array_equal(_bits(a[0]), _bits(b[0]))
    for u, v in zip(a[1] + a[2], b[1] + b[2]):
        np.testing.assert_array_equal(_bits(u), _bits(v))
    after = (eng.particles, eng.particle_weights, eng._buf.stats.cpu().numpy(), eng._buf.weights.cpu().numpy(),
             eng.rng.bit_generator.state)
    for u, v in zip(before[:4], after[:4]):
        np.testing.assert_array_equal(_bits(u), _bits(v))
    assert before[4] == after[4]


@pytest.mark.parametrize('async_update', [False, True])
def test_closed_loop_is_unchanged_by_summaries(obe, async_update):
    n, cycles = 200_000, 40
    a, b = _lorentz_engine(obe, n), _lorentz_engine(obe, n)
    for e in (a, b):
        e.eager_select = True
        e.async_update = async_update
    ma, mb = np.random.default_rng(9), np.random.default_rng(9)
    pending = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        xa, xb = a.opt_setting(), b.opt_setting()
        for t in range(cycles):
            assert xa == xb and a.last_setting_index == b.last_setting_index, f'cycle {t}'
            a.pdf_update((xa, _measure(xa, ma), 500.0))
            b.pdf_update((xb, _measure(xb, mb), 500.0))
            pending += int(a._pending_cycle)
            (lambda: a.quantile((0.1, 0.5, 0.9)), lambda: a.histogram(64), lambda: a.histogram2d(0, 1, 32))[t % 3]()
            xa, xb = a.opt_setting(), b.opt_setting()
    if async_update:
        assert pending > 0, 'no pending device-resample cycle was summarised'
    np.testing.assert_array_equal(_bits(a.particles), _bits(b.particles))
    np.testing.assert_array_equal(_bits(a.particle_weights), _bits(b.particle_weights))


def test_1e8_particles_against_the_oracle(obe):
    n = 100_000_000
    import torch
    eng = obe.ParticlePDF(np.zeros((3, 1)), seed=1)
    g = torch.Generator(device='cuda').manual_seed(7)
    cloud = torch.randn((3, n), generator=g, device='cuda', dtype=torch.float64)
    cloud[1] = cloud[1] * 0.01 + 2.0
    eng.set_pdf(cloud)
    w = torch.rand(n, generator=g, device='cuda', dtype=torch.float64)
    eng.particle_weights = (w / w.sum()).cpu().numpy()
    levels = (0.025, 0.5, 0.975)
    got = eng.quantile(levels)
    mass, edges = eng.histogram(256)
    x, wts = eng.particles, eng.particle_weights
    np.testing.assert_array_equal(_bits(got), _bits(orc.quantiles(x, wts, levels)))
    wq = orc.quantised(wts)
    for r in range(3):
        raw, _ = orc.histogram(x[r], wq, edges[r])
        np.testing.assert_array_equal(_bits(mass[r]), _bits(orc.mass(raw)))


def test_c_level_errors(obe):
    from optbayesexpt_b200 import _lib
    pdf = obe.ParticlePDF(_cloud(1000, 2, 0), seed=0)
    lib, cs, st = pdf._lib, pdf._cs(), pdf._stream()
    out = np.empty(32)
    scratch = pdf._summary_scratch(lib.obe_quantile_scratch_bytes(2, 16))
    q = np.array([0.5, 0.2])

    def quant(params, levels):
        return lib.obe_quantile(cs, _lib.iarr(params), len(params), _lib.dptr(levels), len(levels), scratch,
                                _lib.dptr(out), st)

    assert quant([0, 1], q) == 0
    for params, levels, msg in [([2], q, b'out of range'), ([-1], q, b'out of range'),
                                ([0], np.array([1.5]), b'[0, 1]'), ([0], np.array([np.nan]), b'[0, 1]'),
                                ([0], np.zeros(17), b'n_q')]:
        assert quant(params, levels) != 0
        assert msg in lib.obe_last_error()
    raw = np.empty(8192, dtype=np.uint64)
    up = raw.ctypes.data_as(C.POINTER(C.c_uint64))
    for edges, bins, msg in [(np.linspace(0, 1, 4098), 4097, b'bins'), (np.array([1.0, 0.5, 2.0]), 2, b'decrease'),
                             (np.array([1.0, 1.0]), 1, b'increase'), (np.array([0.0, np.inf]), 1, b'finite')]:
        assert lib.obe_histogram(cs, _lib.iarr([0]), 1, _lib.dptr(edges), bins, scratch, up, None, st) != 0
        assert msg in lib.obe_last_error()
    e = np.linspace(0, 1, 5)
    assert lib.obe_histogram2d(cs, 0, 1, _lib.dptr(np.linspace(0, 1, 300)), 299, _lib.dptr(np.linspace(0, 1, 301)),
                               300, scratch, up, None, st) != 0
    assert b'65536' in lib.obe_last_error()
    pdf.particle_weights = np.zeros(1000)                  # empty posterior
    for call in (lambda: quant([0], q), lambda: lib.obe_histogram(cs, _lib.iarr([0]), 1, _lib.dptr(e), 4, scratch,
                                                                  up, None, st)):
        assert call() != 0
        assert b'empty' in lib.obe_last_error()
    with pytest.raises(_lib.ObeError, match='empty'):
        pdf.quantile(0.5)
    pdf.particle_weights = np.ones(1000)                   # stored as given: the weights sum to 1000
    for call in (lambda: pdf.quantile(0.5), lambda: pdf.histogram(8), lambda: pdf.histogram(8, range=(0, 1)),
                 lambda: pdf.histogram2d(0, 1, 8, range=[[0, 1], [0, 1]])):
        with pytest.raises(_lib.ObeError, match='sum to 4 or more'):
            call()


def test_eight_parameters_and_ranges_that_cut_the_cloud(obe):
    # d = 8: 8 x 16 (parameter, level) pairs share the refinement passes (128 sub-bins each, up to 10 passes), and a
    # 4096-bin histogram of all 8 rows takes two launches of 4 rows each
    n = 500_003
    g = np.random.default_rng(8)
    x = g.normal(size=(8, n)) * np.arange(1, 9)[:, None] + np.arange(8)[:, None]
    x[3, :1000] = 7.0                                      # ties across the gather cap's neighbourhood
    pdf = obe.ParticlePDF(x, seed=8)
    w = g.exponential(size=n)
    pdf.particle_weights = w / w.sum()
    wq = orc.quantised(pdf.particle_weights)
    levels = np.linspace(0.0, 1.0, 16)
    np.testing.assert_array_equal(_bits(pdf.quantile(levels)), _bits(orc.quantiles(pdf.particles, pdf.particle_weights,
                                                                                     levels)))
    assert pdf._lib.obe_summary_passes() >= 3
    mass, edges, counts = pdf.histogram(4096, range=(-1.0, 2.0), return_counts=True)
    assert pdf._lib.obe_summary_passes() == 2
    for r in range(8):
        raw, cnt = orc.histogram(pdf.particles[r], wq, edges[r])
        np.testing.assert_array_equal(_bits(mass[r]), _bits(orc.mass(raw)))
        np.testing.assert_array_equal(counts[r], cnt)
    assert counts.sum() < 8 * n // 2                       # the range drops most of the cloud
    ranges = [(r - 0.5, r + 0.25) for r in range(8)]       # one range per parameter
    mass, edges = pdf.histogram(100, range=ranges)
    for r in range(8):
        np.testing.assert_array_equal(edges[r], np.histogram_bin_edges(np.empty(0), 100, range=ranges[r]))
        np.testing.assert_array_equal(_bits(mass[r]), _bits(orc.mass(orc.histogram(pdf.particles[r], wq, edges[r])[0])))
    m2, xe, ye, c2 = pdf.histogram2d(2, 5, (40, 30), range=[[1.0, 2.5], [4.0, 6.0]], return_counts=True)
    raw2, cnt2 = orc.histogram2d(pdf.particles[2], pdf.particles[5], wq, xe, ye)
    np.testing.assert_array_equal(_bits(m2), _bits(orc.mass(raw2)))
    np.testing.assert_array_equal(c2, cnt2)
    assert 0 < c2.sum() < n // 4
