"""The random-walk drift on the device: the kernel against numpy with its own normals (and those against the oracle's
restated keying), what it must leave alone, the constraint masks, the default path, the agreement of every update
path, the covariance it adds, and a drifting Lorentzian peak that only a matched drift can follow."""
import ctypes as C
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import drift as odr
from oracle import obe_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


def _np(t):
    return t.detach().cpu().numpy().copy()


def _drift_call(pdf, factor, pivot, seed, epoch, mask_le=0, mask_lt=0):
    """obe_drift on the live cloud of a ParticlePDF; returns the (d, n) normals it used."""
    import torch
    from optbayesexpt_b200 import _lib
    buf = pdf._buf
    z = torch.zeros((buf.d, buf.ld), dtype=torch.float64, device=buf.device)
    pdf._check(pdf._lib.obe_drift(pdf._cs(), _lib.darr(np.asarray(factor).reshape(-1)), mask_le, mask_lt, None, 0,
                                  _lib.darr(pivot, _lib.MAX_PARAMS), seed, epoch, C.c_void_p(z.data_ptr()),
                                  pdf._stream()))
    torch.cuda.synchronize()
    return _np(z)[:, :pdf.n_particles]


def _snapshot(pdf):
    b = pdf._buf
    return dict(p=_np(b.particles)[:, :pdf.n_particles], w=_np(b.weights)[:pdf.n_particles], ts=_np(b.tile_sums),
                tp=_np(b.tile_prefix), st=_np(b.stats))


def _factor(d, g):
    from optbayesexpt_b200.drift import drift_factor
    a = g.normal(size=(d, d)) * 0.05
    q = a @ a.T
    if d > 1:
        q[d // 2, :] = q[:, d // 2] = 0.0          # one parameter that does not drift
    return drift_factor(q, d), d // 2 if d > 1 else None


@pytest.mark.parametrize('implicit', [False, True])
@pytest.mark.parametrize('d', [1, 3, 8])
def test_kernel_parity_and_nothing_else_moves(obe, d, implicit):
    n, seed, epoch = 1_000_000, 0x1234567890ABCDEF, 17
    g = np.random.default_rng(d)
    prior = g.normal(size=(d, n)) + np.arange(1, d + 1)[:, None]
    pdf = obe.ParticlePDF(prior, seed=4)
    if implicit:
        pdf.resample()                                    # systematic resample: the weights become implicit
    else:
        pdf.particle_weights = g.uniform(0.0, 1.0, n)
    before = _snapshot(pdf)
    assert (before['st'][62] > 0.0) == implicit
    factor, fixed = _factor(d, g)
    pivot = before['p'].mean(axis=1)
    z = _drift_call(pdf, factor, pivot, seed, epoch)
    after = _snapshot(pdf)
    x = before['p']
    want = x + factor @ z
    assert_allclose(after['p'], want, rtol=1e-12, atol=1e-15)
    # float32 accuracy: the device's approximate log / sqrt / sincos against numpy's; the radius sqrt(-2 log u) of
    # a uniform u near 1 amplifies the absolute error of the log (~5e-7) to ~1e-6 / radius, hence the rare outliers
    dz = np.abs(z.T - odr.drift_normals(n, d, seed, epoch))
    assert dz.max() < 1e-3
    assert np.mean(dz > 1e-5) < 1e-4
    if fixed is not None:
        assert_array_equal(after['p'][fixed], x[fixed])
    # the weights and everything derived from them: bit for bit
    for key in ('w', 'ts', 'tp'):
        assert_array_equal(after[key], before[key], err_msg=key)
    from optbayesexpt_b200 import _lib
    same = [_lib.ST_TOTAL, _lib.ST_INVS, _lib.ST_SUMSQ, _lib.ST_NEFF, _lib.ST_SUMT, _lib.ST_NZERO, _lib.ST_UNIFORM,
            _lib.ST_FIRED]
    assert_array_equal(after['st'][same], before['st'][same])
    # the moments of the moved cloud
    t = np.full(n, before['st'][62]) if implicit else before['w']
    dx = after['p'] - pivot[:, None]
    st = after['st']
    assert_array_equal(st[_lib.ST_PIVOT:_lib.ST_PIVOT + d], pivot)
    m1 = (t * dx).sum(axis=1)
    assert_allclose(st[_lib.ST_M1:_lib.ST_M1 + d], m1, rtol=1e-12, atol=1e-12 * np.abs(t * dx).sum(axis=1).max())
    q = _lib.ST_M2
    for j in range(d):
        for k in range(j, d):
            terms = t * dx[j] * dx[k]
            assert_allclose(st[q], terms.sum(), rtol=1e-12, atol=1e-12 * np.abs(terms).sum())
            q += 1


def test_masks_reject_steps(obe):
    n, seed, epoch = 1_000_000, 99, 3
    g = np.random.default_rng(5)
    prior = np.array([g.uniform(0.0, 1.0, n), g.normal(size=n)])
    pdf = obe.ParticlePDF(prior, seed=1)
    factor = np.diag([0.5, 0.1])
    x = _snapshot(pdf)['p']
    z = _drift_call(pdf, factor, x.mean(axis=1), seed, epoch, mask_le=1)
    moved = _snapshot(pdf)['p']
    step = x + factor @ z
    rejected = step[0] <= 0.0
    assert rejected.sum() > 50_000
    assert np.all(moved[0] > 0.0)
    assert_array_equal(moved[:, rejected], x[:, rejected])
    assert_allclose(moved[:, ~rejected], step[:, ~rejected], rtol=1e-12, atol=1e-15)
    want, ok = odr.drift_step(x, factor, z.T, mask_le=1)
    assert_array_equal(ok, ~rejected)
    assert_allclose(moved, want, rtol=1e-12, atol=1e-15)


def _c1_engine(obe, n, **kw):
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc, n)
    return obe.OptBayesExpt(sc['model'], inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                            default_noise_std=500.0, seed=5, **kw), sc


def test_default_path_is_unchanged(obe):
    a, sc = _c1_engine(obe, 20_000)
    b, _ = _c1_engine(obe, 20_000, drift=None)
    meas = np.random.default_rng(3)
    fired = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(50):
            xa, xb = a.opt_setting(), b.opt_setting()
            assert a.last_setting_index == b.last_setting_index, f'cycle {t}'
            y = orc.model_lorentzian_hwhm(xa, sc['true_pars'], (0.1,)) + meas.normal(0, 500.0)
            a.pdf_update((xa, float(y), 500.0))
            b.pdf_update((xb, float(y), 500.0))
            assert a.just_resampled == b.just_resampled
            fired += int(a.just_resampled)
    assert fired >= 2
    assert_array_equal(_np(a._buf.stats), _np(b._buf.stats))
    assert_array_equal(a.particles, b.particles)
    assert_array_equal(a.particle_weights, b.particle_weights)


class ScriptedRng:
    """random() -> the u0 of cycle t, random(k) -> the K uniforms of cycle t (as in test_gpu_likelihood.py)."""

    def __init__(self, seed, cycles, k):
        g = np.random.default_rng(seed)
        self.u0 = g.random(cycles + 1)
        self.uk = g.random((cycles + 1, k))
        self.t = 0

    def random(self, size=None):
        if size is None:
            return self.u0[self.t]
        return self.uk[self.t, :size].copy()


RABI_SETTINGS = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))


@pytest.mark.parametrize('kind', ['gaussian', 'poisson'])
def test_update_paths_agree(obe, kind):
    """Under drift: the synchronous path, the device-side resample test (obe_cycle resample == 2), obe_cycle with the
    host's decision (resample 0 / 1) and the prefetched model pass take the same decisions and settings; the first
    two leave identical clouds and stats blocks, the other two agree to rounding (their moment pivot / model pass
    differ in the last bits, as without drift)."""
    n, cycles = 50_000, 30
    g = np.random.default_rng(1001)
    prior = np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])
    cons = (100.0, 0.9, 0.5)
    drift = [[0.02, 0.004], [0.004, 0.05]]
    engines = []
    for _ in range(4):
        kw = dict(likelihood_model='poisson') if kind == 'poisson' else {}
        e = obe.OptBayesExpt('rabi', RABI_SETTINGS, prior, cons, scale=False, default_noise_std=10.0, seed=11,
                             drift=drift, **kw)
        e.rng = ScriptedRng(5, cycles, 30)
        engines.append(e)
    sync, dev, cyc, pre = engines
    dev.eager_select = dev.async_update = True
    assert dev._device_test_ok()
    meas = np.random.default_rng(9)
    truth = np.array([3.3, 1.7])

    def record(x):
        mu = orc.model_rabi(x, truth, cons)
        if kind == 'poisson':
            return (x, float(meas.poisson(mu)))
        return (x, float(mu + meas.normal(0, 10.0)), 10.0)

    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        x = [e.opt_setting() for e in engines]
        fired = 0
        for t in range(cycles):
            for e in engines:
                e.rng.t = t + 1
            assert x[0] == x[1] == x[2] == x[3], f'cycle {t}'
            rec = record(x[0])
            sync.pdf_update(rec)
            dev.pdf_update(rec)
            pre.prefetch_model(rec[0])
            pre.pdf_update(rec)
            cyc.run_cycle_async(rec, resample=sync.just_resampled, select=True)
            x = [sync.opt_setting(), dev.opt_setting()]
            ic = int(cyc.best_index_dev.cpu()[0])
            x.append(tuple(cyc.allsettings[:, ic]))
            x.append(pre.opt_setting())
            assert sync.just_resampled == dev.just_resampled == pre.just_resampled, f'cycle {t}'
            assert sync.last_setting_index == dev.last_setting_index == ic == pre.last_setting_index, f'cycle {t}'
            fired += int(sync.just_resampled)
            assert_array_equal(_np(dev._buf.stats)[:63], _np(sync._buf.stats)[:63], err_msg=f'stats, cycle {t}')
        # the drift moved the clouds: the steps are part of what has to agree
        assert sync._drift_epoch == dev._drift_epoch == cyc._drift_epoch == pre._drift_epoch == cycles
    assert 2 <= fired < cycles
    assert_array_equal(dev.particles, sync.particles)
    assert_array_equal(dev.particle_weights, sync.particle_weights)
    for other, name in ((cyc, 'run_cycle_async'), (pre, 'prefetched')):
        assert_allclose(other.particles, sync.particles, rtol=1e-12, err_msg=name)
        assert_allclose(other.particle_weights, sync.particle_weights, rtol=1e-10, err_msg=name)
        assert_allclose(other.mean(), sync.mean(), rtol=1e-12, err_msg=name)


def test_covariance_grows_by_q(obe):
    """Uninformative records: the weights stay uniform and every cycle adds Q to the covariance (a full Q with
    correlations: F^T F in place of F F^T would fail)."""
    n, cycles = 1_000_000, 20
    g = np.random.default_rng(8)
    prior = g.normal(size=(3, n)) * 0.05 + np.array([[3.0], [1.0], [-2.0]])
    q = np.array([[0.010, 0.006, -0.003], [0.006, 0.008, 0.002], [-0.003, 0.002, 0.005]])
    eng = obe.OptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 50),), prior, (0.1,), seed=3, drift=q)
    c0 = eng.covariance()
    for _ in range(cycles):
        eng.pdf_update(((3.0,), 0.0, 1e12))
        assert not eng.just_resampled
    grown = eng.covariance() - c0
    total = c0 + cycles * q
    tol = 6.0 * np.sqrt(np.outer(np.diag(total), np.diag(total)) * 2.0 / n)
    assert np.all(np.abs(grown - cycles * q) < tol), (grown, cycles * q, tol)
    # and the moments the pass wrote are the cloud's
    assert_allclose(eng.mean(), eng.particles.mean(axis=1), rtol=1e-9)


def test_matched_drift_tracks_a_moving_peak(obe):
    """A Lorentzian peak whose centre takes a Gaussian random walk: with the matched drift the estimate stays within
    3 std of the truth at least 90 % of the last 100 cycles; without drift the cloud collapses and loses it."""
    n, cycles, step = 100_000, 300, 0.004
    settings = (np.linspace(1.5, 4.5, 200),)
    cons = (0.1,)
    truth_amp, truth_base, noise = -1200.0, 50400.0, 100.0
    walk = np.random.default_rng(21)
    centre = 3.0 + np.concatenate([[0.0], np.cumsum(walk.normal(0.0, step, cycles))])
    results = {}
    for label, drift in (('matched', [step, 0.0, 0.0]), ('static', None)):
        g = np.random.default_rng(22)
        prior = np.array([g.uniform(2, 4, n), g.uniform(-2000, -400, n), g.normal(50000, 1000, n)])
        eng = obe.OptBayesExpt('lorentzian_hwhm', settings, prior, cons, scale=False, default_noise_std=noise,
                               seed=23, drift=drift)
        meas = np.random.default_rng(24)
        z = []
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', RuntimeWarning)
            for t in range(cycles):
                x = eng.opt_setting()
                y = orc.model_lorentzian_hwhm(x, (centre[t], truth_amp, truth_base), cons) + meas.normal(0, noise)
                eng.pdf_update((x, float(y), noise))
                # after the update the cloud describes the centre at the next measurement
                z.append(abs(eng.mean()[0] - centre[t + 1]) / eng.std()[0])
        results[label] = np.array(z)
    assert np.mean(results['matched'][-100:] < 3.0) >= 0.9, results['matched'][-100:]
    assert results['static'][-1] > 10.0, results['static'][-10:]
