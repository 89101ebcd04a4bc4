"""Poisson, binomial and user (cuda_likelihood) measurement likelihoods in the fused update kernel.

Checked against the scipy restatement in oracle/likelihoods.py: the per-particle likelihood (1e-12 relative, log L
absolutely for large counts, edge cases exact), the update's weights and moments, a seeded closed loop with the
reference's multinomial resampling, and the agreement of every update path of the engine (synchronous, async_update,
the device-side resample test, run_cycle_async).  Also the refusals, and a Poisson Rabi experiment that finds its
parameters.
"""
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import likelihoods as olk
from oracle import obe_oracle as orc

pytestmark = pytest.mark.gpu

# a cuda_likelihood that restates the Poisson pmf: aux unused, lgamma computed per particle
USER_POISSON = r'''
__device__ double user_poisson(const double* y, const double* k, const double* aux, int n) {
    double ll = 0.0;
    for (int c = 0; c < n; ++c) {
        const double lam = y[c];
        if (!(lam >= 0.0)) return nan("");
        ll += ((k[c] == 0.0 ? 0.0 : k[c] * log(lam)) - lam) - lgamma(k[c] + 1.0);
    }
    return ll;
}
'''


def _user_poisson_log(y_model, k, aux):
    return olk.loglik_poisson(y_model, k)


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def user_lik(obe):
    return obe.cuda_likelihood(USER_POISSON, 'user_poisson')


def _line_prior(n, seed=3):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(0.0, 6.0, n), g.uniform(4.0, 14.0, n)])          # lambda = m x + b in [4, 20]


def _dip_prior(n, seed=3):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 0.8, n), g.uniform(0.2, 0.6, n)])   # p in [0.2, 1]


def _lik_engine(obe, kind, user_lik, n, **kw):
    """(engine, oracle model, prior, record, oracle likelihood of a y_model)"""
    if kind == 'binomial':
        prior = _dip_prior(n)
        eng = obe.OptBayesExpt('lorentzian_dip', (np.linspace(1.5, 4.5, 64),), prior, (), likelihood_model='binomial',
                               scale=False, **kw)
        return eng, orc.model_lorentzian_dip, prior, ((3.1,), 41.0, 60.0), \
            lambda y, rec, choke=None: olk.likelihood_binomial(y, rec[1], rec[2], choke)
    prior = _line_prior(n)
    lm = 'poisson' if kind == 'poisson' else user_lik
    eng = obe.OptBayesExpt('line', (np.linspace(0.0, 1.0, 64),), prior, (), likelihood_model=lm, scale=False, **kw)
    return eng, orc.model_line, prior, ((0.7,), 11.0, 0.0), \
        lambda y, rec, choke=None: olk.likelihood_poisson(y, rec[1], choke)


def wclose(actual, desired, rtol=1e-12, msg=''):
    assert_allclose(actual, desired, rtol=rtol, atol=1e-15 * np.max(np.abs(desired)), err_msg=msg)


def cov_close(actual, desired, tol):
    sd = np.sqrt(np.diag(desired))
    err = np.abs(actual - desired) / np.outer(sd, sd)
    assert err.max() < tol, f'covariance off by {err.max():.3g} (correlation units)'


# ---------------------------------------------------------------------------------------------------------------
# likelihood() against scipy
# ---------------------------------------------------------------------------------------------------------------
def test_poisson_likelihood_matches_scipy(obe):
    from scipy.special import gammaln
    lam = np.concatenate([[0.0, -1.0, -1e-300, np.nan, np.inf, 1e-300, 1e-3, 0.5],
                          np.linspace(0.1, 50.0, 200), np.linspace(9.9e5, 1.01e6, 50)])
    n = len(lam)
    eng = obe.OptBayesExpt('line', (np.linspace(0, 1, 5),), _line_prior(n), (), likelihood_model='poisson')
    for k in (0.0, 1.0, 7.0, 40.0, 1e6):
        got = eng.likelihood(lam[None, :], ((0.5,), k))
        want = olk.likelihood_poisson((lam,), k)
        big = want > 1e-300
        if k < 1e3:
            assert_allclose(got[big], want[big], rtol=1e-12, err_msg=f'k={k}')
        else:                                                   # log L absolutely, scaled by its largest term
            ll_want = olk.loglik_poisson((lam,), k)
            scale = np.maximum.reduce([np.abs(k * np.log(np.abs(lam) + 1e-300)), np.abs(lam),
                                       np.full(n, gammaln(k + 1.0))])
            with np.errstate(divide='ignore'):
                ll_got = np.log(got)
            assert np.all(np.abs(ll_got[big] - ll_want[big]) <= 1e-13 * scale[big]), f'k={k}'
        assert np.all(got[~big] <= 1e-290)
        # edge cases exact
        assert got[1] == 0.0 and got[2] == 0.0 and got[3] == 0.0, 'lambda < 0 / NaN must give weight 0'
        assert got[4] == 0.0, 'lambda = +inf must give weight 0'
        assert got[0] == (1.0 if k == 0 else 0.0), 'L(0 | 0) = 1, L(k > 0 | 0) = 0'
    # the third element of a Poisson record is ignored; choke is exp(choke log L)
    eng.choke = 0.25
    got = eng.likelihood(lam[None, :], ((0.5,), 7.0, 123.0))
    want = olk.likelihood_poisson((lam,), 7.0, choke=0.25)
    big = want > 1e-300
    assert_allclose(got[big], want[big], rtol=1e-12)


def test_binomial_likelihood_matches_scipy(obe):
    from scipy.stats import binom
    p = np.concatenate([[0.0, 1.0, -1e-17, 1.0 + 2e-16, np.nan, np.inf, -np.inf, 1e-300, 1.0 - 1e-16],
                        np.linspace(1e-3, 1 - 1e-3, 300)])
    n = len(p)
    eng = obe.OptBayesExpt('lorentzian_dip', (np.linspace(1, 2, 5),), _dip_prior(n), (), likelihood_model='binomial')
    for k, nt in ((0.0, 0.0), (0.0, 10.0), (10.0, 10.0), (3.0, 10.0), (37.0, 100.0), (5e5, 1e6)):
        got = eng.likelihood(p[None, :], ((1.5,), k, nt))
        want = olk.likelihood_binomial((p,), k, nt)
        big = want > 1e-300
        if nt < 1e3:
            assert_allclose(got[big], want[big], rtol=1e-12, err_msg=f'k={k} n={nt}')
            ref = binom.pmf(k, nt, p[9:])
            assert_allclose(got[9:][ref > 1e-300], ref[ref > 1e-300], rtol=1e-11)
        else:
            ll_want = olk.loglik_binomial((p,), k, nt)
            with np.errstate(divide='ignore'):
                ll_got = np.log(got)
            assert np.all(np.abs(ll_got[big] - ll_want[big]) <= 1e-13 * 1.4e7)
        assert got[2] == 0.0 and got[3] == 0.0 and got[4] == 0.0 and got[5] == 0.0 and got[6] == 0.0, \
            'p outside [0, 1] or NaN must give weight 0'
        assert got[0] == (1.0 if k == 0 else 0.0), 'p = 0'
        assert got[1] == (1.0 if k == nt else 0.0), 'p = 1'


def test_user_likelihood_matches_oracle(obe, user_lik):
    lam = np.concatenate([[0.0, -1.0, np.nan], np.linspace(0.1, 50.0, 200)])
    eng = obe.OptBayesExpt('line', (np.linspace(0, 1, 5),), _line_prior(len(lam)), (), likelihood_model=user_lik)
    for k in (0.0, 3.0, 30.0):
        got = eng.likelihood(lam[None, :], ((0.5,), k, 1.0))
        want = olk.likelihood_poisson((lam,), k)
        big = want > 1e-300
        assert_allclose(got[big], want[big], rtol=1e-12)
        assert got[1] == 0.0 and got[2] == 0.0


# ---------------------------------------------------------------------------------------------------------------
# pdf_update against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['poisson', 'binomial', 'user'])
@pytest.mark.parametrize('n', [1, 2047, 2048, 2049, 100_000, 1_000_000])
def test_update_matches_oracle(obe, user_lik, kind, n):
    eng, model, prior, rec, lik = _lik_engine(obe, kind, user_lik, n)
    eng.tuning_parameters['auto_resample'] = False
    w0 = np.ones(n) / n
    w1 = orc.normalized_product(w0, lik((model(rec[0], prior, ()),), rec))
    eng.pdf_update(rec)
    wclose(eng.particle_weights, w1, 1e-12, 'first update')
    rec2 = (rec[0], rec[1] + 2.0, rec[2] + 2.0)
    w2 = orc.normalized_product(w1, lik((model(rec2[0], prior, ()),), rec2))
    eng.pdf_update(rec2)
    wclose(eng.particle_weights, w2, 1e-12, 'second update')
    assert_allclose(eng.n_eff(), orc.n_effective(w2), rtol=1e-12)
    if n > 1:
        assert_allclose(eng.mean(), orc.weighted_mean(prior, w2), rtol=1e-12)
        cov_close(eng.covariance(), orc.weighted_covariance_longdouble(prior, w2), 1e-12)


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_prefetched_and_supplied_model_equal_fused_update(obe, user_lik, kind):
    n = 30_000
    a, model, prior, rec, _ = _lik_engine(obe, kind, user_lik, n)
    b = _lik_engine(obe, kind, user_lik, n)[0]
    c = _lik_engine(obe, kind, user_lik, n)[0]
    for e in (a, b, c):
        e.tuning_parameters['auto_resample'] = False
    a.pdf_update(rec)
    b.prefetch_model(rec[0])
    b.pdf_update(rec)
    c.pdf_update(rec, y_model_data=model(rec[0], prior, ())[None, :])
    assert_array_equal(a.particle_weights, b.particle_weights)
    wclose(c.particle_weights, a.particle_weights, 1e-12)


# ---------------------------------------------------------------------------------------------------------------
# closed loops
# ---------------------------------------------------------------------------------------------------------------
def _rabi_truth(setting):
    return orc.model_rabi(setting, (3.3, 1.7), (100.0, 0.9, 0.5))


def _rabi_prior(n, seed=1001):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])


RABI_SETTINGS = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))


@pytest.mark.parametrize('kind', ['poisson', 'user'])
def test_closed_loop_multinomial_matches_oracle(obe, user_lik, kind):
    """40 cycles of a Poisson Rabi experiment with the reference's multinomial resampling: every chosen setting and
    resample decision identical to the oracle, weights 1e-12 before the first resample and condition-aware after."""
    n, cycles = 5000, 40
    prior = _rabi_prior(n)
    lm = 'poisson' if kind == 'poisson' else user_lik
    eng = obe.OptBayesExpt('rabi', RABI_SETTINGS, prior, (100.0, 0.9, 0.5), likelihood_model=lm, scale=False,
                           default_noise_std=10.0, resampling='multinomial', use_jit=False)
    eng.rng = np.random.default_rng(1003)
    ora = olk.OracleOBELik(orc.model_rabi, RABI_SETTINGS, prior, (100.0, 0.9, 0.5), default_noise_std=10.0,
                           scale=False, rng=np.random.default_rng(1003),
                           likelihood_model='poisson' if kind == 'poisson' else _user_poisson_log)
    meas = np.random.default_rng(1002)
    seen, fired = False, 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(cycles):
            x = eng.opt_setting()
            xo = ora.opt_setting()
            assert eng.last_setting_index == ora.last_setting_index, f'setting index differs at cycle {t}'
            assert x == xo
            k = float(meas.poisson(_rabi_truth(x)))
            rec = (x, k) if t % 2 and kind == 'poisson' else (x, k, 0.0)
            eng.pdf_update(rec)
            ora.pdf_update((x, k, 0.0))
            assert eng.just_resampled == ora.just_resampled, f'resample decision differs at cycle {t}'
            fired += int(eng.just_resampled)
            if not seen and not eng.just_resampled:
                wclose(eng.particle_weights, ora.particle_weights, 1e-12, f'weights t={t}')
            seen = seen or eng.just_resampled
            tol = 1e-9 if seen else 1e-12
            assert_allclose(eng.mean(), ora.mean(), rtol=tol, err_msg=f'mean t={t}')
            cov_close(eng.covariance(), ora.covariance(), max(tol, 1e-9))
    assert fired >= 2


class ScriptedRng:
    """random() -> the u0 of cycle t, random(k) -> the K uniforms of cycle t (as in test_gpu_device_test.py)."""

    def __init__(self, seed, cycles, k):
        g = np.random.default_rng(seed)
        self.u0 = g.random(cycles + 1)
        self.uk = g.random((cycles + 1, k))
        self.t = 0

    def random(self, size=None):
        if size is None:
            return self.u0[self.t]
        return self.uk[self.t, :size].copy()


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_update_paths_agree(obe, kind):
    """Synchronous pdf_update, async_update, the device-side resample test and run_cycle_async: identical decisions,
    settings, particles and weights given the same random numbers."""
    n, cycles = 50_000, 30
    prior = _rabi_prior(n)
    cons = (100.0, 0.9, 0.5) if kind == 'poisson' else (1.0, 0.9, 0.5)    # binomial: the model is a probability
    engines = []
    for _ in range(4):
        e = obe.OptBayesExpt('rabi', RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False,
                             default_noise_std=10.0 if kind == 'poisson' else 0.05, seed=11)
        e.rng = ScriptedRng(5, cycles, 30)
        engines.append(e)
    sync, asy, dev, cyc = engines
    sync.eager_select = True
    asy.eager_select = asy.async_update = True
    asy.device_resample_test = False
    asy.tuning_parameters['resample_threshold'] = 2.0          # (a decision known without N_eff: the async path)
    dev.eager_select = dev.async_update = True
    assert dev._device_test_ok()
    meas = np.random.default_rng(9)

    def record(x):
        mu = orc.model_rabi(x, (3.3, 1.7), cons)
        if kind == 'poisson':
            return (x, float(meas.poisson(mu)))
        return (x, float(meas.binomial(100, mu)), 100.0)

    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        x = [e.opt_setting() for e in engines]
        fired = 0
        for t in range(cycles):
            for e in engines:
                e.rng.t = t + 1
            assert x[0] == x[2] == x[3], f'cycle {t}'
            rec = record(x[0])
            sync.pdf_update(rec)
            dev.pdf_update(rec)
            asy.pdf_update((x[1],) + rec[1:])
            assert asy.just_resampled
            cyc.run_cycle_async(rec, resample=sync.just_resampled, select=True)
            x = [e.opt_setting() for e in engines[:3]]
            ic = int(cyc.best_index_dev.cpu()[0])
            x.append(tuple(cyc.allsettings[:, ic]))
            assert sync.just_resampled == dev.just_resampled, f'cycle {t}'
            assert sync.last_setting_index == dev.last_setting_index == ic, f'cycle {t}'
            fired += int(sync.just_resampled)
    assert 2 <= fired < cycles
    assert_array_equal(dev.particles, sync.particles, err_msg='device resample test')
    assert_array_equal(dev.particle_weights, sync.particle_weights, err_msg='device resample test')
    # run_cycle_async: same decisions and settings (above); the cloud agrees to rounding (the moment pivot of the
    # asynchronous entry lags one update, which moves the last bits of the Liu-West centre)
    assert_allclose(cyc.particles, sync.particles, rtol=1e-13, err_msg='run_cycle_async')
    assert_allclose(cyc.particle_weights, sync.particle_weights, rtol=1e-12, err_msg='run_cycle_async')
    # async_update (forced resample every cycle) against the synchronous path with the same forced decision
    ref = obe.OptBayesExpt('rabi', RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False, seed=11,
                           default_noise_std=10.0 if kind == 'poisson' else 0.05, resample_threshold=2.0)
    a2 = obe.OptBayesExpt('rabi', RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False, seed=11,
                          default_noise_std=10.0 if kind == 'poisson' else 0.05, resample_threshold=2.0)
    a2.async_update = True
    for e in (ref, a2):
        e.rng = np.random.default_rng(77)
    meas = np.random.default_rng(10)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(8):
            xr, xa = ref.opt_setting(), a2.opt_setting()
            assert xr == xa, f'cycle {t}'
            rec = record(xr)
            ref.pdf_update(rec)
            a2.pdf_update(rec)
    assert_array_equal(a2.particles, ref.particles)
    assert_array_equal(a2.particle_weights, ref.particle_weights)


def test_poisson_rabi_finds_its_parameters(obe):
    n = 200_000
    eng = obe.OptBayesExpt('rabi', RABI_SETTINGS, _rabi_prior(n), (100.0, 0.9, 0.5), likelihood_model='poisson',
                           default_noise_std=10.0)
    meas = np.random.default_rng(7)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(300):
            x = eng.opt_setting()
            eng.pdf_update((x, float(meas.poisson(_rabi_truth(x)))))
    m, s = eng.mean(), eng.std()
    assert abs(m[0] - 3.3) < 3 * s[0] and abs(m[1] - 1.7) < 3 * s[1], (m, s)
    assert s[0] < 0.5 and s[1] < 0.5, s


# ---------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------
def test_refusals(obe):
    from optbayesexpt_b200._lib import ObeError
    n = 4096
    prior = _line_prior(n)
    settings = (np.linspace(0, 1, 16),)
    eng = obe.OptBayesExpt('line', settings, prior, (), likelihood_model='poisson')
    for bad in ((0.5,), -1.0), ((0.5,), np.nan), ((0.5,), np.inf), ((0.5,), 2.5):
        with pytest.raises(ValueError):
            eng.pdf_update(bad)
    beng = obe.OptBayesExpt('lorentzian_dip', settings, _dip_prior(n), (), likelihood_model='binomial')
    for bad in (((1.5,), 11.0, 10.0), ((1.5,), -1.0, 10.0), ((1.5,), 1.0, np.inf), ((1.5,), 1.0)):
        with pytest.raises(ValueError):
            beng.pdf_update(bad)
    with pytest.raises(ValueError):
        obe.OptBayesExpt('line', settings, prior, (), likelihood_model='gamma')
    with pytest.raises(TypeError):
        obe.OptBayesExpt('line', settings, prior, (), likelihood_model=3)
    np_prior = np.vstack([prior, np.full(n, 1.0)])
    with pytest.raises(ValueError, match='noise parameter'):
        obe.OptBayesExptNoiseParameter('line', settings, np_prior, (), noise_parameter_index=2,
                                       likelihood_model='poisson')
    with pytest.raises(ValueError, match='Gaussian'):
        obe.OptBayesExptSweeper('line', settings, np_prior, (), noise_parameter_index=2, likelihood_model='poisson')
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    with pytest.raises(ValueError, match='Gaussian'):
        BatchedOptBayesExpt(obe.builtin('line').with_likelihood('poisson'), settings, prior, ())
    from optbayesexpt_b200.sharded import ShardedOptBayesExpt
    with pytest.raises(ValueError, match='Gaussian'):
        ShardedOptBayesExpt('line', settings, prior, (), likelihood_model='poisson')

    class Overrides(obe.OptBayesExpt):
        def likelihood(self, y_model, measurement_record):
            return np.ones(1)

    with pytest.raises(TypeError, match='cuda_likelihood'):
        Overrides('line', settings, prior, ())
    # a compile error in a user likelihood surfaces its log
    broken = obe.cuda_likelihood('__device__ double broken(const double* y, const double* m, const double* a, int n) '
                                 '{ return undeclared_name; }', 'broken')
    with pytest.raises(ObeError, match='undeclared_name'):
        obe.OptBayesExpt('line', settings, prior, (), likelihood_model=broken)
    # the C entries that take no non-Gaussian handle
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    h = eng._model
    rc = lib.obe_update_multi(h, eng._cs(), None, None, 1, None, None, 1, None, 0, 0.0, 0.0, n, None, None, None)
    assert rc != 0
    rc = lib.obe_update_multi(h, eng._cs(), 16, 16, 1, None, None, 1, None, 0, 0.0, 0.0, n, 16, 16, None)
    assert rc != 0 and b'non-Gaussian' in lib.obe_last_error()
