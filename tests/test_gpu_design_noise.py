"""Likelihood-aware setting selection (design_noise='likelihood') on the device.

The utility kernel of a likelihood-aware handle against oracle/design_noise.utility_likelihood_noise: bit for bit for
the rational built-ins (lorentzian_hwhm as Poisson rates, lorentzian_dip as binomial probabilities), 1e-12 for a user
likelihood and for rabi; every branch of the variance method (lanes 8 / 4 / 2 / 1, with and without the shared-memory
cache, K = 3 / 30 / 128), a two-channel model, max-min and pseudo, invalid outputs.  Then closed loops against the
oracle, the agreement of every selection path, a Gaussian engine (where 'likelihood' is 'fixed'), and the errors.
"""
import contextlib
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import design_noise as odn
from oracle import obe_oracle as orc

pytestmark = pytest.mark.gpu

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
__device__ double user_var(double y, double a) { return y >= 0.0 ? y * a : -1.0; }
'''


def _user_var(y, a):
    return np.where(y >= 0.0, y * a, -1.0)


# two channels, rational, non-contracted: numpy's bits
TWO_CH = r'''
__device__ void two_peaks(const double* s, const double* p, const double* c, double* y) {
    const double t = obe_div(obe_sub(s[0], p[0]), c[0]);
    y[0] = obe_add(p[2], obe_div(p[1], obe_add(obe_mul(t, t), 1.0)));
    y[1] = obe_add(p[2], obe_mul(p[1], obe_mul(s[0], 0.1)));
}
'''


def _two_peaks(sets, pars, cons):
    x, = sets
    x0, a, b = pars[:3]
    t = (x - x0) / cons[0]
    return np.array([b + a / (t * t + 1.0), b + a * (x * 0.1)])


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def models(obe):
    """One DeviceModel per model, so that every engine of the module reuses its compiled variants."""
    return dict(peak=obe.builtin('lorentzian_hwhm'), dip=obe.builtin('lorentzian_dip'), rabi=obe.builtin('rabi'),
                two=obe.cuda_source(TWO_CH, 'two_peaks', 1, 3, 1, 2),
                user=obe.cuda_likelihood(USER_POISSON, 'user_poisson', noise_var='user_var'))


@contextlib.contextmanager
def utility_options(lane_fill=50, cache=1):
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    lib.obe_set_option(b'utility_lane_fill', int(lane_fill))
    lib.obe_set_option(b'utility_cache', int(cache))
    try:
        yield
    finally:
        lib.obe_set_option(b'utility_lane_fill', 50)
        lib.obe_set_option(b'utility_cache', 1)


def _lane_fill(n_settings, lanes):
    """The utility_lane_fill percentage at which obe_utility gives a grid of n_settings `lanes` lanes (k >= 8)."""
    import torch
    resident = torch.cuda.get_device_properties(0).multi_processor_count * 8 * 256
    if lanes == 8:
        return 50 if n_settings * 8 * 100 <= resident * 50 else 100
    if lanes == 1:
        return 0
    f = -(-100 * n_settings * lanes // resident)
    assert n_settings * lanes <= resident * f // 100 < 2 * n_settings * lanes
    return f


def _peak_prior(n, seed=3, b_lo=2.0):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(b_lo, 10.0, n)])


def _dip_prior(n, seed=3, a_hi=0.8):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, a_hi, n), g.uniform(0.2, 0.6, n)])


def _case(obe, models, kind, n_settings, k=30, method='variance_approx', n=4096, **prior_kw):
    """(engine with rng seed 8, expected utility of its first selection)"""
    s = (np.linspace(1.5, 4.5, n_settings),)
    if kind == 'binomial':
        prior, cons, model, om, aux = _dip_prior(n, **prior_kw), (), models['dip'], orc.model_lorentzian_dip, 40.0
    else:
        prior, cons, model, om, aux = _peak_prior(n, **prior_kw), (0.3,), models['peak'], orc.model_lorentzian_hwhm, None
    lm, ok = (models['user'], _user_var) if kind == 'user' else (kind, kind)
    if kind == 'user':
        aux = 2.5
    eng = obe.OptBayesExpt(model, s, prior, cons, likelihood_model=lm, design_noise='likelihood', design_aux=aux,
                           n_draws=k, utility_method=method)
    eng.rng = np.random.default_rng(8)
    draws, _ = orc.randdraw(prior, np.ones(n) / n, np.random.default_rng(8).random(k))
    _, ys = orc.yvar_from_draws(om, orc.make_allsettings(s), draws, cons, 1)
    om_method = {'variance_approx': 'variance', 'max_min': 'max_min', 'pseudo_utility': 'pseudo'}[method]
    return eng, odn.utility_likelihood_noise(ys, ok, aux, method=om_method)


# ---------------------------------------------------------------------------------------------------------------
# the utility against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('k', [3, 30, 128])
@pytest.mark.parametrize('branch', ['lanes8', 'lanes4', 'lanes2', 'lanes1_cache', 'lanes1_nocache'])
@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_variance_bit_exact(obe, models, kind, branch, k):
    n_settings = 2000
    lanes = int(branch[5])
    with utility_options(_lane_fill(n_settings, lanes), 0 if branch.endswith('nocache') else 1):
        eng, want = _case(obe, models, kind, n_settings, k=k)
        got = eng.utility()
        assert_array_equal(got, want)
        eng.rng = np.random.default_rng(8)
        eng.opt_setting()
    assert eng.last_setting_index == orc.opt_index(want)
    assert np.all(want > 0)


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_large_grid(obe, models, kind):
    eng, want = _case(obe, models, kind, 300_000)
    assert_array_equal(eng.utility(), want)


def test_user_likelihood(obe, models):
    for branch in ('lanes8', 'lanes1_cache'):
        with utility_options(_lane_fill(2000, int(branch[5]))):
            eng, want = _case(obe, models, 'user', 2000)
            assert_allclose(eng.utility(), want, rtol=1e-12, atol=0)


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_rabi(obe, models, kind):
    n, k = 20_000, 30
    s = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))
    g = np.random.default_rng(5)
    prior = np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])
    cons = (100.0, 0.9, 0.5) if kind == 'poisson' else (1.0, 0.9, 0.5)
    aux = None if kind == 'poisson' else 50.0
    eng = obe.OptBayesExpt(models['rabi'], s, prior, cons, likelihood_model=kind, design_noise='likelihood',
                           design_aux=aux)
    eng.rng = np.random.default_rng(8)
    draws, _ = orc.randdraw(prior, np.ones(n) / n, np.random.default_rng(8).random(k))
    _, ys = orc.yvar_from_draws(orc.model_rabi, orc.make_allsettings(s), draws, cons, 1)
    want = odn.utility_likelihood_noise(ys, kind, aux)
    assert_allclose(eng.utility(), want, rtol=1e-12, atol=1e-12 * np.max(want))


@pytest.mark.parametrize('branch', ['lanes8', 'lanes1_cache', 'lanes1_nocache'])
def test_two_channels(obe, models, branch):
    n, k, n_settings = 4096, 30, 2000
    s = (np.linspace(1.5, 4.5, n_settings),)
    prior, cons = _peak_prior(n), (0.3,)
    with utility_options(_lane_fill(n_settings, int(branch[5])), 0 if branch.endswith('nocache') else 1):
        for lm, ok, aux in (('poisson', 'poisson', None), (models['user'], _user_var, (1.5, 4.0))):
            eng = obe.OptBayesExpt(models['two'], s, prior, cons, likelihood_model=lm, design_noise='likelihood',
                                   design_aux=aux)
            eng.rng = np.random.default_rng(8)
            draws, _ = orc.randdraw(prior, np.ones(n) / n, np.random.default_rng(8).random(k))
            _, ys = orc.yvar_from_draws(_two_peaks, orc.make_allsettings(s), draws, cons, 2)
            want = odn.utility_likelihood_noise(ys, ok, aux)
            assert_array_equal(eng.utility(), want)
            eng.utility_log_form = True
            eng.rng = np.random.default_rng(8)
            assert_allclose(eng.utility(), odn.utility_likelihood_noise(ys, ok, aux, log_form=True), rtol=1e-14)


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_max_min_and_pseudo(obe, models, kind):
    eng, want = _case(obe, models, kind, 3000, method='max_min')
    assert_array_equal(eng.utility(), want)
    eng, want = _case(obe, models, kind, 3000, method='pseudo_utility')
    assert_allclose(eng.utility(), want, rtol=1e-12, atol=0)
    # the accessors of a variance engine select the same kernels
    eng, want = _case(obe, models, kind, 3000, method='max_min')
    ev, _ = _case(obe, models, kind, 3000)
    assert_array_equal(ev.utility_max_min(), want)
    eng, want = _case(obe, models, kind, 3000, method='pseudo_utility')
    ev.rng = np.random.default_rng(8)
    assert_allclose(ev.utility_pseudo(), want, rtol=1e-12, atol=0)


@pytest.mark.parametrize('method', ['variance_approx', 'max_min', 'pseudo_utility'])
@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_invalid_outputs_give_zero(obe, models, kind, method):
    kw = dict(b_lo=-2.0) if kind == 'poisson' else dict(a_hi=1.4)      # negative rates, probabilities below 0
    eng, want = _case(obe, models, kind, 3000, method=method, **kw)
    got = eng.utility()
    zero = want == 0.0
    assert 0 < zero.sum() < len(want)
    assert_array_equal(got[zero], 0.0)
    if method == 'pseudo_utility':
        assert_allclose(got, want, rtol=1e-12, atol=0)
    else:
        assert_array_equal(got, want)


# ---------------------------------------------------------------------------------------------------------------
# closed loops and selection paths
# ---------------------------------------------------------------------------------------------------------------
RABI_SETTINGS = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))


def _rabi_prior(n, seed=1001):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_closed_loop_multinomial_matches_oracle(obe, models, kind):
    """40 cycles with the reference's multinomial resampling: every chosen setting equals OracleOBELik's."""
    n, cycles = 5000, 40
    prior = _rabi_prior(n)
    cons = (100.0, 0.9, 0.5) if kind == 'poisson' else (1.0, 0.9, 0.5)
    aux = None if kind == 'poisson' else 100.0
    eng = obe.OptBayesExpt(models['rabi'], RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False,
                           resampling='multinomial', use_jit=False, design_noise='likelihood', design_aux=aux)
    eng.rng = np.random.default_rng(1003)
    ora = odn.OracleOBEDesign(orc.model_rabi, RABI_SETTINGS, prior, cons, scale=False, rng=np.random.default_rng(1003),
                           likelihood_model=kind, design_noise='likelihood', design_aux=aux)
    meas = np.random.default_rng(1002)
    fired = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(cycles):
            x = eng.opt_setting()
            xo = ora.opt_setting()
            assert eng.last_setting_index == ora.last_setting_index, f'setting index differs at cycle {t}'
            assert x == xo
            mu = orc.model_rabi(x, (3.3, 1.7), cons)
            rec = (x, float(meas.poisson(mu)), 0.0) if kind == 'poisson' else (x, float(meas.binomial(100, mu)), 100.0)
            eng.pdf_update(rec)
            ora.pdf_update(rec)
            assert eng.just_resampled == ora.just_resampled, f'resample decision differs at cycle {t}'
            fired += int(eng.just_resampled)
    assert fired >= 2


class ScriptedRng:
    """random() -> the u0 of cycle t, random(k) -> the K uniforms of cycle t."""

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
def test_selection_paths_agree(obe, models, kind):
    """opt_setting with the eager select beside the resample, the device-side resample test and run_cycle_async
    choose the same settings given the same random numbers; the binomial trial count changes between cycles."""
    n, cycles = 50_000, 30
    prior = _rabi_prior(n)
    cons = (100.0, 0.9, 0.5) if kind == 'poisson' else (1.0, 0.9, 0.5)
    engines = []
    for _ in range(3):
        e = obe.OptBayesExpt(models['rabi'], RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False, seed=11,
                             design_noise='likelihood', design_aux=None if kind == 'poisson' else 100.0)
        e.rng = ScriptedRng(5, cycles, 30)
        engines.append(e)
    sync, dev, cyc = engines
    sync.eager_select = True
    dev.eager_select = dev.async_update = True
    assert dev._device_test_ok()
    meas = np.random.default_rng(9)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        x = [e.opt_setting() for e in engines]
        fired = 0
        for t in range(cycles):
            trials = 100.0 if t % 3 else 20.0 + t
            for e in engines:
                e.rng.t = t + 1
                if kind == 'binomial':
                    e.design_aux = trials
            assert x[0] == x[1] == x[2], f'cycle {t}'
            mu = orc.model_rabi(x[0], (3.3, 1.7), cons)
            rec = (x[0], float(meas.poisson(mu))) if kind == 'poisson' else \
                (x[0], float(meas.binomial(100, mu)), 100.0)
            sync.pdf_update(rec)
            dev.pdf_update(rec)
            cyc.run_cycle_async(rec, resample=sync.just_resampled, select=True)
            x = [e.opt_setting() for e in engines[:2]]
            ic = int(cyc.best_index_dev.cpu()[0])
            x.append(tuple(cyc.allsettings[:, ic]))
            assert sync.just_resampled == dev.just_resampled, f'cycle {t}'
            assert sync.last_setting_index == dev.last_setting_index == ic, f'cycle {t}'
            fired += int(sync.just_resampled)
    assert 2 <= fired < cycles


def test_gaussian_engine_likelihood_equals_fixed(obe, models):
    n = 20_000
    s = (np.linspace(1.5, 4.5, 5000),)
    prior = _peak_prior(n)
    a = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), default_noise_std=3.0, seed=11)
    b = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), default_noise_std=3.0, seed=11, design_noise='likelihood')
    assert b._model.value == a._model.value
    meas = np.random.default_rng(4)
    for e in (a, b):
        e.rng = np.random.default_rng(21)
    for t in range(10):
        assert_array_equal(a.utility(), b.utility())
        xa, xb = a.opt_setting(), b.opt_setting()
        assert xa == xb
        y = float(orc.model_lorentzian_hwhm(xa, (3.1, 50.0, 5.0), (0.3,)) + meas.normal(0, 3.0))
        a.pdf_update((xa, y, 3.0))
        b.pdf_update((xb, y, 3.0))


def test_fixed_and_likelihood_do_not_share_a_handle(obe, models):
    prior = _peak_prior(4096)
    s = (np.linspace(1.5, 4.5, 500),)
    f = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), likelihood_model='poisson', default_noise_std=5.0)
    d = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), likelihood_model='poisson', design_noise='likelihood')
    assert f._model.value != d._model.value
    assert f.model_function.design_noise == 'fixed' and d.model_function.design_noise == 'likelihood'
    for e in (f, d):
        e.rng = np.random.default_rng(2)
    uf, ud = f.utility(), d.utility()
    assert not np.array_equal(uf, ud)
    # the fixed engine is the plain likelihood handle: the variance over default_noise_std^2
    draws, _ = orc.randdraw(prior, np.ones(4096) / 4096, np.random.default_rng(2).random(30))
    var_p, _ = orc.yvar_from_draws(orc.model_lorentzian_hwhm, orc.make_allsettings(s), draws, (0.3,), 1)
    assert_array_equal(uf, orc.utility_variance(var_p, orc.noise_var_default(5.0, 1)))


def test_errors(obe, models):
    prior = _dip_prior(4096)
    s = (np.linspace(1.5, 4.5, 64),)
    eng = obe.OptBayesExpt(models['dip'], s, prior, (), likelihood_model='binomial', design_noise='likelihood',
                           design_aux=30.0)
    for bad in (0.0, -3.0, np.nan, np.inf, None, (1.0, 2.0)):
        with pytest.raises(ValueError):
            eng.design_aux = bad
    assert eng.design_aux == 30.0
    with pytest.raises(ValueError, match='full_kld'):
        eng.utility_full_kld()
    with pytest.raises(ValueError, match='design_noise'):
        obe.OptBayesExpt(models['dip'], s, prior, (), likelihood_model='binomial', design_noise='bayes')
    with pytest.raises(ValueError, match='design_aux'):
        obe.OptBayesExpt(models['dip'], s, prior, (), likelihood_model='binomial', design_noise='likelihood')
    with pytest.raises(ValueError, match='design_aux'):
        obe.OptBayesExpt(models['dip'], s, prior, (), likelihood_model='binomial', design_noise='likelihood',
                         design_aux=0.0)
    with pytest.raises(ValueError, match='full_kld'):
        obe.OptBayesExpt(models['dip'], s, prior, (), likelihood_model='binomial', design_noise='likelihood',
                         design_aux=3.0, utility_method='full_kld_utility')
    with pytest.raises(ValueError, match='noise_var'):
        obe.OptBayesExpt(models['peak'], s, _peak_prior(4096), (0.3,), design_noise='likelihood',
                         likelihood_model=obe.cuda_likelihood(USER_POISSON, 'user_poisson'))
    # the C entry refuses the full-KLD method for a design handle
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    import ctypes as C
    dd = eng._draws_buffer()
    rc = lib.obe_utility(eng._model, C.c_void_p(dd.data_ptr()), 30, C.c_void_p(eng._settings_dev.data_ptr()), eng._lds,
                         64, eng._cons_arr, _lib.darr([30.0], _lib.MAX_CHANNELS), None, None, 3, 0,
                         C.c_void_p(dd.data_ptr()), C.c_void_p(eng._utility_dev.data_ptr()),
                         C.c_void_p(eng._best_dev.data_ptr()), C.c_void_p(eng._select_scratch.data_ptr()),
                         eng._stream())
    assert rc != 0 and b'full KLD' in lib.obe_last_error()
