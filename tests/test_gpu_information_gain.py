"""The information-gain utility (utility_method='information_gain') on the device.

The kernel against oracle/information_gain.information_gain_from_draws within |dev - orc| <= 1e-9 orc + 1e-15:
lorentzian_hwhm and rabi as Poisson rates, lorentzian_dip as binomial probabilities (n = 40), K = 3 / 30 / 128,
1 / 2000 / 1e5 settings, broad and tight priors, invalid outputs, a cost vector.  Then determinism (run to run and
over grid sizes), the agreement of the selection paths, closed loops against the oracle engine and the refusals of
the C entry.
"""
import ctypes as C
import warnings

import numpy as np
import pytest

from oracle import information_gain as oig
from oracle import obe_oracle as orc

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-9, 1e-15

TWO_CH = r'''
__device__ void two_rates(const double* s, const double* p, const double* c, double* y) {
    y[0] = p[2] + p[1] / ((s[0] - p[0]) * (s[0] - p[0]) + 1.0);
    y[1] = p[2];
}
'''


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def models(obe):
    return dict(peak=obe.builtin('lorentzian_hwhm'), dip=obe.builtin('lorentzian_dip'), rabi=obe.builtin('rabi'),
                two=obe.cuda_source(TWO_CH, 'two_rates', 1, 3, 1, 2))


def _lib():
    from optbayesexpt_b200 import _lib
    return _lib, _lib.load()


def _prior(model, n, spread, seed=3, bad=False):
    """broad (spread None) or tight (relative spread) priors; bad: some outputs invalid for the likelihood"""
    g = np.random.default_rng(seed)
    if model == 'peak':
        if spread is None:
            return np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(-2.0 if bad else 2.0, 10.0, n)])
        c = np.array([3.0, 50.0, 5.0])
    elif model == 'dip':
        if spread is None:
            return np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 1.4 if bad else 0.8, n), g.uniform(0.2, 0.6, n)])
        c = np.array([3.0, 0.5, 0.4])
    else:
        if spread is None:
            return np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])
        c = np.array([3.3, 1.7])
    return c[:, None] * (1.0 + spread * g.standard_normal((len(c), n)))


SETUP = {  # model -> (likelihood, constants, design aux, setting axes for S settings)
    'peak': ('poisson', (0.3,), None, lambda s: (np.linspace(1.5, 4.5, s),)),
    'dip': ('binomial', (), 40.0, lambda s: (np.linspace(1.5, 4.5, s),)),
    'rabi': ('poisson', (100.0, 0.9, 0.5), None,
             lambda s: (np.linspace(0, 1, 40), np.linspace(-10, 10, s // 40)) if s >= 40 else
             (np.array([0.3]), np.linspace(-10, 10, s))),
}


class _Cost:
    """a mixin whose cost_estimate() is a fixed vector over the settings"""
    cost_vector = None

    def cost_estimate(self):
        return self.cost_vector


def _case(obe, models, model, n_settings, k, spread=None, bad=False, cost=False, n=4096, utility_method=None):
    """(engine with rng seed 8, oracle utility of its first selection, its draws' outputs (K, 1, S))"""
    lik, cons, aux, axes = SETUP[model]
    s = axes(n_settings)
    prior = _prior(model, n, spread, bad=bad)
    cls = obe.OptBayesExpt
    if cost:
        cls = type('CostEngine', (_Cost, obe.OptBayesExpt), {})
    eng = cls(models[model], s, prior, cons, likelihood_model=lik, design_noise='likelihood', design_aux=aux,
              n_draws=k, utility_method=utility_method or 'information_gain')
    n_set = len(eng.setting_indices)
    cvec = 1.0
    if cost:
        cvec = np.random.default_rng(12).uniform(1.0, 3.0, n_set)
        eng.cost_vector = cvec
    eng.rng = np.random.default_rng(8)
    draws, _ = orc.randdraw(prior, np.ones(n) / n, np.random.default_rng(8).random(k))
    ys = np.stack([eng.eval_over_all_settings(draws[:, j]) for j in range(k)])      # the device's own outputs
    return eng, ys, cvec


def _check(got, ys, kind, aux, cost=1.0, subset=None):
    idx = np.arange(ys.shape[-1]) if subset is None else subset
    want = oig.information_gain_from_draws(ys[..., idx], kind, aux, cost=np.broadcast_to(cost, (ys.shape[-1],))[idx])
    err = np.abs(got[idx] - want)
    assert np.all(err <= RTOL * want + ATOL), (np.max(err / (want + 1e-300)), idx[np.argmax(err - RTOL * want)])
    return want


# ---------------------------------------------------------------------------------------------------------------
# the utility against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spread', [None, 1e-6], ids=['broad', 'tight'])
@pytest.mark.parametrize('k', [3, 30, 128])
@pytest.mark.parametrize('model', ['peak', 'rabi', 'dip'])
def test_utility_matches_oracle(obe, models, model, k, spread):
    eng, ys, _ = _case(obe, models, model, 2000, k, spread)
    got = eng.utility()
    lik, _, aux, _ = SETUP[model]
    want = _check(got, ys, lik, aux)
    assert np.all(want >= 0.0) and np.all(want <= np.log(k) + 1e-12)
    if spread is None:
        assert np.max(want) > 1e-2
    else:
        assert 0.0 < np.max(want) < 1e-5                 # (the tight prior: I of 1e-12 .. 1e-6)
    eng.rng = np.random.default_rng(8)
    eng.opt_setting()
    assert eng.last_setting_index == int(np.argmax(got))
    assert abs(got[eng.last_setting_index] - np.max(want)) <= RTOL * np.max(want)


@pytest.mark.parametrize('model', ['peak', 'dip', 'rabi'])
def test_one_setting(obe, models, model):
    eng, ys, _ = _case(obe, models, model, 1, 30)
    got = eng.utility()
    assert got.shape == (1,)
    _check(got, ys, SETUP[model][0], SETUP[model][2])
    eng.rng = np.random.default_rng(8)
    assert eng.opt_setting() == tuple(eng.allsettings[:, 0])


@pytest.mark.parametrize('model,k', [('peak', 30), ('dip', 128), ('rabi', 30)])
def test_large_grid(obe, models, model, k):
    """1e5 settings: every 97th setting and the argmax against the oracle"""
    eng, ys, _ = _case(obe, models, model, 100_000, k)
    got = eng.utility()
    subset = np.unique(np.concatenate([np.arange(0, got.size, 97), [int(np.argmax(got))]]))
    _check(got, ys, SETUP[model][0], SETUP[model][2], subset=subset)


@pytest.mark.parametrize('model', ['peak', 'dip'])
def test_invalid_outputs_give_zero(obe, models, model):
    eng, ys, _ = _case(obe, models, model, 3000, 30, bad=True)
    got = eng.utility()
    want = _check(got, ys, SETUP[model][0], SETUP[model][2])
    zero = ~np.all(oig.valid_outputs(ys[:, 0], SETUP[model][0]), axis=0)
    assert 0 < zero.sum() < len(want)
    assert np.all(got[zero] == 0.0)


@pytest.mark.parametrize('spread', [None, 1e-6], ids=['broad', 'tight'])
@pytest.mark.parametrize('model', ['peak', 'dip'])
def test_cost_vector(obe, models, model, spread):
    eng, ys, cvec = _case(obe, models, model, 2000, 30, spread, cost=True)
    got = eng.utility()
    _check(got, ys, SETUP[model][0], SETUP[model][2], cost=cvec)
    eng.rng = np.random.default_rng(8)
    eng.opt_setting()
    assert eng.last_setting_index == int(np.argmax(got))


def test_accessor_log_form_and_good_setting(obe, models):
    """utility_information_gain() of a variance engine is the kernel of an information-gain engine; the log form
    is ignored; good_setting picks a setting of positive utility."""
    eng, ys, _ = _case(obe, models, 'peak', 2000, 30)
    ev, _, _ = _case(obe, models, 'peak', 2000, 30, utility_method='variance_approx')
    u = eng.utility()
    np.testing.assert_array_equal(ev.utility_information_gain(), u)
    assert ev.utility_method == 'variance_approx' and ev._utility_code == 0
    eng.utility_log_form = True
    eng.rng = np.random.default_rng(8)
    np.testing.assert_array_equal(eng.utility(), u)
    eng.rng = np.random.default_rng(8)
    eng.good_setting(pickiness=4)
    assert u[eng.last_setting_index] > 0.0


# ---------------------------------------------------------------------------------------------------------------
# determinism
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('model', ['peak', 'dip'])
def test_same_bits_run_to_run_and_over_grids(obe, models, model):
    _l, lib = _lib()
    eng, _, _ = _case(obe, models, model, 20_000, 30)
    ref = eng.utility()
    best = eng._best_dev.cpu().numpy().copy()
    try:
        for blocks in (0, 0, 1, 7, 100, 5000):
            lib.obe_set_option(b'utility_info_blocks', blocks)
            eng.rng = np.random.default_rng(8)
            assert np.array_equal(eng.utility(), ref), blocks
            assert np.array_equal(eng._best_dev.cpu().numpy(), best), blocks
    finally:
        lib.obe_set_option(b'utility_info_blocks', 0)
    assert best[0] == int(np.argmax(ref))


# ---------------------------------------------------------------------------------------------------------------
# selection paths and closed loops
# ---------------------------------------------------------------------------------------------------------------
RABI_SETTINGS = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))


def _rabi_prior(n, seed=1001):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])


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
                             design_noise='likelihood', design_aux=None if kind == 'poisson' else 100.0,
                             utility_method='information_gain')
        e.rng = ScriptedRng(5, cycles, 30)
        engines.append(e)
    sync, dev, cyc = engines
    sync.eager_select = True
    dev.eager_select = dev.async_update = True
    assert dev._device_test_ok() and cyc._early_select_ok()
    meas = np.random.default_rng(9)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        x = [e.opt_setting() for e in engines]
        fired = 0
        for t in range(cycles):
            trials = 100.0 if t % 3 else float(20 + t)
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


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_closed_loop_multinomial_matches_oracle(obe, models, kind):
    """40 cycles with multinomial resampling: the device's choice is the oracle's argmax (or ties with it within
    the tolerance), and the oracle follows the device's choice."""
    n, cycles = 5000, 40
    prior = _rabi_prior(n)
    cons = (100.0, 0.9, 0.5) if kind == 'poisson' else (1.0, 0.9, 0.5)
    aux = None if kind == 'poisson' else 100.0
    eng = obe.OptBayesExpt(models['rabi'], RABI_SETTINGS, prior, cons, likelihood_model=kind, scale=False,
                           resampling='multinomial', use_jit=False, design_noise='likelihood', design_aux=aux,
                           utility_method='information_gain')
    eng.rng = np.random.default_rng(1003)
    ora = oig.OracleOBEInfo(orc.model_rabi, RABI_SETTINGS, prior, cons, scale=False, rng=np.random.default_rng(1003),
                            likelihood_model=kind, design_aux=aux)
    meas = np.random.default_rng(1002)
    fired = ties = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(cycles):
            x = eng.opt_setting()
            ora.opt_setting()
            i, u = eng.last_setting_index, ora.last_utility
            if i != ora.last_setting_index:
                top = np.sort(u)[-2:]
                assert top[1] - top[0] <= RTOL * top[1] + ATOL, f'setting index differs at cycle {t}'
                assert u[i] >= top[1] - (RTOL * top[1] + ATOL), f'cycle {t}'
                ties += 1
            ora.last_setting_index = i
            mu = orc.model_rabi(x, (3.3, 1.7), cons)
            rec = (x, float(meas.poisson(mu)), 0.0) if kind == 'poisson' else (x, float(meas.binomial(100, mu)), 100.0)
            eng.pdf_update(rec)
            ora.pdf_update(rec)
            assert eng.just_resampled == ora.just_resampled, f'resample decision differs at cycle {t}'
            fired += int(eng.just_resampled)
    assert fired >= 2 and ties <= 2


# ---------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------
def _call(eng, method, k=30, aux=None):
    _l, lib = _lib()
    dd = eng._draws_buffer()
    vn = _l.darr([1.0 if aux is None else aux] * 2, _l.MAX_CHANNELS)
    n_set = len(eng.setting_indices)
    rc = lib.obe_utility(eng._model, C.c_void_p(dd.data_ptr()), k, C.c_void_p(eng._settings_dev.data_ptr()),
                         eng._lds, n_set, eng._cons_arr, vn, None, None, method, 0, None,
                         C.c_void_p(eng._utility_dev.data_ptr()), C.c_void_p(eng._best_dev.data_ptr()),
                         C.c_void_p(eng._select_scratch.data_ptr()), eng._stream())
    return rc, lib.obe_last_error()


def test_c_entry_refusals(obe, models):
    prior = _prior('peak', 4096, None)
    s = (np.linspace(1.5, 4.5, 64),)
    gauss = obe.OptBayesExpt(models['peak'], s, prior, (0.3,))
    plain = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), likelihood_model='poisson')
    design = obe.OptBayesExpt(models['peak'], s, prior, (0.3,), likelihood_model='poisson', design_noise='likelihood')
    two = obe.OptBayesExpt(models['two'], s, prior, (0.3,), likelihood_model='poisson', design_noise='likelihood')
    dip = obe.OptBayesExpt(models['dip'], s, _prior('dip', 4096, None), (), likelihood_model='binomial',
                           design_noise='likelihood', design_aux=40.0)
    for eng, kw, what in ((gauss, {}, b'design handle'), (plain, {}, b'design handle'), (two, {}, b'single-channel'),
                          (dip, dict(aux=2.5), b'integer'), (dip, dict(aux=0.0), b'integer'),
                          (design, dict(k=129), b'n_draws')):
        rc, err = _call(eng, 4, **kw)
        assert rc != 0 and b'information gain' in err and what in err, err
    rc, err = _call(design, 5)
    assert rc != 0 and b'unknown utility method' in err
    # the accepted cases run
    assert _call(design, 4)[0] == 0 and _call(dip, 4, aux=40.0)[0] == 0
    # the Python layer refuses before the device
    for eng in (gauss, plain, two):
        with pytest.raises(ValueError, match='information_gain'):
            eng.utility_information_gain()
    dip.design_aux = 2.5                      # (a variance engine takes any positive aux ...)
    with pytest.raises(ValueError, match='integer'):
        dip.utility_information_gain()        # (... but cannot run the information gain with it)
    with pytest.raises(SyntaxError, match='information_gain'):
        obe.OptBayesExpt(models['peak'], s, prior, (0.3,), utility_method='information_gains')
    ig = obe.OptBayesExpt(models['dip'], s, _prior('dip', 4096, None), (), likelihood_model='binomial',
                          design_noise='likelihood', design_aux=40.0, utility_method='information_gain')
    with pytest.raises(ValueError, match='integer'):
        ig.design_aux = 12.5
    assert ig.design_aux == 40.0
    ig.design_aux = 12
    ig.utility()
