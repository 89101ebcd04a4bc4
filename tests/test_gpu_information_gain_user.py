"""The information gain of a user count likelihood (cuda_likelihood(..., window=)) on the device.

The kernel against oracle/information_gain_user.information_gain_user within |dev - orc| <= 1e-8 orc + 1e-14 s sqrt(orc)
(s: the size of the log-pmf's terms, see tests/test_information_gain_user_host.py) for a negative binomial, the
two-Poisson readout and a beta-binomial (oracle/count_pmfs.py), K = 3 / 30 / 128, 1 / 2000 / 1e5 settings, broad and
tight priors and a cost vector; the user-restated Poisson against built-in method 4 on the same draws; every invalid
setting exactly 0; determinism over grid sizes; the agreement of the selection paths; a closed loop against the
oracle engine; the refusals of the C entry.
"""
import ctypes as C
import warnings

import numpy as np
import pytest
from scipy.special import gammaln

from oracle import count_pmfs as cp
from oracle import information_gain_user as oigu
from oracle import obe_oracle as orc

pytestmark = pytest.mark.gpu

RTOL, SQ = 1e-8, 1e-14
NAN = '__longlong_as_double(0x7ff8000000000000LL)'


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def models(obe):
    return dict(peak=obe.builtin('lorentzian_hwhm'), dip=obe.builtin('lorentzian_dip'), rabi=obe.builtin('rabi'))


def _lib():
    from optbayesexpt_b200 import _lib
    return _lib, _lib.load()


# pmf -> (model, constants, design aux); the peak gives rates of 2 .. 90 counts, the dip probabilities in (0, 1)
PMFS = {'negbin': ('peak', (0.3,), 20.0), 'readout': ('dip', (), 1.0), 'betabinom': ('dip', (), 40.0),
        'poisson': ('peak', (0.3,), 1.0)}


def _prior(model, n, spread, seed=3, bad=False):
    g = np.random.default_rng(seed)
    if model == 'peak':
        if spread is None:
            return np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(-2.0 if bad else 2.0, 10.0, n)])
        c = np.array([3.0, 50.0, 5.0])
    else:
        if spread is None:
            return np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 1.4 if bad else 0.8, n), g.uniform(0.2, 0.6, n)])
        c = np.array([3.0, 0.5, 0.4])
    return c[:, None] * (1.0 + spread * g.standard_normal((len(c), n)))


class _Cost:
    cost_vector = None

    def cost_estimate(self):
        return self.cost_vector


def _engine(obe, models, lik, model, settings, prior, cons, aux, k=30, cost=False, **kw):
    cls = type('CostEngine', (_Cost, obe.OptBayesExpt), {}) if cost else obe.OptBayesExpt
    return cls(models[model], settings, prior, cons, likelihood_model=lik, design_noise='likelihood',
               design_aux=aux, n_draws=k, utility_method='information_gain', **kw)


def _case(obe, models, name, n_settings, k, spread=None, cost=False, bad=False, n=4096):
    """(engine with rng seed 8, its first draws' outputs (K, 1, S), cost, numpy twins, aux)"""
    src, entry, nv, win, lp, nv_np, win_np = cp.pmf(name)
    model, cons, aux = PMFS[name]
    prior = _prior(model, n, spread, bad=bad)
    lik = obe.cuda_likelihood(src, entry, noise_var=nv, window=win)
    eng = _engine(obe, models, lik, model, (np.linspace(1.5, 4.5, n_settings),), prior, cons, aux, k, cost)
    cvec = 1.0
    if cost:
        cvec = np.random.default_rng(12).uniform(1.0, 3.0, n_settings)
        eng.cost_vector = cvec
    eng.rng = np.random.default_rng(8)
    draws, _ = orc.randdraw(prior, np.ones(n) / n, np.random.default_rng(8).random(k))
    ys = np.stack([eng.eval_over_all_settings(draws[:, j]) for j in range(k)])
    return eng, ys, cvec, (lp, nv_np, win_np), aux


def _scale(ys, nv, aux):
    x = ys.reshape(-1)
    x = x[np.isfinite(x)]
    with np.errstate(invalid='ignore'):
        v = np.maximum(np.nan_to_num(np.asarray(nv(x, aux), dtype=np.float64)), 0.0)
    mu = x * aux if np.all((x >= 0) & (x <= 1.0)) and aux > 1.0 else x
    return max(1.0, float(gammaln(np.max(mu + 3.0 * np.sqrt(v)) + 1.0)) / 100.0)


def _check(got, ys, twins, aux, cost=1.0, subset=None):
    lp, nv, win = twins
    idx = np.arange(ys.shape[-1]) if subset is None else subset
    c = np.broadcast_to(np.asarray(cost, dtype=np.float64), (ys.shape[-1],))[idx]
    want = oigu.information_gain_user(lp, win, ys[..., idx], aux, noise_var=nv, cost=c)
    tol = RTOL * want + SQ * _scale(ys[..., idx], nv, aux) * np.sqrt(want)
    err = np.abs(got[idx] - want)
    assert np.all(err <= tol), (np.max(err / (tol + 1e-300)), idx[np.argmax(err - tol)])
    return want


def _subset(n, got, step):
    return np.unique(np.concatenate([np.arange(0, n, step), [int(np.argmax(got))]]))


# ---------------------------------------------------------------------------------------------------------------
# the utility against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spread', [None, 1e-6], ids=['broad', 'tight'])
@pytest.mark.parametrize('k', [3, 30, 128])
@pytest.mark.parametrize('name', ['negbin', 'readout', 'betabinom'])
def test_utility_matches_oracle(obe, models, name, k, spread):
    eng, ys, _, twins, aux = _case(obe, models, name, 2000, k, spread)
    got = eng.utility()
    idx = _subset(2000, got, 10 if k < 128 else 40)
    want = _check(got, ys, twins, aux, subset=idx)
    assert np.all(want >= 0.0) and np.all(want <= np.log(k) + 1e-12)
    if spread is None:
        assert np.max(want) > 1e-3
    else:
        assert 0.0 < np.max(want) < 1e-5
    eng.rng = np.random.default_rng(8)
    eng.opt_setting()
    assert eng.last_setting_index == int(np.argmax(got))


@pytest.mark.parametrize('name', ['negbin', 'readout', 'betabinom'])
def test_one_setting_and_large_grid(obe, models, name):
    eng, ys, _, twins, aux = _case(obe, models, name, 1, 30)
    got = eng.utility()
    assert got.shape == (1,)
    _check(got, ys, twins, aux)
    eng, ys, _, twins, aux = _case(obe, models, name, 100_000, 30)
    got = eng.utility()
    _check(got, ys, twins, aux, subset=_subset(100_000, got, 997))


@pytest.mark.parametrize('spread', [None, 1e-6], ids=['broad', 'tight'])
@pytest.mark.parametrize('name', ['negbin', 'readout'])
def test_cost_vector(obe, models, name, spread):
    eng, ys, cvec, twins, aux = _case(obe, models, name, 2000, 30, spread, cost=True)
    got = eng.utility()
    _check(got, ys, twins, aux, cost=cvec, subset=_subset(2000, got, 10))
    eng.rng = np.random.default_rng(8)
    eng.opt_setting()
    assert eng.last_setting_index == int(np.argmax(got))


@pytest.mark.parametrize('spread', [None, 1e-6], ids=['broad', 'tight'])
@pytest.mark.parametrize('k', [3, 30, 128])
def test_user_poisson_matches_builtin(obe, models, k, spread):
    """The Poisson restated as a user pmf against built-in method 4 on the same draws."""
    eng, ys, _, twins, aux = _case(obe, models, 'poisson', 2000, k, spread)
    got = eng.utility()
    prior = _prior('peak', 4096, spread)
    ref = _engine(obe, models, 'poisson', 'peak', (np.linspace(1.5, 4.5, 2000),), prior, (0.3,), None, k)
    ref.rng = np.random.default_rng(8)
    want = ref.utility()
    tol = RTOL * want + SQ * _scale(ys, cp.poisson_var, 1.0) * np.sqrt(want)
    assert np.all(np.abs(got - want) <= tol), np.max(np.abs(got - want) / (tol + 1e-300))
    assert int(np.argmax(got)) == int(np.argmax(want)) or abs(np.max(got) - np.max(want)) <= tol.max()


# ---------------------------------------------------------------------------------------------------------------
# invalid settings
# ---------------------------------------------------------------------------------------------------------------
# a Poisson pmf whose window (or log-pmf) breaks in one way where the rate x exceeds 30: mode = design aux
BROKEN = cp.POISSON_SOURCE + r'''
__device__ double br_lp(const double* ym, const double* y, const double* aux, int n) {
    const double v = pois_lp(ym, y, aux, n);
    if (ym[0] > 30.0 && y[0] == floor(ym[0])) {
        if (aux[0] == 7.0) return NAN_;
        if (aux[0] == 8.0) return -(NEG_INF_);
    }
    return v;
}
__device__ double br_var(double x, double a) { return (a == 9.0 && x > 30.0) ? NAN_ : x; }
__device__ void br_win(double x, double a, double* lo, double* hi) {
    pois_win(x, a, lo, hi);
    if (x <= 30.0) return;
    if (a == 1.0) *lo = NAN_;
    if (a == 2.0) *hi = *hi + 0.5;
    if (a == 3.0) *lo = -1.0;
    if (a == 4.0) *lo = *hi + 1.0;
    if (a == 5.0) *hi = 9007199254740994.0;
    if (a == 6.0) *hi = *lo + 2097152.0;
}
'''.replace('NAN_', NAN).replace('NEG_INF_', cp.NEG_INF)


def _broken_twins(mode):
    def lp(x, y, a):
        v = cp.poisson_logpmf(x, y)
        x, y = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64))
        hit = (x > 30.0) & (y == np.floor(x))
        if mode == 7:
            return np.where(hit, np.nan, v)
        if mode == 8:
            return np.where(hit, np.inf, v)
        return v

    def nv(x, a):
        x = np.asarray(x, np.float64)
        return np.where((x > 30.0) & (mode == 9), np.nan, x)

    def win(x, a):
        lo, hi = cp.poisson_window(x)
        big = np.asarray(x) > 30.0
        if mode == 1:
            lo = np.where(big, np.nan, lo)
        elif mode == 2:
            hi = np.where(big, hi + 0.5, hi)
        elif mode == 3:
            lo = np.where(big, -1.0, lo)
        elif mode == 4:
            lo = np.where(big, hi + 1.0, lo)
        elif mode == 5:
            hi = np.where(big, 9007199254740994.0, hi)
        elif mode == 6:
            hi = np.where(big, lo + 2097152.0, hi)
        return lo, hi
    return lp, nv, win


@pytest.mark.parametrize('mode', [1, 2, 3, 4, 5, 6, 7, 8, 9],
                         ids=['lo_nan', 'hi_fraction', 'lo_negative', 'lo_above_hi', 'hi_above_2p53', 'union_cap',
                              'logpmf_nan', 'logpmf_plus_inf', 'noise_var_nan'])
def test_invalid_settings_give_zero(obe, models, mode):
    lik = obe.cuda_likelihood(BROKEN, 'br_lp', noise_var='br_var', window='br_win')
    prior = _prior('peak', 4096, None)
    eng = _engine(obe, models, lik, 'peak', (np.linspace(1.5, 4.5, 600),), prior, (0.3,), float(mode))
    eng.rng = np.random.default_rng(8)
    draws, _ = orc.randdraw(prior, np.ones(4096) / 4096, np.random.default_rng(8).random(30))
    ys = np.stack([eng.eval_over_all_settings(draws[:, j]) for j in range(30)])
    got = eng.utility()
    hit = np.any(ys[:, 0] > 30.0, axis=0)
    assert 0 < hit.sum() < hit.size
    assert np.all(got[hit] == 0.0)
    assert np.all(got[~hit] > 0.0)
    _check(got, ys, _broken_twins(mode), float(mode), subset=np.arange(0, 600, 7))


def test_invalid_outputs_give_zero(obe, models):
    """readout with P(bright) below 0 for some draws (a dip deeper than 1): the noise variance is negative there"""
    eng, ys, _, twins, aux = _case(obe, models, 'readout', 3000, 30, bad=True)
    got = eng.utility()
    zero = np.any((ys[:, 0] < 0.0) | (ys[:, 0] > 1.0), axis=0)
    assert 0 < zero.sum() < zero.size
    assert np.all(got[zero] == 0.0)
    _check(got, ys, twins, aux, subset=_subset(3000, got, 11))


# ---------------------------------------------------------------------------------------------------------------
# determinism, selection paths, closed loop
# ---------------------------------------------------------------------------------------------------------------
def test_same_bits_over_grids(obe, models):
    _l, lib = _lib()
    eng, _, _, _, _ = _case(obe, models, 'readout', 20_000, 30)
    ref = eng.utility()
    best = eng._best_dev.cpu().numpy().copy()
    try:
        for blocks in (0, 1, 7, 148, 1000, 1184):
            lib.obe_set_option(b'utility_info_blocks', blocks)
            eng.rng = np.random.default_rng(8)
            assert np.array_equal(eng.utility(), ref), blocks
            assert np.array_equal(eng._best_dev.cpu().numpy(), best), blocks
    finally:
        lib.obe_set_option(b'utility_info_blocks', 0)
    assert best[0] == int(np.argmax(ref))


RABI_SETTINGS = (np.linspace(0, 1, 31), np.linspace(-10, 10, 31))
RABI_CONS = (1.0, 0.9, 0.5)
LAM_D, LAM_B = 0.5, 3.0


def _rabi_prior(n, seed=1001):
    g = np.random.default_rng(seed)
    return np.array([g.uniform(1.0, 5.0, n), g.uniform(-5.0, 5.0, n)])


def _readout_count(g, p):
    return float(g.poisson(LAM_B if g.random() < p else LAM_D))


class ScriptedRng:
    def __init__(self, seed, cycles, k):
        g = np.random.default_rng(seed)
        self.u0 = g.random(cycles + 1)
        self.uk = g.random((cycles + 1, k))
        self.t = 0

    def random(self, size=None):
        if size is None:
            return self.u0[self.t]
        return self.uk[self.t, :size].copy()


def test_selection_paths_agree(obe, models):
    """opt_setting with the eager select, the device-side resample test and run_cycle_async choose the same
    settings given the same random numbers."""
    src, entry, nv, win = cp.pmf('readout', lam_d=LAM_D, lam_b=LAM_B)[:4]
    lik = obe.cuda_likelihood(src, entry, noise_var=nv, window=win)
    n, cycles = 50_000, 30
    prior = _rabi_prior(n)
    engines = []
    for _ in range(3):
        e = _engine(obe, models, lik, 'rabi', RABI_SETTINGS, prior, RABI_CONS, None, scale=False, seed=11)
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
            for e in engines:
                e.rng.t = t + 1
            assert x[0] == x[1] == x[2], f'cycle {t}'
            rec = (x[0], _readout_count(meas, orc.model_rabi(x[0], (3.3, 1.7), RABI_CONS)), 1.0)
            sync.pdf_update(rec)
            dev.pdf_update(rec)
            cyc.run_cycle_async(rec, resample=sync.just_resampled, select=True)
            x = [e.opt_setting() for e in engines[:2]]
            ic = int(cyc.best_index_dev.cpu()[0])
            x.append(tuple(cyc.allsettings[:, ic]))
            assert sync.just_resampled == dev.just_resampled, f'cycle {t}'
            assert sync.last_setting_index == dev.last_setting_index == ic, f'cycle {t}'
            fired += int(sync.just_resampled)
    assert fired >= 1


def test_closed_loop_readout_matches_oracle(obe, models):
    """40 cycles of single-shot readout with multinomial resampling: the device's choice is the oracle's argmax
    (or ties with it within the tolerance), and the oracle follows the device's choice."""
    src, entry, nv, win, lp, nv_np, win_np = cp.pmf('readout', lam_d=LAM_D, lam_b=LAM_B)
    lik = obe.cuda_likelihood(src, entry, noise_var=nv, window=win)
    n, cycles = 5000, 40
    prior = _rabi_prior(n)
    eng = _engine(obe, models, lik, 'rabi', RABI_SETTINGS, prior, RABI_CONS, None, scale=False,
                  resampling='multinomial', use_jit=False)
    eng.rng = np.random.default_rng(1003)
    ora = oigu.OracleOBEInfoUser(orc.model_rabi, RABI_SETTINGS, prior, RABI_CONS, scale=False,
                            rng=np.random.default_rng(1003), likelihood_model=lambda ym, y, a: lp(ym[0], y, a),
                            noise_var=nv_np, window=win_np)
    meas = np.random.default_rng(1002)
    ties = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(cycles):
            x = eng.opt_setting()
            ora.opt_setting()
            i, u = eng.last_setting_index, ora.last_utility
            if i != ora.last_setting_index:
                top = np.sort(u)[-2:]
                tol = RTOL * top[1] + SQ * np.sqrt(top[1])
                assert top[1] - top[0] <= tol, f'setting index differs at cycle {t}'
                assert u[i] >= top[1] - tol, f'cycle {t}'
                ties += 1
            ora.last_setting_index = i
            rec = (x, _readout_count(meas, orc.model_rabi(x, (3.3, 1.7), RABI_CONS)), 1.0)
            eng.pdf_update(rec)
            ora.pdf_update(rec)
            assert eng.just_resampled == ora.just_resampled, f'resample decision differs at cycle {t}'
    assert ties <= 2


# ---------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------
def _call(eng, method, k=30):
    _l, lib = _lib()
    dd = eng._draws_buffer()
    vn = _l.darr([1.0] * 2, _l.MAX_CHANNELS)
    rc = lib.obe_utility(eng._model, C.c_void_p(dd.data_ptr()), k, C.c_void_p(eng._settings_dev.data_ptr()),
                         eng._lds, len(eng.setting_indices), eng._cons_arr, vn, None, None, method, 0, None,
                         C.c_void_p(eng._utility_dev.data_ptr()), C.c_void_p(eng._best_dev.data_ptr()),
                         C.c_void_p(eng._select_scratch.data_ptr()), eng._stream())
    return rc, lib.obe_last_error()


def test_c_entry_refusals(obe, models):
    src, entry, nv, win = cp.pmf('readout')[:4]
    prior = _prior('dip', 4096, None)
    s = (np.linspace(1.5, 4.5, 64),)
    no_window = obe.OptBayesExpt(models['dip'], s, prior, (), design_noise='likelihood',
                                 likelihood_model=obe.cuda_likelihood(src, entry, noise_var=nv))
    rc, err = _call(no_window, 4)
    assert rc != 0 and b'information gain' in err and b'window' in err, err
    with pytest.raises(ValueError, match='poisson'):
        no_window.utility_information_gain()
    windowed = _engine(obe, models, obe.cuda_likelihood(src, entry, noise_var=nv, window=win), 'dip', s, prior, (),
                       None)
    rc, err = _call(windowed, 4, k=129)
    assert rc != 0 and b'n_draws' in err, err
    assert _call(windowed, 4)[0] == 0
    plain = obe.OptBayesExpt(models['dip'], s, prior, (),
                             likelihood_model=obe.cuda_likelihood(src, entry, noise_var=nv, window=win))
    rc, err = _call(plain, 4)
    assert rc != 0 and b'design handle' in err, err
