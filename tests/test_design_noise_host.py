"""CPU tests of the likelihood-aware setting selection (design_noise='likelihood'): the oracle's noise variance
against scipy.stats, its zero / inf / invalid-output rules, the NVRTC compile of the design handles (the compile
needs no GPU; loading the cubin does), and the argument checks that need no device."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import design_noise as odn


def test_oracle_noise_variance_equals_scipy():
    from scipy.stats import binom, poisson
    lam = np.concatenate([[0.0, 1e-300, 1e-3], np.linspace(0.01, 80.0, 400), [1e6]])
    assert_allclose(odn.noise_var_from_draws(lam[None, None, :], 'poisson')[0], poisson.var(lam), rtol=1e-15)
    p = np.concatenate([[0.0, 1.0], np.linspace(1e-4, 1 - 1e-4, 500)])
    for n in (1.0, 7.0, 100.0, 1e6):
        got = odn.noise_var_from_draws(p[None, None, :], 'binomial', n)[0]
        assert_allclose(got, binom.var(n, p) / n ** 2, rtol=1e-11)    # (scipy: n p (1 - p), rounded otherwise)
    # K draws: the mean of nu over the draws, per channel (aux per channel)
    g = np.random.default_rng(4)
    y = g.uniform(0.0, 1.0, (30, 2, 50))
    got = odn.noise_var_from_draws(y, 'binomial', (10.0, 40.0))
    want = np.stack([np.mean(binom.var(10, y[:, 0]) / 100.0, axis=0), np.mean(binom.var(40, y[:, 1]) / 1600.0, axis=0)])
    assert_allclose(got, want, rtol=1e-14)
    # Poisson: bit for bit np.var's own mean
    lamk = g.uniform(0.0, 50.0, (30, 1, 64))
    assert_array_equal(odn.noise_var_from_draws(lamk, 'poisson'), np.mean(lamk, axis=0))


def test_oracle_utility_rules():
    k = 8
    y = np.full((k, 1, 6), 0.5)
    y[:, 0, 1] = np.linspace(0.1, 0.9, k)                    # ordinary setting
    y[:, 0, 2] = [0.0, 1.0] * (k // 2)                       # v = 0, var > 0: +inf
    y[:, 0, 3] = 0.0                                          # var = 0, v = 0: 0
    y[3, 0, 4] = 1.0 + 1e-12                                  # one draw outside [0, 1]: 0
    y[5, 0, 5] = np.nan                                       # NaN: 0
    u = odn.utility_likelihood_noise(y, 'binomial', 20.0)
    assert u[0] == 0.0 and u[3] == 0.0 and u[4] == 0.0 and u[5] == 0.0
    assert u[2] == np.inf
    yb = y[:, 0, 1]
    assert_allclose(u[1], np.var(yb) / (np.mean(yb * (1 - yb)) / 20.0), rtol=1e-15)
    # max-min and pseudo divide their spread by the same v
    v = np.mean(yb * (1 - yb)) / 20.0
    assert_allclose(odn.utility_likelihood_noise(y, 'binomial', 20.0, method='max_min')[1], (0.8 ** 2) / v, rtol=1e-14)
    um = odn.utility_likelihood_noise(y, 'binomial', 20.0, method='max_min')
    assert um[2] == np.inf and um[3] == 0.0 and um[4] == 0.0
    # log form and cost
    assert_allclose(odn.utility_likelihood_noise(y, 'binomial', 20.0, log_form=True, cost=2.0)[1],
                    np.log(1 + u[1]) / 2.0, rtol=1e-15)
    # Poisson: lambda < 0, NaN, +inf invalid; lambda = 0 everywhere: 0
    lam = np.abs(y) * 10.0
    lam[2, 0, 1] = -1e-300
    lam[0, 0, 2] = np.inf
    up = odn.utility_likelihood_noise(lam, 'poisson')
    assert up[0] == 0.0 and up[1] == 0.0 and up[2] == 0.0 and up[3] == 0.0 and up[5] == 0.0
    assert_allclose(up[4], np.var(lam[:, 0, 4]) / np.mean(lam[:, 0, 4]), rtol=1e-15)
    # user: nu negative or NaN invalid, +inf allowed (r = 0)
    nv = lambda yy, a: np.where(yy > 0.95, -1.0, np.where(yy < 0.05, np.inf, a * yy))      # noqa: E731
    uu = odn.utility_likelihood_noise(y, nv, 2.0)
    assert_allclose(uu[1], np.var(yb) / np.mean(2.0 * yb), rtol=1e-15)
    assert uu[2] == 0.0                                       # y = 1.0 gives nu = -1
    assert uu[3] == 0.0 and uu[5] == 0.0                      # nu = +inf, var = 0; NaN


@pytest.fixture(scope='module')
def lib(obe_lib):
    return obe_lib


USER = b'''__device__ double user_ll(const double* y, const double* m, const double* a, int n) {
    double s = 0.0;
    for (int c = 0; c < n; ++c) s += (m[c] == 0.0 ? 0.0 : m[c] * log(y[c])) - y[c];
    return s;
}
__device__ double user_var(double y, double a) { return y * a; }'''
MODEL = b'__device__ void mline(const double* s, const double* p, const double* c, double* y) { y[0] = p[0] * s[0] + p[1]; }'


@pytest.mark.parametrize('args', [
    (b'line', None, None, 0, 2, 0, 0, 0, b'poisson', None, None, None),
    (b'lorentzian_dip', None, None, 0, 4, 0, 0, 0, b'binomial', None, None, None),
    (b'lockin_coil', None, None, 0, 3, 0, 0, 0, b'user', USER, b'user_ll', b'user_var'),
    (None, MODEL, b'mline', 1, 2, 2, 0, 1, b'poisson', None, None, None),
], ids=['poisson', 'binomial', 'user_two_channels', 'user_model'])
def test_design_handles_compile(lib, args):
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    rc = lib.obe_model_compile_likelihood_design(*args, C.byref(h), log, len(log))
    if rc == 0:
        lib.obe_model_free(h)
    else:                                      # without a GPU: compiled, then the cubin could not be loaded
        err = lib.obe_last_error()
        assert b'NVRTC' not in err and b'cudaLibraryLoadData' in err, err


def test_design_handle_refusals(lib):
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    # a user likelihood without its noise_var entry
    assert lib.obe_model_compile_likelihood_design(b'line', None, None, 0, 2, 0, 0, 0, b'user', USER, b'user_ll', None,
                                                   C.byref(h), log, len(log)) != 0
    assert b'noise_var' in lib.obe_last_error()
    assert lib.obe_model_compile_likelihood_design(b'line', None, None, 0, 2, 0, 0, 0, b'gamma', None, None, None,
                                                   C.byref(h), log, len(log)) != 0
    assert b'unknown likelihood' in lib.obe_last_error()
    # a noise_var entry that does not compile surfaces its log
    rc = lib.obe_model_compile_likelihood_design(b'line', None, None, 0, 2, 0, 0, 0, b'user', USER, b'user_ll',
                                                 b'no_such_function', C.byref(h), log, len(log))
    assert rc != 0 and b'no_such_function' in lib.obe_last_error()


def test_design_variants_need_no_gpu():
    import optbayesexpt_b200 as obe
    m = obe.builtin('rabi')
    p = m.with_likelihood('poisson')
    d = m.with_likelihood('poisson', 'likelihood')
    assert d is not p and d.design_noise == 'likelihood' and p.design_noise == 'fixed'
    assert m.with_likelihood('poisson', 'likelihood') is d and m.with_likelihood('poisson') is p
    assert d.with_likelihood('poisson', 'likelihood') is d and d.with_likelihood('poisson') is not d
    assert m.with_likelihood('gaussian', 'likelihood') is m             # Gaussian: the fixed variance by definition
    with pytest.raises(ValueError, match='design_noise'):
        m.with_likelihood('poisson', 'adaptive')
    src = '__device__ double f(const double*, const double*, const double*, int) { return 0; }\n' \
          '__device__ double v(double y, double a) { return y; }'
    plain, nv = obe.cuda_likelihood(src, 'f'), obe.cuda_likelihood(src, 'f', noise_var='v')
    assert plain != nv and hash(plain) != hash(nv) and nv == obe.cuda_likelihood(src, 'f', noise_var='v')
    assert hash(nv) == hash(obe.cuda_likelihood(src, 'f', noise_var='v'))
    assert m.with_likelihood(nv, 'likelihood').likelihood == nv
    with pytest.raises(ValueError, match='noise_var'):
        m.with_likelihood(plain, 'likelihood')
    assert m.with_likelihood(plain).likelihood == plain                   # ('fixed' needs no noise_var)


def test_engine_argument_checks_before_the_device():
    import optbayesexpt_b200 as obe
    prior = np.array([np.linspace(2.0, 4.0, 16), np.full(16, 0.5), np.full(16, 0.3)])
    settings = (np.linspace(1.5, 4.5, 8),)
    src = '__device__ double f(const double*, const double*, const double*, int) { return 0; }'
    cases = [
        (dict(likelihood_model='binomial', design_noise='adaptive', design_aux=10.0), 'design_noise'),
        (dict(likelihood_model='binomial', design_noise='likelihood'), 'design_aux'),
        (dict(likelihood_model='poisson', design_noise='likelihood', utility_method='full_kld_utility'), 'full_kld'),
        (dict(likelihood_model=obe.cuda_likelihood(src, 'f'), design_noise='likelihood'), 'noise_var'),
    ]
    for kw, match in cases:
        with pytest.raises(ValueError, match=match):
            obe.OptBayesExpt('lorentzian_dip', settings, prior, (), **kw)


def test_design_aux_setter():
    from optbayesexpt_b200.obe_base import OptBayesExpt
    prop = OptBayesExpt.design_aux
    eng = SimpleNamespace(_design_lik=True, likelihood_model='binomial', n_channels=2)
    prop.fset(eng, 25.0)
    assert_array_equal(eng._design_aux_arr, [25.0, 25.0]) and prop.fget(eng) == 25.0
    prop.fset(eng, (10.0, 30.0))
    assert_array_equal(eng._design_aux_arr, [10.0, 30.0])
    for bad in (0.0, -1.0, np.nan, np.inf, (1.0, 0.0), (1.0, 2.0, 3.0), None):
        with pytest.raises(ValueError):
            prop.fset(eng, bad)
    assert_array_equal(eng._design_aux_arr, [10.0, 30.0])                # (a refused value changes nothing)
    eng.likelihood_model = 'poisson'
    prop.fset(eng, None)                                                # Poisson reads no aux
    assert_array_equal(eng._design_aux_arr, [1.0, 1.0])
