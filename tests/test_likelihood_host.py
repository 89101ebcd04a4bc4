"""CPU tests of the non-Gaussian likelihoods: the oracle against scipy.stats, the record checks of the engine, and
the NVRTC compile of every likelihood handle (the compile needs no GPU; loading the cubin does)."""
import ctypes as C

import numpy as np
import pytest
from numpy.testing import assert_allclose

from oracle import likelihoods as olk


def test_oracle_poisson_equals_scipy():
    from scipy.stats import poisson
    lam = np.concatenate([[0.0, 1e-300, 1e-3], np.linspace(0.01, 80.0, 400), [1e6, 1.0001e6]])
    for k in (0, 1, 2, 17, 60, 1000000):
        want = poisson.pmf(k, lam)
        got = olk.likelihood_poisson((lam,), float(k))
        ok = want > 1e-300
        assert_allclose(got[ok], want[ok], rtol=1e-12 if k < 1000 else 1e-8)
    # edge cases: xlogy(0, 0) = 0, invalid means weigh 0
    got = olk.likelihood_poisson((np.array([0.0, 0.0, -1.0, np.nan, np.inf]),), 0.0)
    assert list(got) == [1.0, 1.0, 0.0, 0.0, 0.0]
    got = olk.likelihood_poisson((np.array([0.0, -1.0, np.nan, np.inf]),), 3.0)
    assert list(got) == [0.0, 0.0, 0.0, 0.0]


def test_oracle_binomial_equals_scipy():
    from scipy.stats import binom
    p = np.concatenate([[0.0, 1.0], np.linspace(1e-4, 1 - 1e-4, 500)])
    for k, n in ((0, 0), (0, 5), (5, 5), (2, 5), (37, 100), (400, 1000)):
        want = binom.pmf(k, n, p)
        got = olk.likelihood_binomial((p,), float(k), float(n))
        ok = want > 1e-300
        assert_allclose(got[ok], want[ok], rtol=1e-12 if n < 1000 else 1e-10)
    got = olk.likelihood_binomial((np.array([0.0, 1.0, -1e-17, 1.0 + 2e-16, np.nan]),), 0.0, 4.0)
    assert list(got) == [1.0, 0.0, 0.0, 0.0, 0.0]
    got = olk.likelihood_binomial((np.array([0.0, 1.0]),), 4.0, 4.0)
    assert list(got) == [0.0, 1.0]


def test_oracle_choke_and_channels():
    y = (np.array([2.0, 3.0]), np.array([5.0, 0.5]))
    want = olk.likelihood_poisson((y[0],), 1.0) * olk.likelihood_poisson((y[1],), 4.0)
    assert_allclose(olk.likelihood_poisson(y, (1.0, 4.0)), want, rtol=1e-14)
    assert_allclose(olk.likelihood_poisson(y, (1.0,)), olk.likelihood_poisson((y[0],), 1.0), rtol=0)  # zip truncation
    assert_allclose(olk.likelihood_poisson(y, (1.0, 4.0), choke=0.5), np.exp(0.5 * np.log(want)), rtol=1e-14)


def test_likelihood_selection_needs_no_gpu():
    import optbayesexpt_b200 as obe
    m = obe.builtin('rabi')
    assert m.likelihood == 'gaussian'
    p = m.with_likelihood('poisson')
    assert p.likelihood == 'poisson' and m.with_likelihood('poisson') is p and p.with_likelihood('gaussian') is not p
    lk = obe.cuda_likelihood('__device__ double f(const double*, const double*, const double*, int) { return 0; }', 'f')
    assert m.with_likelihood(lk).likelihood == lk
    with pytest.raises(ValueError):
        m.with_likelihood('gamma')
    with pytest.raises(TypeError):
        m.with_likelihood(None)


USER = b'''__device__ double user_ll(const double* y, const double* m, const double* a, int n) {
    double s = 0.0;
    for (int c = 0; c < n; ++c) s += -0.5 * (y[c] - m[c]) * (y[c] - m[c]) / (a[c] * a[c]);
    return s;
}'''
MODEL = b'__device__ void mline(const double* s, const double* p, const double* c, double* y) { y[0] = p[0] * s[0] + p[1]; }'


@pytest.mark.parametrize('args', [
    (b'line', None, None, 0, 2, 0, 0, 0, b'poisson', None, None),
    (b'lorentzian_dip', None, None, 0, 4, 0, 0, 0, b'binomial', None, None),
    (b'lockin_coil', None, None, 0, 3, 0, 0, 0, b'user', USER, b'user_ll'),
    (None, MODEL, b'mline', 1, 2, 2, 0, 1, b'poisson', None, None),
], ids=['poisson', 'binomial', 'user_two_channels', 'user_model'])
def test_likelihood_handles_compile(obe_lib, args):
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    rc = obe_lib.obe_model_compile_likelihood(*args, C.byref(h), log, len(log))
    if rc == 0:
        obe_lib.obe_model_free(h)
    else:                                      # without a GPU: compiled, then the cubin could not be loaded
        err = obe_lib.obe_last_error()
        assert b'NVRTC' not in err and b'cudaLibraryLoadData' in err, err


def test_likelihood_handle_refusals(obe_lib):
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    assert obe_lib.obe_model_compile_likelihood(b'line', None, None, 0, 2, 0, 0, 0, b'gamma', None, None,
                                                C.byref(h), log, len(log)) != 0
    assert b'unknown likelihood' in obe_lib.obe_last_error()
    assert obe_lib.obe_model_compile_likelihood(b'no_such', None, None, 0, 2, 0, 0, 0, b'poisson', None, None,
                                                C.byref(h), log, len(log)) != 0
    assert obe_lib.obe_model_compile_likelihood(b'line', None, None, 0, 2, 0, 0, 0, b'user', None, None,
                                                C.byref(h), log, len(log)) != 0
    assert obe_lib.obe_model_compile_likelihood(b'lorentzian_dip', None, None, 0, 2, 0, 0, 0, b'poisson', None, None,
                                                C.byref(h), log, len(log)) != 0          # fewer rows than parameters
    rc = obe_lib.obe_model_compile_likelihood(b'line', None, None, 0, 2, 0, 0, 0, b'user',
                                              b'__device__ double bad(const double* y, const double* m, const double* a, '
                                              b'int n) { return undeclared_name; }', b'bad', C.byref(h), log, len(log))
    assert rc != 0 and b'undeclared_name' in obe_lib.obe_last_error() and b'undeclared_name' in log.value


@pytest.mark.parametrize('kind', ['poisson', 'binomial'])
def test_counting_records_are_checked_on_the_host(kind):
    from types import SimpleNamespace

    from optbayesexpt_b200.obe_base import OptBayesExpt
    eng = SimpleNamespace(likelihood_model=kind, n_channels=1)
    spec = lambda rec: OptBayesExpt._counting_spec(eng, rec)          # noqa: E731
    good = [((0.5,), 3.0, 10.0), ((0.5,), 0.0, 0.0), ((0.5,), np.array([3.0]), np.array([3.0]))]
    bad = [((0.5,), -1.0, 10.0), ((0.5,), np.nan, 10.0), ((0.5,), np.inf, 10.0), ((0.5,), 2.5, 10.0)]
    if kind == 'poisson':
        good += [((0.5,), 7.0)]
    else:
        bad += [((0.5,), 11.0, 10.0), ((0.5,), 1.0, np.inf), ((0.5,), 1.0), ((0.5,), 1.0, 2.5)]
    for rec in good:
        k, n, ni, n_lik = spec(rec)
        assert n_lik == 1 and ni is None and float(k[0]) == float(np.ravel(rec[1])[0])
        assert (n is None) == (kind == 'poisson')
    for rec in bad:
        with pytest.raises(ValueError):
            spec(rec)
