"""CPU tests of the information-gain utility (utility_method='information_gain'): the oracle against a 50-digit
mpmath evaluation of the definition, its closed forms, the argument checks of the engine and of the design_aux
setter, and the NVRTC compile of the design handles that carry the kernel (the compile needs no GPU; loading the
cubin does)."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import information_gain as oig


def _mp_information_gain(x, kind, n=None):
    """I = (1/K) sum_k sum_y p_k log(p_k / pbar) at 50 digits, over a window wider than the oracle's."""
    import mpmath as mp
    mp.mp.dps = 50
    x = [mp.mpf(float(v)) for v in x]
    K = len(x)
    if kind == 'poisson':
        lo = max(0, int(min(float(v) - 12.0 * float(mp.sqrt(v)) - 60.0 for v in x)))
        hi = int(max(float(v) + 12.0 * float(mp.sqrt(v)) + 60.0 for v in x))
    else:
        lo, hi = 0, int(n)
    total = mp.mpf(0)
    for y in range(lo, hi + 1):
        ps = []
        for v in x:
            if kind == 'poisson':
                if v == 0:
                    ps.append(mp.mpf(1) if y == 0 else mp.mpf(0))
                else:
                    ps.append(mp.exp(y * mp.log(v) - v - mp.loggamma(y + 1)))
            else:
                if v == 0 or v == 1:
                    ps.append(mp.mpf(1) if y == (0 if v == 0 else n) else mp.mpf(0))
                else:
                    ps.append(mp.exp(mp.loggamma(n + 1) - mp.loggamma(y + 1) - mp.loggamma(n - y + 1)
                                     + y * mp.log(v) + (n - y) * mp.log1p(-v)))
        pbar = mp.fsum(ps) / K
        if pbar == 0:
            continue
        total += mp.fsum(p * mp.log(p / pbar) for p in ps if p > 0)
    return float(total / K)


def _draws(kind, k, level, spread, seed=0, n=None):
    """K outputs around `level` (a mean count, or a probability) with relative spread `spread`."""
    g = np.random.default_rng(seed)
    z = g.standard_normal(k)
    if kind == 'poisson':
        return level * np.exp(spread * z)
    logit = np.log(level / (1.0 - level)) + spread * z
    return 1.0 / (1.0 + np.exp(-logit))


CASES = [
    # Poisson: mean counts 0.01 .. 1e4, K = 2 / 3 / 30, broad and tight draws
    ('poisson', 2, 0.01, 1.0, None), ('poisson', 3, 0.01, 1e-5, None), ('poisson', 30, 0.01, 0.5, None),
    ('poisson', 2, 1.0, 1e-6, None), ('poisson', 3, 1.0, 1.0, None), ('poisson', 30, 1.0, 1e-5, None),
    ('poisson', 30, 1.0, 2.0, None),
    ('poisson', 2, 100.0, 1e-7, None), ('poisson', 3, 100.0, 0.5, None), ('poisson', 30, 100.0, 1e-6, None),
    ('poisson', 30, 100.0, 0.3, None),
    ('poisson', 2, 1e4, 1e-8, None), ('poisson', 3, 1e4, 0.05, None), ('poisson', 30, 1e4, 1e-7, None),
    # binomial: n = 1 / 10 / 1000
    ('binomial', 2, 0.3, 1e-6, 1), ('binomial', 3, 0.5, 2.0, 1), ('binomial', 30, 0.4, 1e-4, 1),
    ('binomial', 2, 0.7, 1e-7, 10), ('binomial', 3, 0.2, 1.5, 10), ('binomial', 30, 0.5, 1e-5, 10),
    ('binomial', 30, 0.5, 1.0, 10),
    ('binomial', 2, 0.5, 1e-8, 1000), ('binomial', 3, 0.1, 1.0, 1000), ('binomial', 30, 0.6, 1e-7, 1000),
]


@pytest.mark.parametrize('kind,k,level,spread,n', CASES,
                         ids=[f'{c[0]}-K{c[1]}-{c[2]:g}-{c[3]:g}' + (f'-n{c[4]}' if c[4] else '') for c in CASES])
def test_oracle_against_mpmath(kind, k, level, spread, n):
    x = _draws(kind, k, level, spread, seed=k, n=n)
    got = oig.information_gain_from_draws(x[:, None], kind, n)[0]
    want = _mp_information_gain(x, kind, n)
    assert 0.0 < want <= np.log(k) + 1e-15
    assert abs(got - want) <= 1e-12 * want, (got, want)
    if spread <= 1e-5:
        assert want < 1e-3                               # (the tight cases reach I of 1e-6 .. 1e-14)


POINT_CASES = [
    ('poisson', [0.0, 0.0, 3.0]), ('poisson', [0.0, 1e-3, 2.5, 40.0]), ('poisson', [0.0, 5.0, 5.0 * (1 + 1e-9)]),
    ('binomial', [0.0, 1.0, 0.0]), ('binomial', [0.0, 1.0, 0.5]), ('binomial', [1.0, 0.999, 0.2]),
]


@pytest.mark.parametrize('kind,x', POINT_CASES)
@pytest.mark.parametrize('n', [1, 10])
def test_oracle_point_masses(kind, x, n):
    x = np.asarray(x)
    got = oig.information_gain_from_draws(x[:, None], kind, n)[0]
    want = _mp_information_gain(x, kind, n)
    assert abs(got - want) <= 1e-12 * want + 1e-15, (got, want)


def test_closed_forms():
    # identical draws: exactly 0, whatever the level
    for kind, x in (('poisson', 7.3), ('poisson', 0.0), ('binomial', 0.25), ('binomial', 1.0)):
        assert oig.information_gain_from_draws(np.full((5, 1), x), kind, 12)[0] == 0.0
    # Poisson means far apart: log K (to the rounding of log-pmfs of order 1e3 that cancel in the weight)
    for k in (2, 3, 30):
        lam = 1e3 * np.arange(1, k + 1) ** 2
        assert abs(oig.information_gain_from_draws(lam[:, None], 'poisson')[0] - np.log(k)) < 1e-11 * np.log(k)
    # K = 2, means lam and lam (1 + delta): I ~ lam delta^2 / 8 to relative O(delta)
    for lam in (1.0, 30.0, 1e3):
        for dl in (1e-2, 1e-3, 1e-4):
            got = oig.information_gain_from_draws(np.array([[lam], [lam * (1 + dl)]]), 'poisson')[0]
            want = lam * dl * dl / 8.0
            assert abs(got / want - 1.0) < 2.0 * dl, (lam, dl, got, want)
    # all draws point masses at 0 and n: the entropy of the split
    got = oig.information_gain_from_draws(np.array([[0.0], [1.0], [1.0]]), 'binomial', 5)[0]
    assert abs(got - (-(1 / 3) * np.log(1 / 3) - (2 / 3) * np.log(2 / 3))) < 1e-15


def test_oracle_rules():
    y = np.full((4, 6), 3.0)
    y[:, 1] = [1.0, 2.0, 3.0, 4.0]
    y[2, 2] = -1e-300                                    # a negative rate: 0
    y[0, 3] = np.nan
    y[1, 4] = np.inf
    u = oig.information_gain_from_draws(y, 'poisson', cost=np.array([1.0, 2.0, 1.0, 1.0, 1.0, 1.0]))
    assert u[0] == 0.0 and u[2] == 0.0 and u[3] == 0.0 and u[4] == 0.0 and u[5] == 0.0
    assert u[1] == oig.information_gain_from_draws(y[:, 1:2], 'poisson')[0] / 2.0
    p = np.full((3, 3), 0.5)
    p[:, 1] = [0.2, 0.5, 1.0 + 1e-12]
    p[:, 2] = [0.2, 0.5, 0.9]
    ub = oig.information_gain_from_draws(p, 'binomial', 20)
    assert ub[0] == 0.0 and ub[1] == 0.0 and ub[2] > 0.0
    for bad in (0.0, 2.5, np.nan):
        with pytest.raises(ValueError):
            oig.information_gain_from_draws(p, 'binomial', bad)
    # the windows cover the mass: beyond them a component's pmf is below 1e-17
    from scipy.stats import binom, poisson
    for lam in (0.01, 1.0, 100.0, 1e4):
        lo, hi = oig.windows(np.array([lam]), 'poisson')
        assert poisson.cdf(lo[0] - 1, lam) + poisson.sf(hi[0], lam) < 1e-17
    for n, q in ((10, 0.5), (1000, 0.01), (1000, 0.5)):
        lo, hi = oig.windows(np.array([q]), 'binomial', n)
        assert binom.cdf(lo[0] - 1, n, q) + binom.sf(hi[0], n, q) < 1e-17


def test_logpmf_against_scipy_and_mpmath():
    import mpmath as mp
    from scipy.stats import binom, poisson
    mp.mp.dps = 40
    for lam in (0.01, 1.0, 37.5, 1e4):
        y = np.arange(0.0, lam + 10.0 * np.sqrt(lam) + 30.0)
        got = oig.logpmf(y, 'poisson', lam)
        np.testing.assert_allclose(got, poisson.logpmf(y, lam), rtol=1e-12, atol=1e-9)
        for yy in y[::max(1, len(y) // 25)]:
            want = float(yy * mp.log(lam) - lam - mp.loggamma(yy + 1))
            assert abs(oig.logpmf(np.array([yy]), 'poisson', lam)[0] - want) <= 1e-14 * max(1.0, abs(want))
    for n, q in ((1, 0.3), (10, 0.01), (1000, 0.5), (1000, 0.999)):
        y = np.arange(0.0, n + 1.0)
        got = oig.logpmf(y, 'binomial', q, float(n))
        np.testing.assert_allclose(got, binom.logpmf(y, n, q), rtol=1e-12, atol=1e-9)
        for yy in y[::max(1, len(y) // 25)]:
            want = float(mp.loggamma(n + 1) - mp.loggamma(yy + 1) - mp.loggamma(n - yy + 1) + yy * mp.log(q)
                         + (n - yy) * mp.log1p(-q))
            assert abs(oig.logpmf(np.array([yy]), 'binomial', q, float(n))[0] - want) <= 1e-14 * max(1.0, abs(want))


def test_phi_series_matches_closed_form():
    import mpmath as mp
    mp.mp.dps = 40
    for d in (-0.4999, -1e-3, -1e-9, 1e-12, 3e-4, 0.2, 0.4999, 0.5, 2.0, -3.0, -40.0):
        want = float(mp.mpf(d) * mp.exp(d) - mp.expm1(d))
        assert abs(oig.phi(np.array([d]))[0] - want) <= 1e-15 * want
    assert oig.phi(np.array([-np.inf]))[0] == 1.0


# ---------------------------------------------------------------------------------------------------------------
# the engine's argument checks (before anything reaches the device)
# ---------------------------------------------------------------------------------------------------------------
def test_engine_refusals():
    import optbayesexpt_b200 as obe
    prior = np.array([np.linspace(2.0, 4.0, 16), np.full(16, 0.5), np.full(16, 0.3)])
    settings = (np.linspace(1.5, 4.5, 8),)
    src = '__device__ double f(const double*, const double*, const double*, int) { return 0; }\n' \
          '__device__ double v(double y, double a) { return y; }'
    ig = dict(utility_method='information_gain')
    cases = [
        (dict(design_noise='likelihood', **ig), 'poisson'),                                       # Gaussian
        (dict(likelihood_model=obe.cuda_likelihood(src, 'f', noise_var='v'), design_noise='likelihood', **ig),
         'poisson'),
        (dict(likelihood_model='poisson', **ig), "design_noise='likelihood'"),
        (dict(likelihood_model='binomial', design_aux=10.0, **ig), "design_noise='likelihood'"),
        (dict(likelihood_model='binomial', design_noise='likelihood', design_aux=2.5, **ig), 'integer'),
        (dict(likelihood_model='binomial', design_noise='likelihood', design_aux=0.5, **ig), 'integer'),
        (dict(likelihood_model='binomial', design_noise='likelihood', **ig), 'design_aux'),
    ]
    for kw, match in cases:
        with pytest.raises(ValueError, match=match):
            obe.OptBayesExpt('lorentzian_dip', settings, prior, (), **kw)
    two = obe.cuda_source('__device__ void m2(const double* s, const double* p, const double* c, double* y) '
                          '{ y[0] = p[0]; y[1] = p[1]; }', 'm2', 1, 3, 0, 2)
    with pytest.raises(ValueError, match='single-channel'):
        obe.OptBayesExpt(two, settings, prior, (), likelihood_model='poisson', design_noise='likelihood', **ig)


def test_design_aux_setter_checks_trials():
    from optbayesexpt_b200.obe_base import OptBayesExpt
    prop = OptBayesExpt.design_aux
    eng = SimpleNamespace(_design_lik=True, likelihood_model='binomial', n_channels=1, _utility_code=4)
    prop.fset(eng, 25.0)
    assert eng._design_aux_arr.tolist() == [25.0]
    for bad in (2.5, 0.5, 1.0 + 1e-9, np.nan, np.inf, 0.0, -3.0, None):
        with pytest.raises(ValueError):
            prop.fset(eng, bad)
    assert prop.fget(eng) == 25.0                                        # (a refused value changes nothing)
    prop.fset(eng, 1)
    assert eng._design_aux_arr.tolist() == [1.0]
    eng._utility_code = 0                                                 # another utility: any positive aux
    prop.fset(eng, 2.5)
    eng._utility_code, eng.likelihood_model = 4, 'poisson'                # Poisson reads no trial count
    prop.fset(eng, 2.5)


@pytest.fixture(scope='module')
def lib(obe_lib):
    return obe_lib


@pytest.mark.parametrize('args', [
    (b'rabi', None, None, 0, 2, 0, 0, 0, b'poisson', None, None, None),
    (b'lorentzian_hwhm', None, None, 0, 3, 0, 0, 0, b'poisson', None, None, None),
    (b'lorentzian_dip', None, None, 0, 4, 0, 0, 0, b'binomial', None, None, None),
], ids=['poisson_rabi', 'poisson_peak', 'binomial_dip'])
def test_design_handles_with_the_kernel_compile(lib, args):
    """The design module, obe_k_utility_info included, compiles for Poisson and binomial models."""
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    rc = lib.obe_model_compile_likelihood_design(*args, C.byref(h), log, len(log))
    if rc == 0:
        lib.obe_model_free(h)
    else:                                      # without a GPU: compiled, then the cubin could not be loaded
        err = lib.obe_last_error()
        assert b'NVRTC' not in err and b'cudaLibraryLoadData' in err, err

