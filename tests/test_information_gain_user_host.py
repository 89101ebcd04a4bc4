"""CPU tests of the information gain of a user count likelihood (cuda_likelihood(..., window=)): the oracle
(oracle/information_gain_user.information_gain_user) against a 50-digit mpmath evaluation of the definition for a
negative binomial, a two-Poisson readout and a beta-binomial, the user-restated Poisson against the built-in oracle,
the windows' tail mass, the engine's argument checks, and the NVRTC compile of a window handle and its error log
(the compile needs no GPU; loading the cubin does)."""
import ctypes as C

import numpy as np
import pytest

from oracle import count_pmfs as cp
from oracle import information_gain as oig
from oracle import information_gain_user as oigu

#: |oracle - exact| <= RTOL I + SQ s sqrt(I): d_k is a difference of two log-pmfs, each with an absolute error of
#: about one ulp of its largest term (lgamma of the counts that carry the mass), so the error of I is about that
#: times sqrt(I) for tight draws, and relative for broad ones.  s = max(1, lgamma(mu + 3 sigma + 1) / 100) over the
#: draws grows with that term: 1 up to about 40 counts, 20 at 400, 850 at 1e4.
RTOL, SQ = 1e-8, 1e-14


def _scale(x, noise_var, aux):
    """s of the bound above, for outputs x whose mean is x (or n x for a beta-binomial's probabilities)"""
    from scipy.special import gammaln
    x = np.asarray(x, dtype=np.float64)
    v = np.maximum(np.asarray(noise_var(x, aux), dtype=np.float64), 0.0)
    mu = x * aux if np.all(x <= 1.0) and aux > 1.0 else x
    top = np.max(mu + 3.0 * np.sqrt(v))
    return max(1.0, float(gammaln(top + 1.0)) / 100.0)


def _mp_logpmf(name, x, y, aux, **kw):
    """log p(y | x, aux) at the current mpmath precision, None where p = 0."""
    import mpmath as mp
    x = mp.mpf(float(x))
    if name == 'negbin':
        r = mp.mpf(aux)
        if x == 0:
            return mp.mpf(0) if y == 0 else None
        return mp.loggamma(y + r) - mp.loggamma(r) - mp.loggamma(y + 1) + r * mp.log(r / (r + x)) + y * mp.log(x / (r + x))
    if name == 'readout':
        lb, ld = mp.mpf(kw['lam_b']), mp.mpf(kw['lam_d'])
        p = x * mp.exp(y * mp.log(lb) - lb) + (1 - x) * mp.exp(y * mp.log(ld) - ld)
        return None if p == 0 else mp.log(p) - mp.loggamma(y + 1)
    if name == 'betabinom':
        n, phi = int(aux), mp.mpf(kw['phi'])
        if x == 0 or x == 1:
            return mp.mpf(0) if y == (0 if x == 0 else n) else None
        a, b = x * phi, (1 - x) * phi
        return (mp.loggamma(n + 1) - mp.loggamma(y + 1) - mp.loggamma(n - y + 1) + mp.loggamma(y + a)
                + mp.loggamma(n - y + b) - mp.loggamma(n + phi) - mp.loggamma(a) - mp.loggamma(b) + mp.loggamma(phi))
    if name == 'poisson':
        if x == 0:
            return mp.mpf(0) if y == 0 else None
        return y * mp.log(x) - x - mp.loggamma(y + 1)
    raise ValueError(name)


def _mp_information_gain(name, x, aux, hi, **kw):
    """I = (1/K) sum_k sum_y p_k log(p_k / pbar) at 50 digits over the counts 0 .. hi."""
    import mpmath as mp
    mp.mp.dps = 50
    K = len(x)
    total = mp.mpf(0)
    for y in range(0, int(hi) + 1):
        ps = []
        for v in x:
            lp = _mp_logpmf(name, v, y, aux, **kw)
            ps.append(mp.mpf(0) if lp is None else mp.exp(lp))
        pbar = mp.fsum(ps) / K
        if pbar == 0:
            continue
        total += mp.fsum(p * mp.log(p / pbar) for p in ps if p > 0)
    return float(total / K)


def _draws(kind, k, level, spread, seed):
    """K outputs around `level` with relative (mean) or logit (probability) spread `spread`."""
    z = np.random.default_rng(seed).standard_normal(k)
    if kind == 'mean':
        return level * np.exp(spread * z)
    logit = np.log(level / (1.0 - level)) + spread * z
    return 1.0 / (1.0 + np.exp(-logit))


CASES = [
    # negative binomial: (shape r, mean, spread, K); r 1 .. 50, means 0.01 .. 1e3
    ('negbin', dict(r=1.0), 0.01, 1.0, 3), ('negbin', dict(r=1.0), 1.0, 1e-5, 3),
    ('negbin', dict(r=5.0), 1.0, 1e-6, 2), ('negbin', dict(r=2.5), 10.0, 0.5, 30),
    ('negbin', dict(r=1.0), 100.0, 1e-6, 2), ('negbin', dict(r=20.0), 100.0, 0.3, 3),
    ('negbin', dict(r=50.0), 1e3, 0.3, 3), ('negbin', dict(r=50.0), 1e3, 1e-6, 2),
    # two-Poisson readout: P(bright) = x, lam_d 0.1 .. 2, lam_b 3 .. 30
    ('readout', dict(lam_d=0.1, lam_b=3.0), 0.5, 1.0, 3), ('readout', dict(lam_d=0.5, lam_b=3.0), 0.3, 1e-6, 30),
    ('readout', dict(lam_d=2.0, lam_b=30.0), 0.7, 0.5, 3), ('readout', dict(lam_d=1.0, lam_b=10.0), 0.1, 1e-7, 2),
    ('readout', dict(lam_d=0.5, lam_b=3.0), 0.999, 2.0, 30),
    # beta-binomial, n = 1 .. 100
    ('betabinom', dict(phi=20.0, n=1.0), 0.3, 1.0, 3), ('betabinom', dict(phi=5.0, n=10.0), 0.5, 1e-6, 2),
    ('betabinom', dict(phi=20.0, n=100.0), 0.2, 0.5, 30), ('betabinom', dict(phi=100.0, n=100.0), 0.6, 1e-7, 3),
]


def _setup(name, kw):
    """(logpmf, noise_var, window, aux, mp keywords) of a case"""
    if name == 'negbin':
        _, _, _, _, lp, nv, win = cp.pmf('negbin')
        return lp, nv, win, kw['r'], {}
    if name == 'readout':
        lp, nv, win = cp.readout(kw['lam_d'], kw['lam_b'])
        return lp, nv, win, 1.0, kw
    lp, nv, win = cp.betabinom(kw['phi'])
    return lp, nv, win, kw['n'], dict(phi=kw['phi'])


@pytest.mark.parametrize('name,kw,level,spread,k', CASES,
                         ids=[f'{c[0]}-{"-".join(f"{a}{b:g}" for a, b in c[1].items())}-{c[2]:g}-{c[3]:g}-K{c[4]}'
                              for c in CASES])
def test_oracle_against_mpmath(name, kw, level, spread, k):
    lp, nv, win, aux, mkw = _setup(name, kw)
    x = _draws('mean' if name == 'negbin' else 'prob', k, level, spread, seed=k)
    got = oigu.information_gain_user(lp, win, x[:, None], aux, noise_var=nv)[0]
    _, hi = win(x, aux)
    want = _mp_information_gain(name, x, aux, np.max(hi), **mkw)
    assert 0.0 < want <= np.log(k) + 1e-15
    assert abs(got - want) <= RTOL * want + SQ * _scale(x, nv, aux) * np.sqrt(want), (got, want)
    if spread <= 1e-5:
        assert want < 1e-8                               # (the tight cases reach I of 1e-10 .. 1e-14)


@pytest.mark.parametrize('name,kw,x', [
    ('readout', dict(lam_d=0.5, lam_b=3.0), [0.0, 1.0, 0.0]),           # point masses of the mixture weight
    ('readout', dict(lam_d=0.2, lam_b=20.0), [0.0, 0.4, 1.0]),
    ('readout', dict(lam_d=0.5, lam_b=3.0), [0.0, 0.0, 1e-9]),
    ('negbin', dict(r=3.0), [0.0, 0.0, 4.0]),                            # a point mass at 0
    ('betabinom', dict(phi=20.0, n=10.0), [0.0, 1.0, 0.5]),             # point masses at 0 and n
    ('betabinom', dict(phi=20.0, n=10.0), [0.0, 1.0, 1.0]),             # disjoint supports: the entropy of the split
])
def test_oracle_point_masses(name, kw, x):
    lp, nv, win, aux, mkw = _setup(name, kw)
    x = np.asarray(x)
    got = oigu.information_gain_user(lp, win, x[:, None], aux, noise_var=nv)[0]
    want = _mp_information_gain(name, x, aux, np.max(win(x, aux)[1]), **mkw)
    assert abs(got - want) <= RTOL * want + SQ * _scale(x, nv, aux) * np.sqrt(want) + 1e-15, (got, want)


def test_user_poisson_matches_the_builtin_oracle():
    """The Poisson restated as a user pmf, with the built-in's windows: the same I as the built-in oracle."""
    g = np.random.default_rng(4)
    for level in (0.01, 1.0, 100.0, 1e4):
        for spread in (1.0, 1e-3, 1e-6):
            for k in (2, 30):
                x = level * np.exp(spread * g.standard_normal(k))
                want = oig.information_gain_from_draws(x[:, None], 'poisson')[0]
                got = oigu.information_gain_user(cp.poisson_logpmf, cp.poisson_window, x[:, None], 1.0,
                                                noise_var=cp.poisson_var)[0]
                tol = RTOL * want + SQ * _scale(x, cp.poisson_var, 1.0) * np.sqrt(want)
                assert abs(got - want) <= tol, (level, spread, k, got, want)
    x = np.array([0.0, 2.0, 2.0 * (1 + 1e-9)])
    assert abs(oigu.information_gain_user(cp.poisson_logpmf, cp.poisson_window, x[:, None], 1.0)[0]
               - oig.information_gain_from_draws(x[:, None], 'poisson')[0]) < 1e-14


def test_windows_hold_the_mass():
    """each window leaves out less than 1e-17 of its component's mass"""
    from scipy.stats import nbinom, poisson
    for r in (1.0, 2.5, 10.0, 50.0):
        for m in (0.01, 1.0, 30.0, 1e3):
            _, hi = cp.negbin_window(np.array([m]), r)
            assert nbinom.sf(hi[0], r, r / (r + m)) < 1e-17, (r, m)
    for lam_d, lam_b in ((0.1, 3.0), (2.0, 30.0)):
        lp, nv, win = cp.readout(lam_d, lam_b)
        _, hi = win(np.array([1.0]))
        assert poisson.sf(hi[0], lam_b) < 1e-17 and poisson.sf(hi[0], lam_d) < 1e-17
    # and the numpy pmfs are normalised over them
    for name, kw, x in (('negbin', dict(r=2.0), 40.0), ('readout', dict(lam_d=0.5, lam_b=3.0), 0.4),
                        ('betabinom', dict(phi=7.0, n=50.0), 0.3)):
        lp, nv, win, aux, _ = _setup(name, kw)
        lo, hi = win(np.array([x]), aux)
        y = np.arange(lo[0], hi[0] + 1.0)
        assert abs(np.sum(np.exp(lp(x, y, aux))) - 1.0) < 1e-13, name


def test_oracle_rules():
    lp, nv, win = cp.readout(0.5, 3.0)
    y = np.full((4, 5), 0.5)
    y[:, 1] = [0.1, 0.2, 0.3, 0.9]
    y[2, 2] = 1.0 + 1e-12                                # P > 1: the noise variance is negative
    y[0, 3] = np.nan
    u = oigu.information_gain_user(lp, win, y, 1.0, noise_var=nv, cost=np.array([1.0, 2.0, 1.0, 1.0, 1.0]))
    assert u[0] == 0.0 and u[2] == 0.0 and u[3] == 0.0 and u[4] == 0.0
    assert u[1] == oigu.information_gain_user(lp, win, y[:, 1:2], 1.0, noise_var=nv)[0] / 2.0 > 0.0
    x = np.array([[0.2], [0.4], [0.6]])

    def windows(lo, hi):
        return lambda v, a: (np.full(v.shape, lo), np.full(v.shape, hi))
    assert oigu.information_gain_user(lp, windows(0.0, 60.0), x, 1.0)[0] > 0.0
    for lo, hi in ((np.nan, 10.0), (0.0, np.nan), (0.5, 10.0), (0.0, 10.5), (-1.0, 10.0), (5.0, 4.0),
                   (0.0, 2.0 ** 53 + 2.0), (0.0, float(oigu.USER_MAX_COUNTS))):
        assert oigu.information_gain_user(lp, windows(lo, hi), x, 1.0)[0] == 0.0, (lo, hi)
    assert oigu.information_gain_user(lp, windows(0.0, float(oigu.USER_MAX_COUNTS - 1)), x[:2], 1.0)[0] > 0.0

    def nan_at_7(v, yy, a):
        out = lp(v, yy, a)
        return np.where(yy == 7.0, np.nan, out)

    def inf_at_7(v, yy, a):
        out = lp(v, yy, a)
        return np.where(yy == 7.0, np.inf, out)
    assert oigu.information_gain_user(nan_at_7, win, x, 1.0)[0] == 0.0
    assert oigu.information_gain_user(inf_at_7, win, x, 1.0)[0] == 0.0


# ---------------------------------------------------------------------------------------------------------------
# the engine's argument checks (before anything reaches the device)
# ---------------------------------------------------------------------------------------------------------------
def test_cuda_likelihood_window_identity():
    import optbayesexpt_b200 as obe
    a = obe.cuda_likelihood('src', 'f', noise_var='v', window='w')
    assert a == obe.cuda_likelihood('src', 'f', noise_var='v', window='w')
    assert hash(a) == hash(obe.cuda_likelihood('src', 'f', noise_var='v', window='w'))
    assert a != obe.cuda_likelihood('src', 'f', noise_var='v')
    assert a != obe.cuda_likelihood('src', 'f', noise_var='v', window='w2')
    assert "window='w'" in repr(a) and 'window' not in repr(obe.cuda_likelihood('src', 'f', noise_var='v'))
    m = obe.builtin('lorentzian_dip')
    ia = m.with_likelihood(a, 'likelihood')
    assert m.with_likelihood(obe.cuda_likelihood('src', 'f', noise_var='v', window='w'), 'likelihood') is ia
    assert m.with_likelihood(obe.cuda_likelihood('src', 'f', noise_var='v'), 'likelihood') is not ia


def test_engine_refusals():
    import optbayesexpt_b200 as obe
    prior = np.array([np.linspace(2.0, 4.0, 16), np.full(16, 0.5), np.full(16, 0.3)])
    settings = (np.linspace(1.5, 4.5, 8),)
    src, entry, nv, win = cp.pmf('readout')[:4]
    ig = dict(utility_method='information_gain')
    # a noise_var without a window keeps the old refusal and its message
    with pytest.raises(ValueError, match='poisson'):
        obe.OptBayesExpt('lorentzian_dip', settings, prior, (), design_noise='likelihood', **ig,
                         likelihood_model=obe.cuda_likelihood(src, entry, noise_var=nv))
    # a window needs the likelihood-aware design, which needs noise_var
    with pytest.raises(ValueError, match="design_noise='likelihood'"):
        obe.OptBayesExpt('lorentzian_dip', settings, prior, (), **ig,
                         likelihood_model=obe.cuda_likelihood(src, entry, noise_var=nv, window=win))
    with pytest.raises(ValueError, match='noise_var'):
        obe.OptBayesExpt('lorentzian_dip', settings, prior, (), design_noise='likelihood', **ig,
                         likelihood_model=obe.cuda_likelihood(src, entry, window=win))
    two = obe.cuda_source('__device__ void m2(const double* s, const double* p, const double* c, double* y) '
                          '{ y[0] = p[0]; y[1] = p[1]; }', 'm2', 1, 3, 0, 2)
    with pytest.raises(ValueError, match='single-channel'):
        obe.OptBayesExpt(two, settings, prior, (), design_noise='likelihood', **ig,
                         likelihood_model=obe.cuda_likelihood(src, entry, noise_var=nv, window=win))


@pytest.fixture(scope='module')
def lib(obe_lib):
    return obe_lib


def _compile(lib, source, entry, nv, win, model=b'lorentzian_dip', d=4):
    h = C.c_void_p()
    log = C.create_string_buffer(1 << 16)
    rc = lib.obe_model_compile_likelihood_window(model, None, None, 0, d, 0, 0, 0, b'user', source.encode(),
                                                 entry.encode(), nv.encode(), None if win is None else win.encode(),
                                                 C.byref(h), log, len(log))
    return rc, h, log.value.decode(errors='replace'), lib.obe_last_error()


@pytest.mark.parametrize('name', ['poisson', 'negbin', 'readout', 'betabinom'])
def test_window_handles_compile(lib, name):
    """The design module of a user likelihood with a window, obe_k_utility_info included, compiles."""
    src, entry, nv, win = cp.pmf(name)[:4]
    rc, h, _, err = _compile(lib, src, entry, nv, win)
    if rc == 0:
        lib.obe_model_free(h)
    else:                                      # without a GPU: compiled, then the cubin could not be loaded
        assert b'NVRTC' not in err and b'cudaLibraryLoadData' in err, err


def test_window_compile_errors(lib):
    src, entry, nv, win = cp.pmf('readout')[:4]
    broken = src.replace('*hi = floor(', '*hi = floor_not_a_function(')
    rc, _, log, err = _compile(lib, broken, entry, nv, win)
    assert rc != 0 and b'NVRTC' in err and 'floor_not_a_function' in log, (log, err)
    rc, _, log, err = _compile(lib, src, entry, nv, 'no_such_window')
    assert rc != 0 and 'no_such_window' in log, log
    # a window with a built-in likelihood is refused
    h = C.c_void_p()
    rc = lib.obe_model_compile_likelihood_window(b'rabi', None, None, 0, 2, 0, 0, 0, b'poisson', None, None, None,
                                                 b'w', C.byref(h), None, 0)
    assert rc != 0 and b'user likelihood only' in lib.obe_last_error()
