"""CPU tests of the batched engines' count likelihoods: the restated count sampler (oracle/batched_counts.py) against
scipy's distributions on both sides of each algorithm switch, its point masses and invalid inputs, the independence of
its Philox stream, the host checks of batched count records and of the simulator's arguments, and the refusals of the
constructor (all before any device is touched)."""
import re
from pathlib import Path

import numpy as np
import pytest
from scipy import stats

from optbayesexpt_b200.batched import BatchedOptBayesExpt, count_record, simulator_noise
from oracle import batched_counts as obc

N_DRAWS = 1_000_000
POISSON = [1e-3, 0.5, 3.0, 9.99, 10.0, 37.0, 1e3, 1e6]
BINOMIAL = [(1, 0.3), (10, 0.05), (40, 0.5), (1000, 0.002), (1000, 0.97), (10 ** 6, 0.4), (20, 0.9)]


def chi2_pvalue(k, pmf, lo, hi):
    """Chi-square goodness of fit of the integer draws k to pmf over [lo, hi]; bins are merged from the left until
    each expects >= 5 draws, the remainder joins the last bin, and the mass outside [lo, hi] is folded into the ends."""
    ks = np.arange(lo, hi + 1)
    expect = pmf(ks) * len(k)
    obs = np.bincount((np.clip(k, lo, hi) - lo).astype(np.int64), minlength=hi - lo + 1)
    e_bins, o_bins, ce, co = [], [], 0.0, 0
    for ee, oo in zip(expect, obs):
        ce, co = ce + ee, co + oo
        if ce >= 5:
            e_bins.append(ce)
            o_bins.append(co)
            ce, co = 0.0, 0
    e_bins[-1] += ce
    o_bins[-1] += co
    e = np.array(e_bins)
    o = np.array(o_bins)
    e *= o.sum() / e.sum()
    return stats.chisquare(o, e).pvalue if len(e) > 1 else 1.0


def poisson_window(lam):
    return int(max(0.0, lam - 12 * np.sqrt(lam) - 5)), int(lam + 12 * np.sqrt(lam) + 20)


def binomial_window(n, p):
    mu, sd = n * p, np.sqrt(n * p * (1 - p))
    return int(max(0.0, mu - 12 * sd - 5)), int(min(n, mu + 12 * sd + 20))


@pytest.mark.parametrize('lam', POISSON)
def test_oracle_poisson_distribution(lam):
    k, margin = obc.poisson_counts(lam, 20261022, np.arange(N_DRAWS), cycle=3)
    assert not np.any(np.isnan(k))
    lo, hi = poisson_window(lam)
    assert chi2_pvalue(k, lambda x: stats.poisson.pmf(x, lam), lo, hi) >= 1e-6


@pytest.mark.parametrize('n,p', BINOMIAL)
def test_oracle_binomial_distribution(n, p):
    k, margin = obc.binomial_counts(n, p, 20261022, np.arange(N_DRAWS), cycle=3)
    assert not np.any(np.isnan(k))
    assert np.all((k >= 0) & (k <= n))
    lo, hi = binomial_window(n, p)
    assert chi2_pvalue(k, lambda x: stats.binom.pmf(x, n, p), lo, hi) >= 1e-6


def test_arms_cover_both_sides_of_each_switch():
    assert any(lam < obc.MEAN_SWITCH for lam in POISSON) and any(lam >= obc.MEAN_SWITCH for lam in POISSON)
    means = [n * min(p, 1 - p) for n, p in BINOMIAL]
    assert any(m < obc.MEAN_SWITCH for m in means) and any(m >= obc.MEAN_SWITCH for m in means)
    assert any(p > 0.5 and n * (1 - p) < obc.MEAN_SWITCH for n, p in BINOMIAL)     # inversion with symmetry
    assert any(p > 0.5 and n * (1 - p) >= obc.MEAN_SWITCH for n, p in BINOMIAL)    # rejection with symmetry


def test_point_masses():
    inst = np.arange(10000)
    assert np.all(obc.poisson_counts(0.0, 5, inst, 0)[0] == 0)
    assert np.all(obc.binomial_counts(37, 0.0, 5, inst, 0)[0] == 0)
    assert np.all(obc.binomial_counts(37, 1.0, 5, inst, 0)[0] == 37)
    assert np.all(obc.binomial_counts(10 ** 6, 1.0, 5, inst, 0)[0] == 10 ** 6)
    assert np.all(obc.binomial_counts(0, 0.4, 5, inst, 0)[0] == 0)


@pytest.mark.parametrize('lam', [-1e-300, -1.0, np.nan, np.inf, -np.inf])
def test_invalid_poisson_mean_gives_nan(lam):
    assert np.all(np.isnan(obc.poisson_counts(lam, 5, np.arange(8), 0)[0]))


@pytest.mark.parametrize('n,p', [(10, -0.1), (10, 1.0 + 1e-15), (10, np.nan), (-1, 0.5), (10.5, 0.5),
                                 (np.nan, 0.5), (np.inf, 0.5), (2.0 ** 31 + 1, 0.5)])
def test_invalid_binomial_gives_nan(n, p):
    assert np.all(np.isnan(obc.binomial_counts(n, p, 5, np.arange(8), 0)[0]))


def test_margins_are_reported():
    """Inversion draws report the distance of u from the CDF, rejection draws the acceptance test's distance."""
    k, m = obc.poisson_counts(3.0, 5, np.arange(1000), 0)
    assert np.all(np.isfinite(m)) and np.all(m >= 0)
    k, m = obc.binomial_counts(10 ** 6, 0.4, 5, np.arange(20000), 0)
    assert np.any(np.isfinite(m)) and np.any(np.isinf(m))          # box acceptances take no transcendental test
    assert np.mean(m < 1e-12) <= 1e-3


def _counter_words(path, name):
    text = Path(path).read_text()
    return int(re.search(rf'#define {name} (0x[0-9A-Fa-f]+)u', text).group(1), 16)


def test_count_stream_is_its_own():
    """The third counter word of the count sampler (0x60000000 | channel, key = simulator seed) differs from every
    other stream's: the Liu-West jitter's and the Gaussian simulator's call word (< 2), the packed normals'
    (0x80000000 | D), the drift's and the truth walk's (0x40000000 | c, 0x50000000 | c); the batch uniforms put their
    tag 0x0B5E0001 in the fourth word, where the sampler has its attempt (< 64)."""
    csrc = Path(__file__).resolve().parent.parent / 'optbayesexpt_b200' / 'csrc' / 'obe_device.cuh'
    assert _counter_words(csrc, 'OBE_COUNT_CTR') == obc.COUNT_CTR
    count = {obc.COUNT_CTR | c for c in range(4)}
    taken = set(range(2)) | {0x80000000 | d for d in range(1, 9)}
    taken |= {_counter_words(csrc, 'OBE_DRIFT_CTR') | c for c in range(2)}
    taken |= {_counter_words(csrc, 'OBE_TRUTH_CTR') | c for c in range(2)}
    assert not (count & taken)
    assert obc.COUNT_TRIES < 0x0B5E0001
    # and the uniforms themselves differ from the batch uniforms of the same seed and instance
    from oracle.obe_oracle import batch_uniform
    u, v = obc.count_uniforms(77, np.arange(64), 0, 0, 0)
    assert not np.any(np.isin(u, batch_uniform(77, 0, 0, np.arange(64))))


def test_count_record_checks():
    B = 3
    y, a = count_record('poisson', [[0.0], [3.0], [17.0]], None, B, 1)
    assert y.shape == (3, 1) and np.all(a == 0)
    for bad in ([[1.5], [0.0], [1.0]], [[-1.0], [0.0], [1.0]], [[np.nan], [0.0], [1.0]], [[np.inf], [0.0], [1.0]]):
        with pytest.raises(ValueError):
            count_record('poisson', bad, None, B, 1)
    y, a = count_record('binomial', [0.0, 5.0, 100.0], 100, B, 1)
    assert np.all(a == 100)
    y, a = count_record('binomial', [0.0, 5.0, 7.0], [1.0, 10.0, 7.0], B, 1)
    assert np.all(a[:, 0] == [1.0, 10.0, 7.0])
    for k, n in (([0.0, 5.0, 101.0], 100), ([0.0, 0.5, 1.0], 10), ([0.0, -1.0, 1.0], 10), ([0.0, np.nan, 1.0], 10),
                 ([0.0, 1.0, 1.0], 10.5), ([0.0, 1.0, 1.0], None)):
        with pytest.raises(ValueError):
            count_record('binomial', k, n, B, 1)
    with pytest.raises(ValueError):
        count_record(object(), [0.0, 1.0, 2.0], None, B, 1)          # a cuda_likelihood record needs its aux


def test_simulator_arguments():
    assert simulator_noise('gaussian', 2.0, None) == 2.0
    assert simulator_noise('poisson', None, None) == 0.0
    assert np.all(simulator_noise('binomial', None, [10, 20]) == [10, 20])
    for args in (('gaussian', None, None), ('poisson', 1.0, None), ('poisson', None, 10), ('binomial', None, None),
                 ('binomial', 1.0, 10), ('binomial', None, 10.5), ('binomial', None, -1), ('binomial', None, np.nan),
                 ('binomial', None, 2.0 ** 31 + 1), (object(), None, None)):
        with pytest.raises(ValueError):
            simulator_noise(*args)


def _prior(B=2, d=3, n=100):
    return np.random.default_rng(0).uniform(1.0, 2.0, size=(B, d, n))


def test_constructor_refusals():
    from optbayesexpt_b200.models import builtin
    for model in ('line', builtin('line').with_likelihood('poisson')):
        with pytest.raises(ValueError, match='n_instances, n_dims, n_particles'):      # one cloud, not a batch
            BatchedOptBayesExpt(model, (np.linspace(0, 1, 5),), _prior()[0, :2], ())
    with pytest.raises(ValueError, match='noise parameter is the sigma of the Gaussian'):
        BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 5),), _prior(d=4), (), likelihood_model='poisson',
                            noise_parameter_index=3)
    with pytest.raises(ValueError, match='integer'):
        BatchedOptBayesExpt('lorentzian_dip', (np.linspace(0, 1, 5),), _prior(d=4), (), likelihood_model='binomial',
                            design_noise='likelihood', design_aux=10.5)
    with pytest.raises(ValueError, match='design_noise'):
        BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 5),), _prior(d=4), (), likelihood_model='poisson',
                            design_noise='bogus')
    with pytest.raises(ValueError, match='design_aux'):
        BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 5),), _prior(d=4), (), likelihood_model='poisson',
                            design_noise='likelihood', design_aux=-1.0)
    with pytest.raises(ValueError, match='unknown likelihood_model'):
        BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 5),), _prior(d=4), (), likelihood_model='cauchy')


def test_count_record_feeds_the_likelihood_oracles():
    """The batched record's per-record constants are the log-factorial terms of oracle/likelihoods.py's pmfs."""
    from scipy.special import gammaln

    from oracle.likelihoods import loglik_binomial, loglik_poisson
    k, a, lc = obc.count_record([4.0], None, 'poisson')
    lam = np.array([0.5, 3.0, 8.0])
    assert np.allclose(loglik_poisson([lam], k), k[0] * np.log(lam) - lam - lc[0], rtol=1e-14)
    k, a, lc = obc.count_record([4.0], [30.0], 'binomial')
    p = np.array([0.1, 0.5])
    assert np.allclose(loglik_binomial([p], k, a), lc[0] + 4 * np.log(p) + 26 * np.log1p(-p), rtol=1e-14)
    assert lc[0] == (gammaln(31.0) - gammaln(5.0)) - gammaln(27.0)
