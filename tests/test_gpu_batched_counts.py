"""GPU tests of the batched engines' count likelihoods: the device count sampler against its restatement
(oracle/batched_counts.py) and against scipy's distributions, instance b of a batched Poisson / binomial / user-likelihood
engine against a single OptBayesExpt fed the same counts and uniforms, closed loops on the device with the count
simulators (with and without drift), the isolation of an instance with invalid counts, and the refusals."""
import warnings

import numpy as np
import pytest
import torch

from oracle import batched_counts as obc
from oracle import obe_oracle as orc

from test_batched_counts_host import BINOMIAL, POISSON, binomial_window, chi2_pvalue, poisson_window

pytestmark = pytest.mark.gpu

SEED = 987654321
B_SIM = 4096


def _sim_engine(likelihood):
    """A batched engine on `line` (m x + b) whose simulator, at truth (0, value), draws with mean / probability
    `value` exactly."""
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    prior = np.random.default_rng(0).uniform(0.0, 1.0, size=(B_SIM, 2, 64))
    return BatchedOptBayesExpt('line', (np.array([1.0]),), prior, (), likelihood_model=likelihood, seed=1)


def _device_draws(beng, cycles):
    out = np.empty((cycles, B_SIM))
    third = np.empty((cycles, B_SIM))
    for t in range(cycles):
        beng.cycle = t
        rec = beng.simulate_measurement().cpu().numpy()
        out[t], third[t] = rec[:, 4], rec[:, 8]
    return out, third


def _compare_with_oracle(dev, oracle_fn):
    n_bad = n_all = 0
    for t in range(dev.shape[0]):
        k, margin = oracle_fn(t)
        differ = ~((dev[t] == k) | (np.isnan(dev[t]) & np.isnan(k)))
        assert np.all(margin[differ] < 1e-12), f'cycle {t}: counts differ at decisive margins {margin[differ]}'
        n_bad += int(np.sum(margin < 1e-12))
        n_all += k.size
    assert n_bad <= 1e-6 * n_all


@pytest.mark.parametrize('lam', POISSON)
def test_device_poisson_sampler(lam):
    from scipy import stats
    beng = _sim_engine('poisson')
    beng.set_simulator(np.array([0.0, lam]), seed=SEED)
    cycles = -(-1_000_000 // B_SIM)
    dev, third = _device_draws(beng, cycles)
    inst = np.arange(B_SIM)
    _compare_with_oracle(dev[:20], lambda t: obc.poisson_counts(lam, SEED, inst, t))
    lo, hi = poisson_window(lam)
    assert chi2_pvalue(dev.reshape(-1), lambda x: stats.poisson.pmf(x, lam), lo, hi) >= 1e-6


@pytest.mark.parametrize('n,p', BINOMIAL)
def test_device_binomial_sampler(n, p):
    from scipy import stats
    beng = _sim_engine('binomial')
    beng.set_simulator(np.array([0.0, p]), trials=n, seed=SEED)
    cycles = -(-1_000_000 // B_SIM)
    dev, third = _device_draws(beng, cycles)
    assert np.all(third == n), 'the trials are the record\'s third element'
    inst = np.arange(B_SIM)
    _compare_with_oracle(dev[:20], lambda t: obc.binomial_counts(n, p, SEED, inst, t))
    lo, hi = binomial_window(n, p)
    assert chi2_pvalue(dev.reshape(-1), lambda x: stats.binom.pmf(x, n, p), lo, hi) >= 1e-6


def test_device_sampler_invalid_and_per_instance_trials():
    beng = _sim_engine('binomial')
    trials = np.arange(B_SIM, dtype=np.float64) % 50
    beng.set_simulator(np.array([0.0, 0.3]), trials=trials, seed=SEED)
    dev, third = _device_draws(beng, 3)
    assert np.all(third == trials)
    for t in range(3):
        k, _ = obc.binomial_counts(trials, 0.3, SEED, np.arange(B_SIM), t)
        assert np.array_equal(dev[t], k)
    beng.set_simulator(np.array([0.0, 1.5]), trials=10, seed=SEED)        # p > 1
    assert np.all(np.isnan(_device_draws(beng, 1)[0]))
    beng = _sim_engine('poisson')
    beng.set_simulator(np.array([0.0, -0.5]), seed=SEED)                 # lambda < 0
    assert np.all(np.isnan(_device_draws(beng, 1)[0]))
    beng.set_simulator(np.array([0.0, 0.0]), seed=SEED)                  # lambda = 0
    assert np.all(_device_draws(beng, 2)[0] == 0)


# ---- instance b against a single engine fed the same counts and uniforms ------------------------------------------
USER_POISSON = r'''
__device__ double upois(const double* y, const double* ym, const double* aux, int n) {
    double ll = 0.0;
    for (int c = 0; c < n; ++c) {
        const double lam = y[c], k = ym[c];
        if (!(lam >= 0.0)) return __longlong_as_double(0x7ff8000000000000ll);
        ll += ((k == 0.0 ? 0.0 : k * log(lam)) - lam) - lgamma(k + 1.0);
    }
    return ll;
}
__device__ double upois_var(double y, double a) { return y; }
'''


def _run_pair(B, n, cycles, model, cons, settings, prior_fn, truths, counts_fn, single_kwargs, batched_kwargs,
              aux=None):
    """test_gpu_batched.py's pairing harness for count records: every chosen setting and resample decision
    identical, means / N_eff / weights to 1e-9."""
    import optbayesexpt_b200 as obe
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    priors = np.stack([prior_fn(np.random.default_rng(100 + b), n) for b in range(B)])
    beng = BatchedOptBayesExpt(model, (settings,), priors, cons, n_draws=30, scale=False, seed=4321, **batched_kwargs)
    singles = []
    for b in range(B):
        e = obe.OptBayesExpt(model, (settings,), priors[b], cons, scale=False, n_draws=30, **single_kwargs)
        e.rng = orc.ReplayRng(4321, b, 30)
        e._philox_seed = beng._seed_normal + b
        e._epoch = 0
        singles.append(e)
    rng = np.random.default_rng(7)
    n_res = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(cycles):
            idx, sets = beng.opt_setting()
            for b, e in enumerate(singles):
                e.opt_setting()
                assert e.last_setting_index == idx[b], f'cycle {t} instance {b}: setting index differs'
            ys = counts_fn(sets[0], truths, rng)
            beng.pdf_update(ys, aux)
            flags = beng.just_resampled
            means, neff = beng.mean(), beng.n_eff()
            for b, e in enumerate(singles):
                rec = (float(sets[0, b]), float(ys[b]))
                if aux is not None:
                    rec = rec + (float(aux),)
                e.pdf_update(rec)
                assert bool(e.just_resampled) == bool(flags[b]), f'cycle {t} instance {b}: resample decision differs'
                np.testing.assert_allclose(means[b], e.mean(), rtol=1e-9, err_msg=f'mean {t} {b}')
                np.testing.assert_allclose(neff[b], e.n_eff(), rtol=1e-9)
                e.rng.next_cycle()
            n_res += int(flags.sum())
    assert n_res > 0, 'no resample fired'
    for b, e in enumerate(singles):
        w = e.particle_weights
        np.testing.assert_allclose(beng.particle_weights(b), w, rtol=1e-9, atol=1e-15 * w.max())


PEAK_SETTINGS = np.linspace(1.5, 4.5, 241)


def _peak_prior(g, n):
    return np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(2.0, 20.0, n)])


def _dip_prior(g, n):
    return np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 0.8, n), g.uniform(0.2, 0.6, n)])


def _peak_truths(B):
    return [(3.1 + 0.1 * b, 40.0, 10.0) for b in range(B)]


def _poisson_counts(x, truths, rng):
    return np.array([rng.poisson(orc.model_lorentzian_hwhm((x[b],), truths[b], (0.3,))) for b in range(len(truths))],
                    dtype=np.float64)


@pytest.mark.parametrize('mode', ['fixed', 'likelihood'])
def test_batched_poisson_matches_single_engines(mode):
    _run_pair(4, 5000, 30, 'lorentzian_hwhm', (0.3,), PEAK_SETTINGS, _peak_prior, _peak_truths(4), _poisson_counts,
              dict(likelihood_model='poisson', design_noise=mode, default_noise_std=5.0),
              dict(likelihood_model='poisson', design_noise=mode, default_noise_std=5.0))


def test_batched_binomial_matches_single_engines():
    truths = [(3.0 + 0.1 * b, 0.5, 0.4) for b in range(4)]

    def counts(x, tr, rng):
        return np.array([rng.binomial(100, orc.model_lorentzian_dip((x[b],), tr[b], ())) for b in range(len(tr))],
                        dtype=np.float64)
    kw = dict(likelihood_model='binomial', design_noise='likelihood', design_aux=100)
    _run_pair(4, 5000, 30, 'lorentzian_dip', (), PEAK_SETTINGS, _dip_prior, truths, counts, kw, kw, aux=100.0)


def test_batched_user_likelihood_matches_single_engines():
    import optbayesexpt_b200 as obe
    lik = obe.cuda_likelihood(USER_POISSON, 'upois', noise_var='upois_var')
    kw = dict(likelihood_model=lik, design_noise='likelihood', design_aux=1.0)
    _run_pair(4, 5000, 30, 'lorentzian_hwhm', (0.3,), PEAK_SETTINGS, _peak_prior, _peak_truths(4), _poisson_counts,
              kw, kw, aux=1.0)


# ---- closed loops on the device -----------------------------------------------------------------------------------
def _coverage(beng, truths):
    err = np.abs(beng.mean() - truths) / beng.std()
    return np.mean(err < 4.0, axis=0)


def _closed_loop(beng, cycles):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        torch.cuda.set_sync_debug_mode('error')          # a host synchronisation inside the loop raises
        try:
            for _ in range(cycles):
                beng.closed_loop_cycle()
        finally:
            torch.cuda.set_sync_debug_mode('default')


@pytest.mark.parametrize('drift', [False, True])
def test_poisson_closed_loop_on_device(drift):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B, n = 512, 10000
    g = np.random.default_rng(3)
    prior = np.stack([_peak_prior(g, n) for _ in range(B)])
    truths = np.stack([g.uniform(2.8, 3.4, B), np.full(B, 40.0), np.full(B, 10.0)], axis=1)
    step = [0.002, 0.0, 0.0] if drift else None
    beng = BatchedOptBayesExpt('lorentzian_hwhm', (PEAK_SETTINGS,), prior, (0.3,), likelihood_model='poisson',
                               design_noise='likelihood', seed=11, drift=step)
    beng.set_simulator(truths, seed=12, drift=step)
    _closed_loop(beng, 150)
    cov = _coverage(beng, beng.simulator_truth())
    assert np.all(cov >= 0.95), cov


@pytest.mark.parametrize('drift', [False, True])
def test_binomial_closed_loop_on_device(drift):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B, n = 512, 10000
    g = np.random.default_rng(4)
    prior = np.stack([_dip_prior(g, n) for _ in range(B)])
    truths = np.stack([g.uniform(2.8, 3.4, B), np.full(B, 0.5), np.full(B, 0.4)], axis=1)
    trials = g.integers(50, 201, B).astype(np.float64)
    step = [0.002, 0.0, 0.0] if drift else None
    beng = BatchedOptBayesExpt('lorentzian_dip', (PEAK_SETTINGS,), prior, (), likelihood_model='binomial',
                               design_noise='likelihood', design_aux=100, seed=13, drift=step)
    beng.set_simulator(truths, trials=trials, seed=14, drift=step)
    _closed_loop(beng, 150)
    rec = beng._record.cpu().numpy()
    assert np.array_equal(rec[:, 8], trials)
    cov = _coverage(beng, beng.simulator_truth())
    assert np.all(cov >= 0.95), cov


def test_bad_instance_is_isolated():
    """An instance whose truth gives lambda < 0 gets NaN counts; every other instance is bit for bit what it is
    without it."""
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B, n = 8, 5000
    g = np.random.default_rng(5)
    prior = np.stack([_peak_prior(g, n) for _ in range(B)])
    good = np.stack([g.uniform(2.8, 3.4, B), np.full(B, 40.0), np.full(B, 10.0)], axis=1)
    bad = good.copy()
    bad[3] = (3.0, 1.0, -5.0)                             # lambda in (-5, -4] at every setting
    runs = []
    for truths in (good, bad):
        beng = BatchedOptBayesExpt('lorentzian_hwhm', (PEAK_SETTINGS,), prior, (0.3,), likelihood_model='poisson',
                                   design_noise='likelihood', seed=21)
        beng.set_simulator(truths, seed=22)
        idx, rec = [], []
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', RuntimeWarning)
            for _ in range(40):
                beng.closed_loop_cycle()
                idx.append(beng.last_setting_index)
                rec.append(beng._record.cpu().numpy().copy())
        runs.append((np.array(idx), np.array(rec), beng.mean(), beng.std(), beng.n_eff(),
                     [beng.particle_weights(b) for b in range(B)]))
    (i0, r0, m0, s0, n0, w0), (i1, r1, m1, s1, n1, w1) = runs
    keep = np.arange(B) != 3
    assert np.all(np.isnan(r1[:, 3, 4]))
    assert np.array_equal(i0[:, keep], i1[:, keep])
    assert np.array_equal(r0[:, keep], r1[:, keep])
    for a, b in ((m0, m1), (s0, s1), (n0, n1)):
        assert np.array_equal(a[keep], b[keep])
    for b in np.flatnonzero(keep):
        assert np.array_equal(w0[b], w1[b])


def test_refusals_before_the_device():
    import optbayesexpt_b200 as obe
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B, n = 4, 1000
    g = np.random.default_rng(6)
    prior = np.stack([_peak_prior(g, n) for _ in range(B)])
    prior4 = np.concatenate([prior, np.ones((B, 1, n))], axis=1)
    with pytest.raises(ValueError, match='noise parameter'):
        BatchedOptBayesExpt('lorentzian_hwhm', (PEAK_SETTINGS,), prior4, (0.3,), likelihood_model='poisson',
                            noise_parameter_index=3)
    with pytest.raises(ValueError, match='integer'):
        BatchedOptBayesExpt('lorentzian_dip', (PEAK_SETTINGS,), prior, (), likelihood_model='binomial',
                            design_noise='likelihood', design_aux=99.5)
    lik = obe.cuda_likelihood(USER_POISSON, 'upois', noise_var='upois_var')
    user = BatchedOptBayesExpt('lorentzian_hwhm', (PEAK_SETTINGS,), prior, (0.3,), likelihood_model=lik)
    with pytest.raises(ValueError, match='no sampler'):
        user.set_simulator(_peak_truths(B))
    binom = BatchedOptBayesExpt('lorentzian_dip', (PEAK_SETTINGS,), prior, (), likelihood_model='binomial',
                                design_noise='likelihood', design_aux=100)
    with pytest.raises(ValueError, match='trials'):
        binom.set_simulator([(3.0, 0.5, 0.4)] * B)
    with pytest.raises(ValueError, match='integer'):
        binom.design_aux = 12.5
    pois = BatchedOptBayesExpt('lorentzian_hwhm', (PEAK_SETTINGS,), prior, (0.3,), likelihood_model='poisson')
    with pytest.raises(ValueError, match='noise_level'):
        pois.set_simulator(_peak_truths(B), 5.0)
    w_before = pois.particle_weights(0)
    for bad in ([1.0, 2.5, 3.0, 4.0], [1.0, -1.0, 3.0, 4.0], [1.0, np.nan, 3.0, 4.0]):
        with pytest.raises(ValueError):
            pois.pdf_update(bad)
    with pytest.raises(ValueError):
        binom.pdf_update([1.0, 2.0, 101.0, 4.0], 100)
    assert pois.cycle == 0 and binom.cycle == 0
    assert np.array_equal(pois.particle_weights(0), w_before)
