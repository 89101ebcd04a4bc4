"""CPU oracle for the non-Gaussian measurement likelihoods  --  TEST INFRASTRUCTURE, NOT PRODUCT.

The Poisson and binomial likelihoods of the update kernel (``likelihood_model='poisson' | 'binomial'``) and of a
user ``cuda_likelihood``, written with ``scipy.special`` (``xlogy``, ``xlog1py``, ``gammaln``) in the same order as
the kernel, and :class:`OracleOBELik`, the orchestration of :class:`~oracle.obe_oracle.OracleOBE` with one of them,
so that closed-loop trajectories can be replayed.
"""
import numpy as np

from .obe_oracle import OracleOBE, normalized_product, resample_decision


def from_log(ll, choke=None, nonpos=True):
    """exp(choke * log L) in the order of the update kernel: a pmf's log is clamped to <= 0 first (rounding-level
    positive sums), and NaN (an invalid model output) gives weight 0, as nan_to_num of scipy's nan does."""
    ll = np.asarray(ll, dtype=np.float64)
    with np.errstate(invalid='ignore'):
        if nonpos:
            ll = np.where(ll > 0.0, 0.0, ll)
        if choke is not None:
            ll = ll * choke
        return np.where(np.isnan(ll), 0.0, np.exp(ll))


def loglik_poisson(y_model, counts):
    """sum_c xlogy(k_c, lam_c) - lam_c - gammaln(k_c + 1) (scipy.stats.poisson.logpmf), zip-truncated like the
    Gaussian likelihood; lam < 0, NaN or +inf give NaN."""
    from scipy.special import gammaln, xlogy
    ll = 0.0
    for lam, k in zip(y_model, np.atleast_1d(counts)):
        lam = np.asarray(lam, dtype=np.float64)
        with np.errstate(all='ignore'):
            lc = (xlogy(k, lam) - lam) - gammaln(k + 1.0)
            ll = ll + np.where(lam >= 0.0, lc, np.nan)
    return ll


def loglik_binomial(y_model, k_succ, n_trials):
    """sum_c gammaln(n+1) - gammaln(k+1) - gammaln(n-k+1) + xlogy(k, p) + xlog1py(n-k, -p)
    (scipy.stats.binom.logpmf); p outside [0, 1] gives NaN."""
    from scipy.special import gammaln, xlog1py, xlogy
    ll = 0.0
    for p, k, n in zip(y_model, np.atleast_1d(k_succ), np.atleast_1d(n_trials)):
        p = np.asarray(p, dtype=np.float64)
        lconst = (gammaln(n + 1.0) - gammaln(k + 1.0)) - gammaln(n - k + 1.0)
        with np.errstate(all='ignore'):
            lc = (lconst + xlogy(k, p)) + xlog1py(n - k, -p)
            ll = ll + np.where((p >= 0.0) & (p <= 1.0), lc, np.nan)
    return ll


def likelihood_poisson(y_model, counts, choke=None):
    """Poisson pmf of the counts given the expected counts y_model, per particle."""
    return from_log(loglik_poisson(y_model, counts), choke)


def likelihood_binomial(y_model, k_succ, n_trials, choke=None):
    """Binomial pmf of k successes in n trials given the success probabilities y_model, per particle."""
    return from_log(loglik_binomial(y_model, k_succ, n_trials), choke)


class OracleOBELik(OracleOBE):
    """OracleOBE with ``likelihood_model``: 'gaussian', 'poisson', 'binomial', or a callable
    (y_model, y_meas, aux) -> log L (the restatement of a cuda_likelihood)."""

    def __init__(self, *args, likelihood_model='gaussian', **kwargs):
        OracleOBE.__init__(self, *args, **kwargs)
        self.likelihood_model = likelihood_model

    def likelihood(self, y_model, record):
        if self.likelihood_model == 'poisson':
            return likelihood_poisson(y_model, record[1], self.choke)
        if self.likelihood_model == 'binomial':
            return likelihood_binomial(y_model, record[1], record[2], self.choke)
        return from_log(self.likelihood_model(y_model, record[1], record[2]), self.choke, nonpos=False)

    def pdf_update(self, record, forced_resample=False):
        if self.likelihood_model == 'gaussian':
            return OracleOBE.pdf_update(self, record, forced_resample)
        y_model = self.eval_over_all_parameters(record[0])
        self.particle_weights = normalized_product(self.particle_weights, self.likelihood(y_model, record))
        self.just_resampled = False
        if self.tuning_parameters['auto_resample'] or forced_resample:
            do, _ = resample_decision(self.particle_weights, self.tuning_parameters['resample_threshold'])
            if do or forced_resample:
                self.resample()
                self.just_resampled = True
        if self.just_resampled:
            self.enforce_parameter_constraints()
        return self.particles, self.particle_weights
