"""CPU oracle for the likelihood-aware utility  --  TEST INFRASTRUCTURE, NOT PRODUCT.

``OptBayesExpt(..., design_noise='likelihood')`` divides the spread of the drawn model curves at each setting by the
likelihood's own noise variance, averaged over the draws.  :func:`noise_var_from_draws` and
:func:`utility_likelihood_noise` restate that utility in numpy in the kernel's order, and :class:`OracleOBEDesign`
is :class:`~oracle.likelihoods.OracleOBELik` selecting with it, so that closed-loop trajectories can be replayed.
"""
import numpy as np

from .likelihoods import OracleOBELik
from .obe_oracle import OracleOBE, lockin_cost, randdraw, yvar_from_draws


def noise_nu(y, kind, aux):
    """(nu, valid) of model outputs y for one channel with aux a: Poisson nu = y (valid: 0 <= y < inf), binomial
    nu = y (1 - y) (valid: 0 <= p <= 1), a callable kind(y, a) (a cuda_likelihood's noise_var; valid: nu >= 0)."""
    y = np.asarray(y, dtype=np.float64)
    with np.errstate(all='ignore'):
        if kind == 'poisson':
            return y, (y >= 0.0) & (y <= np.finfo(np.float64).max)
        if kind == 'binomial':
            return y * (1.0 - y), (y >= 0.0) & (y <= 1.0)
        nu = np.asarray(kind(y, aux), dtype=np.float64)
        return nu, nu >= 0.0


def _aux_column(aux, n_channels):
    return np.broadcast_to(np.asarray(1.0 if aux is None else aux, dtype=np.float64).reshape(-1),
                           (n_channels,)).reshape(n_channels, 1)


def noise_var_from_draws(y_space, kind, aux=None):
    """(C, S) noise variance of the likelihood averaged over the K draws of y_space (K, C, S):
    np.mean(nu(y_space), axis=0), then / aux for binomial.  numpy reduces axis 0 sequentially over k, the
    association of np.var's own mean and of the kernel."""
    y_space = np.asarray(y_space, dtype=np.float64)
    a = _aux_column(aux, y_space.shape[1])
    nu, _ = noise_nu(y_space, kind, a[None])
    v = np.mean(nu, axis=0)
    if kind == 'binomial':
        v = v / a
    return v


def utility_likelihood_noise(y_space, kind, aux=None, method='variance', cost=1.0, log_form=False):
    """sum_c r_c / cost over settings, r_c = 0 where the spread is 0 and spread / v_c otherwise (+inf for v_c = 0),
    v_c = noise_var_from_draws; spread is np.var (variance), (max - min)^2 (max_min) or exp(2H)/(2 pi e) (pseudo).
    A setting where some draw's output is invalid for the likelihood gets exactly 0."""
    y_space = np.asarray(y_space, dtype=np.float64)
    a = _aux_column(aux, y_space.shape[1])
    v = noise_var_from_draws(y_space, kind, aux)
    with np.errstate(all='ignore'):
        if method == 'variance':
            spread = np.var(y_space, axis=0)
        elif method == 'max_min':
            spread = (np.max(y_space, axis=0) - np.min(y_space, axis=0)) ** 2
        elif method == 'pseudo':
            from scipy.stats import differential_entropy
            spread = np.exp(2 * differential_entropy(y_space, axis=0)) / (2 * np.pi * np.e)
        else:
            raise ValueError(f'unknown method {method!r}')
        r = np.where(spread == 0.0, 0.0, spread / v)
        terms = np.log(1 + r) if log_form else r
        u = np.sum(terms, axis=0) / cost
    _, ok = noise_nu(y_space, kind, a[None])
    return np.where(np.all(ok, axis=(0, 1)), u, 0.0)


class OracleOBEDesign(OracleOBELik):
    """OracleOBELik with ``design_noise``: 'fixed' selects as OracleOBELik does, 'likelihood' with
    :func:`utility_likelihood_noise` (aux = ``design_aux``).  ``noise_var`` (y, a) -> variance restates the noise_var
    of a cuda_likelihood when ``likelihood_model`` is a callable."""

    def __init__(self, *args, design_noise='fixed', design_aux=None, noise_var=None, **kwargs):
        OracleOBELik.__init__(self, *args, **kwargs)
        self.design_noise = design_noise
        self.design_aux = design_aux
        self.noise_var = noise_var

    def utility(self):
        if self.design_noise == 'fixed' or self.likelihood_model == 'gaussian':
            return OracleOBE.utility(self)
        draws, _ = randdraw(self.particles, self.particle_weights, self.rng.random(self.N_DRAWS))
        _, y_space = yvar_from_draws(self.model, self.allsettings, draws, self.cons, self.n_channels)
        cost = 1.0
        if self.cost_of_changing_setting is not None:
            cost = lockin_cost(self.allsettings.shape[1], self.last_setting_index, self.cost_of_changing_setting)
        kind = self.likelihood_model if isinstance(self.likelihood_model, str) else self.noise_var
        self.last_utility = utility_likelihood_noise(y_space, kind, self.design_aux, cost=cost)
        return self.last_utility
