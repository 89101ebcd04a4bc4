"""CPU oracle for the information gain of a user count pmf  --  TEST INFRASTRUCTURE, NOT PRODUCT.

``cuda_likelihood(source, entry, noise_var=, window=)`` declares the integer count range of one measurement, and with
it that ``entry`` is a normalised log-pmf.  ``OptBayesExpt(..., utility_method='information_gain')`` then ranks
settings by the same mutual information as for the built-in likelihoods (see :mod:`oracle.information_gain`),

    I(s) = (1/K) sum_k sum_y p_k(y) log(p_k(y) / pbar(y)),   pbar = (1/K) sum_j p_j,

summed over the union of the K draws' declared windows.  :func:`information_gain_user` restates the kernel's formula
in numpy, and :class:`OracleOBEInfoUser` is :class:`~oracle.information_gain.OracleOBEInfo` selecting with it, so that
closed-loop trajectories can be replayed.

There is no analytic reference draw: at each count y, with l_k = log p(y | x_k), M = max_k l_k,
L = log1p(mean_k expm1(l_k - M)), d_k = l_k - M - L = log(p_k / pbar), and the term is exp(M + L) sum_k phi(d_k),
every term non-negative (phi as in :mod:`oracle.information_gain`).  A y that no draw reaches contributes 0.
"""
import numpy as np

from .information_gain import OracleOBEInfo, phi, union_counts
from .obe_oracle import lockin_cost, randdraw, yvar_from_draws

#: the largest union of windows a user pmf's setting may sum over; a larger one gives the setting 0
USER_MAX_COUNTS = 2 ** 20


def _windows_ok(lo, hi):
    with np.errstate(invalid='ignore'):
        return (lo >= 0.0) & (lo <= hi) & (hi <= 2.0 ** 53) & (lo == np.floor(lo)) & (hi == np.floor(hi))


def _one_setting(logpmf, x, aux, lo, hi):
    """I of one setting of a user pmf (windows valid, outputs not all equal), or None when it is invalid."""
    y = union_counts(lo, hi)
    if y.size > USER_MAX_COUNTS:
        return None
    ell = np.asarray(logpmf(x[:, None], y[None, :], aux), dtype=np.float64)
    ell = np.broadcast_to(ell, (len(x), y.size))
    if np.any(np.isnan(ell) | (ell == np.inf)):
        return None
    M = np.max(ell, axis=0)
    live = M > -np.inf                                   # (a count no draw reaches contributes 0)
    ell, M = ell[:, live], M[live]
    K = len(x)
    L = np.log1p(np.sum(np.expm1(ell - M), axis=0) / K)
    d = (ell - M) - L
    return float(np.sum(np.exp(np.minimum(M + L, 0.0)) * np.sum(phi(d), axis=0)) / K)


def information_gain_user(logpmf, window, outputs, aux, noise_var=None, cost=1.0):
    """(S,) information gain in nats of a user count pmf, the twin of the kernel of ``cuda_likelihood(...,
    window=)``: ``logpmf(x, y, aux)`` = log p(y | x, aux) (broadcasting), ``window(x, aux)`` -> (lo, hi) per output,
    ``noise_var(x, aux)`` (optional) the declared variance.  ``outputs`` (K, S) or (K, 1, S) are the draws' model
    outputs.  Divided by ``cost``; exactly 0 where a variance is negative or NaN, a window has NaN / non-integer
    bounds, lo < 0, lo > hi or hi > 2^53, some l_k is NaN or +inf, the union exceeds :data:`USER_MAX_COUNTS`, or all
    K outputs are equal."""
    y_space = np.asarray(outputs, dtype=np.float64)
    if y_space.ndim == 3:
        if y_space.shape[1] != 1:
            raise ValueError('information gain: single-channel outputs only')
        y_space = y_space[:, 0, :]
    K, S = y_space.shape
    aux = float(np.asarray(aux, dtype=np.float64).reshape(-1)[0])
    out = np.zeros(S)
    ok = np.ones(S, dtype=bool)
    for s in range(S):
        x = y_space[:, s]
        if noise_var is not None:
            with np.errstate(invalid='ignore'):
                if not np.all(np.asarray(noise_var(x, aux)) >= 0.0):
                    ok[s] = False
                    continue
        lo, hi = (np.broadcast_to(np.asarray(v, dtype=np.float64), x.shape) for v in window(x, aux))
        if not np.all(_windows_ok(lo, hi)):
            ok[s] = False
            continue
        if np.all(x == x[0]):
            continue
        v = _one_setting(logpmf, x, aux, lo, hi)
        if v is None:
            ok[s] = False
        else:
            out[s] = v
    cost = np.broadcast_to(np.asarray(cost, dtype=np.float64), (S,))
    with np.errstate(invalid='ignore', divide='ignore'):
        u = out / cost
    return np.where(ok, u, 0.0)


class OracleOBEInfoUser(OracleOBEInfo):
    """OracleOBEInfo for a user likelihood (``likelihood_model`` a callable (y_model, y_meas, aux) -> log L, as in
    OracleOBELik): selects with :func:`information_gain_user` over ``logpmf(x, y, aux)`` (default:
    ``likelihood_model((x,), y, aux)``, the one-channel outputs with y in place of the record's count), ``window`` and
    ``noise_var``; aux = ``design_aux`` (default 1)."""

    def __init__(self, *args, window=None, logpmf=None, **kwargs):
        OracleOBEInfo.__init__(self, *args, **kwargs)
        self.window = window
        self.logpmf = logpmf if logpmf is not None else (lambda x, y, aux: self.likelihood_model((x,), y, aux))

    def utility(self):
        if self.method != 'information_gain':
            return OracleOBEInfo.utility(self)
        draws, _ = randdraw(self.particles, self.particle_weights, self.rng.random(self.N_DRAWS))
        _, y_space = yvar_from_draws(self.model, self.allsettings, draws, self.cons, self.n_channels)
        cost = 1.0
        if self.cost_of_changing_setting is not None:
            cost = lockin_cost(self.allsettings.shape[1], self.last_setting_index, self.cost_of_changing_setting)
        aux = 1.0 if self.design_aux is None else self.design_aux
        self.last_utility = information_gain_user(self.logpmf, self.window, y_space, aux, noise_var=self.noise_var,
                                                  cost=cost)
        return self.last_utility
