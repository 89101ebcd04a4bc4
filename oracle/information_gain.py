"""CPU oracle for the information-gain utility  --  TEST INFRASTRUCTURE, NOT PRODUCT.

``OptBayesExpt(..., utility_method='information_gain')`` ranks settings by the mutual information between the
parameters, uniform over the K drawn sets, and the next count:

    I(s) = (1/K) sum_k sum_y p_k(y) log(p_k(y) / pbar(y)),   pbar = (1/K) sum_j p_j.

:func:`information_gain_from_draws` restates it in numpy / scipy over an explicit window of counts, independent
of the kernel's arithmetic, and :class:`OracleOBEInfo` is :class:`~oracle.design_noise.OracleOBEDesign` selecting
with it, so that closed-loop trajectories can be replayed.

Numerics (float64 reaches 1e-12 relative to a 50-digit evaluation in every regime):
- the log-pmfs are differences delta_k = log p_k - log p_r from a reference draw r (the median interior draw),
  written through log1p, so that large counts do not cancel; log p_r itself is :func:`logpmf`, the saddle-point form
  (checked against scipy.stats' logpmf in the tests);
- the mixture density pbar(y) = p_r(y) mean_k exp(delta_k) is formed with ``scipy.special.logsumexp``; the log ratios
  d_k = log(p_k / pbar) are formed as delta_k - M - log1p(mean_k expm1(delta_k - M)), M = max_k delta_k, the same
  number written so that it keeps its digits when the draws agree (logsumexp of values that all round to 0 loses
  them);
- I = (1/K) sum_y pbar(y) sum_k phi(d_k), phi(d) = d e^d - expm1(d) >= 0, its series below |d| = 1/2: every term is
  non-negative, so an I of 1e-12 is not the difference of two numbers of order 1.
"""
import numpy as np

from .design_noise import OracleOBEDesign
from .obe_oracle import lockin_cost, randdraw, yvar_from_draws

#: the half-width of a component's window is sqrt(79 var) + 27 counts: Bernstein's bound
#: exp(-t^2 / (2 (var + t/3))) then leaves less than 1e-17 of its mass outside
WINDOW_VAR, WINDOW_PAD = 79.0, 27.0


def valid_outputs(x, kind):
    """Poisson: 0 <= lambda < inf; binomial: 0 <= p <= 1 (NaN invalid)."""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(invalid='ignore'):
        if kind == 'poisson':
            return (x >= 0.0) & (x <= np.finfo(np.float64).max)
        if kind == 'binomial':
            return (x >= 0.0) & (x <= 1.0)
    raise ValueError(f'information gain: unknown likelihood {kind!r} (poisson or binomial)')


def windows(x, kind, n=None):
    """(lo, hi) integer count windows of the K components: mu -+ (sqrt(79 var) + 27), clipped to the support; a point
    mass (var = 0) is its own point."""
    x = np.asarray(x, dtype=np.float64)
    if kind == 'poisson':
        mu, var, top = x, x, np.inf
    else:
        mu = n * x
        var, top = mu * (1.0 - x), n
    t = np.where(var > 0.0, np.sqrt(WINDOW_VAR * var) + WINDOW_PAD, 0.0)
    return np.maximum(np.ceil(mu - t), 0.0), np.minimum(np.floor(mu + t), top)


def union_counts(lo, hi):
    """The integers of the union of the intervals [lo_k, hi_k], ascending."""
    order = np.argsort(lo, kind='stable')
    parts, clo, chi = [], lo[order[0]], hi[order[0]]
    for i in order[1:]:
        if lo[i] <= chi + 1.0:
            chi = max(chi, hi[i])
        else:
            parts.append(np.arange(clo, chi + 1.0))
            clo, chi = lo[i], hi[i]
    parts.append(np.arange(clo, chi + 1.0))
    return np.concatenate(parts)


def phi(d):
    """d e^d - expm1(d) = r log r - r + 1 at r = e^d (>= 0, 1 at d = -inf), its series on |d| < 1/2."""
    d = np.asarray(d, dtype=np.float64)
    out = np.ones_like(d)
    small = np.abs(d) < 0.5
    ds = d[small]
    # sum_{m >= 2} (m - 1) d^m / m!, through m = 16
    coef = [(m - 1) / float(np.prod(np.arange(1, m + 1, dtype=np.float64))) for m in range(16, 1, -1)]
    p = np.zeros_like(ds)
    for c in coef:
        p = p * ds + c
    out[small] = p * ds * ds
    big = ~small & np.isfinite(d)
    db = d[big]
    out[big] = db * np.exp(db) - np.expm1(db)
    return out


def _stirlerr(y):
    """log(y!) - [(y + 1/2) log y - y + log(2 pi)/2] for integers y >= 1 (Stirling's error, Loader 2000)."""
    from scipy.special import gammaln
    y = np.asarray(y, dtype=np.float64)
    small = y <= 15.0
    ys = np.where(small, y, 16.0)
    exact = gammaln(ys + 1.0) - (ys + 0.5) * np.log(ys) + ys - 0.5 * np.log(2.0 * np.pi)
    yb = np.where(small, 16.0, y)
    r2 = 1.0 / (yb * yb)
    series = (1.0 / 12.0 - r2 * (1.0 / 360.0 - r2 * (1.0 / 1260.0 - r2 * (1.0 / 1680.0 - r2 / 1188.0)))) / yb
    return np.where(small, exact, series)


def _bd0(x, m):
    """x log(x / m) + m - x >= 0 (the deviance term, Loader 2000), without cancellation when x is close to m."""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        near = np.abs(x - m) < 0.25 * (x + m)
        d = np.log1p((x - m) / m)
        out = np.where(near, m * phi(np.where(near, d, 0.0)), x * np.log(x / m) + m - x)
    return np.where(x == 0.0, m, out)


def logpmf(y, kind, x, n=None):
    """log P(y) of the Poisson (mean x) or binomial (n trials, probability x, 0 < x < 1) law in the saddle-point form
    of Loader (2000): -stirlerr - bd0 - log(2 pi y)/2 and its binomial twin.  Its terms are of order 1, so it keeps
    an absolute error near 1e-15 where scipy.stats' logpmf (a difference of lgamma values of order y log y) is off by
    1e-11 at 1e4 counts -- enough to miss a 1e-12 relative agreement on I."""
    y = np.asarray(y, dtype=np.float64)
    with np.errstate(divide='ignore', invalid='ignore'):
        if kind == 'poisson':
            yy = np.maximum(y, 1.0)
            lp = -_stirlerr(yy) - _bd0(yy, x) - 0.5 * np.log(2.0 * np.pi * yy)
            return np.where(y == 0.0, -x, lp)
        yy = np.clip(y, 1.0, n - 1.0) if n > 1 else np.ones_like(y)
        lp = (_stirlerr(n) - _stirlerr(yy) - _stirlerr(n - yy) - _bd0(yy, n * x) - _bd0(n - yy, n * (1.0 - x))
              + 0.5 * np.log(n / (2.0 * np.pi * yy * (n - yy))))
        return np.where(y == 0.0, n * np.log1p(-x), np.where(y == n, n * np.log(x), lp))


def _one_setting(x, kind, n):
    """I of one setting from the K outputs x (all valid, not all equal)."""
    from scipy.special import logsumexp
    K = len(x)
    interior = x > 0.0 if kind == 'poisson' else (x > 0.0) & (x < 1.0)
    if not np.any(interior):                      # binomial point masses at 0 and n only: the entropy of the split
        f = np.array([np.sum(x == 0.0), np.sum(x == 1.0)], dtype=np.float64) / K
        f = f[f > 0]
        return float(-np.sum(f * np.log(f)))
    idx = np.flatnonzero(interior)
    r = idx[np.argsort(x[idx], kind='stable')[(len(idx) - 1) // 2]]
    xr = x[r]
    y = union_counts(*windows(x, kind, n))
    xk = x[:, None]
    with np.errstate(divide='ignore', invalid='ignore'):
        if kind == 'poisson':
            B = xk - xr
            A = np.log1p(B / xr)
            delta = np.where(y[None, :] == 0.0, -B, y[None, :] * A - B)
            logp_r = logpmf(y, 'poisson', xr)
        else:
            A = np.log1p((xk - xr) / xr)
            B = np.log1p((xr - xk) / (1.0 - xr))
            ta = np.where(y[None, :] > 0.0, y[None, :] * A, 0.0)
            tb = np.where(y[None, :] < n, (n - y[None, :]) * B, 0.0)
            delta = ta + tb
            logp_r = logpmf(y, 'binomial', xr, n)
    delta[r] = 0.0
    # the mixture: log pbar = log p_r + logsumexp(delta) - log K
    logpbar = logp_r + logsumexp(delta, axis=0, b=1.0 / K)
    # the log ratios, with the digits of a mixture close to every component
    M = np.max(delta, axis=0)
    with np.errstate(invalid='ignore'):
        L = np.log1p(np.mean(np.expm1(delta - M), axis=0))
        d = (delta - M) - L
    terms = np.exp(logpbar) * np.sum(phi(d), axis=0)
    return float(np.sum(terms) / K)


def information_gain_from_draws(y_space, kind, aux=None, cost=1.0):
    """(S,) information gain in nats of y_space (K, S) or (K, 1, S), the K draws' model outputs at every setting:
    expected counts for ``kind='poisson'``, success probabilities for ``kind='binomial'`` with ``aux`` = n trials.
    Divided by ``cost``; exactly 0 where some draw's output is invalid and where all K outputs are equal."""
    y_space = np.asarray(y_space, dtype=np.float64)
    if y_space.ndim == 3:
        if y_space.shape[1] != 1:
            raise ValueError('information gain: single-channel outputs only')
        y_space = y_space[:, 0, :]
    n = None
    if kind == 'binomial':
        n = float(np.asarray(aux, dtype=np.float64).reshape(-1)[0])
        if not (n >= 1.0 and n == np.floor(n)):
            raise ValueError(f'information gain: the binomial trial count must be an integer >= 1, got {aux!r}')
    K, S = y_space.shape
    ok = np.all(valid_outputs(y_space, kind), axis=0)
    out = np.zeros(S)
    for s in range(S):
        x = y_space[:, s]
        if ok[s] and not np.all(x == x[0]):
            out[s] = _one_setting(x, kind, n)
    cost = np.broadcast_to(np.asarray(cost, dtype=np.float64), (S,))
    with np.errstate(invalid='ignore', divide='ignore'):
        u = out / cost
    return np.where(ok, u, 0.0)


class OracleOBEInfo(OracleOBEDesign):
    """OracleOBEDesign with ``method='information_gain'``: selects with :func:`information_gain_from_draws`
    (aux = ``design_aux``); any other method selects as OracleOBEDesign does.  A closed loop that follows another
    engine's choice sets ``last_setting_index`` to it and measures there."""

    def __init__(self, *args, method='information_gain', **kwargs):
        kwargs.setdefault('design_noise', 'likelihood')
        OracleOBEDesign.__init__(self, *args, **kwargs)
        self.method = method

    def utility(self):
        if self.method != 'information_gain':
            return OracleOBEDesign.utility(self)
        draws, _ = randdraw(self.particles, self.particle_weights, self.rng.random(self.N_DRAWS))
        _, y_space = yvar_from_draws(self.model, self.allsettings, draws, self.cons, self.n_channels)
        cost = 1.0
        if self.cost_of_changing_setting is not None:
            cost = lockin_cost(self.allsettings.shape[1], self.last_setting_index, self.cost_of_changing_setting)
        self.last_utility = information_gain_from_draws(y_space, self.likelihood_model, self.design_aux, cost=cost)
        return self.last_utility

