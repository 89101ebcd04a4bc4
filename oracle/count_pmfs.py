"""User count likelihoods for ``cuda_likelihood(..., window=)``  --  TEST INFRASTRUCTURE, NOT PRODUCT.

Each pmf is given twice: as CUDA source (entry, noise_var and window device functions, as a user would write them)
and as its numpy twin for :func:`oracle.information_gain_user.information_gain_user` and the oracle engines.  The numpy
functions take ``(y_model, y, aux)`` like the CUDA entry and broadcast; ``window(x, aux)`` returns float (lo, hi).

- ``poisson``: the built-in Poisson restated as a user pmf, with the built-in's windows;
- ``negbin``: a negative binomial with mean ``x`` and shape ``r = aux`` (variance x + x^2 / r);
- ``readout``: single-shot state readout, ``P Pois(lam_b) + (1 - P) Pois(lam_d)`` with ``P = x``;
- ``betabinom``: a beta-binomial with ``n = aux`` trials, mean probability ``x`` and ``alpha + beta = phi``.

Every window leaves out less than 1e-17 of its component's mass (checked in tests/test_information_gain_user_host.py).
"""
import numpy as np
from scipy.special import gammaln

from .information_gain import WINDOW_PAD, WINDOW_VAR


def _lit(v):
    return repr(float(v))


#: -inf in NVRTC source (which has no math.h macros)
NEG_INF = '__longlong_as_double(0xfff0000000000000LL)'

POISSON_SOURCE = r'''
__device__ double pois_lp(const double* ym, const double* y, const double* aux, int n) {
    const double lam = ym[0], k = y[0];
    if (lam == 0.0) return k == 0.0 ? 0.0 : NEG_INF;
    return k * log(lam) - lam - lgamma(k + 1.0);
}
__device__ double pois_var(double lam, double a) { return lam; }
__device__ void pois_win(double lam, double a, double* lo, double* hi) {
    const double t = lam > 0.0 ? sqrt(79.0 * lam) + 27.0 : 0.0;
    *lo = fmax(ceil(lam - t), 0.0);
    *hi = floor(lam + t);
}
'''.replace('NEG_INF', NEG_INF)

NEGBIN_SOURCE = r'''
__device__ double nb_lp(const double* ym, const double* y, const double* aux, int n) {
    const double m = ym[0], k = y[0], r = aux[0];
    if (m == 0.0) return k == 0.0 ? 0.0 : NEG_INF;
    return ((lgamma(k + r) - lgamma(r)) - lgamma(k + 1.0)) - r * log1p(m / r) + k * (log(m) - log(r + m));
}
__device__ double nb_var(double m, double r) { return m + m * m / r; }
__device__ void nb_win(double m, double r, double* lo, double* hi) {
    *lo = 0.0;
    *hi = floor(m + sqrt(80.0 * (m + m * m / r)) + 80.0 * (1.0 + m / r));
}
'''.replace('NEG_INF', NEG_INF)


def readout_source(lam_d, lam_b):
    return r'''
__device__ double ro_lp(const double* ym, const double* y, const double* aux, int n) {
    const double P = ym[0], k = y[0];
    const double a = log(P) + (k * log(LAM_B) - LAM_B), b = log1p(-P) + (k * log(LAM_D) - LAM_D);
    const double m = fmax(a, b);
    if (m == NEG_INF) return NEG_INF;
    return (m + log1p(exp(-fabs(a - b)))) - lgamma(k + 1.0);
}
__device__ double ro_var(double P, double a) {
    if (!(P >= 0.0 && P <= 1.0)) return -1.0;
    return P * LAM_B + (1.0 - P) * LAM_D + P * (1.0 - P) * (LAM_B - LAM_D) * (LAM_B - LAM_D);
}
__device__ void ro_win(double P, double a, double* lo, double* hi) {
    *lo = 0.0;
    *hi = floor(LAM_B + sqrt(79.0 * LAM_B) + 27.0);
}
'''.replace('NEG_INF', NEG_INF).replace('LAM_B', _lit(lam_b)).replace('LAM_D', _lit(lam_d))


def betabinom_source(phi):
    return r'''
__device__ double bb_lp(const double* ym, const double* y, const double* aux, int nc) {
    const double mu = ym[0], k = y[0], n = aux[0];
    if (mu == 0.0) return k == 0.0 ? 0.0 : NEG_INF;
    if (mu == 1.0) return k == n ? 0.0 : NEG_INF;
    const double a = mu * PHI, b = (1.0 - mu) * PHI;
    return ((lgamma(n + 1.0) - lgamma(k + 1.0)) - lgamma(n - k + 1.0))
         + (((lgamma(k + a) + lgamma(n - k + b)) - lgamma(n + PHI)) - ((lgamma(a) + lgamma(b)) - lgamma(PHI)));
}
__device__ double bb_var(double mu, double n) { return n * mu * (1.0 - mu) * (PHI + n) / (PHI + 1.0); }
__device__ void bb_win(double mu, double n, double* lo, double* hi) {
    *lo = 0.0;
    *hi = n;
}
'''.replace('NEG_INF', NEG_INF).replace('PHI', _lit(phi))


# ---- the numpy twins --------------------------------------------------------------------------------------------
def _safe(fn, *args):
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        return fn(*args)


def poisson_logpmf(x, y, aux=None):
    def f(x, y):
        x, y = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64))
        lp = y * np.log(x) - x - gammaln(y + 1.0)
        return np.where(x == 0.0, np.where(y == 0.0, 0.0, -np.inf), lp)
    return _safe(f, x, y)


def poisson_var(x, aux=None):
    return np.asarray(x, np.float64)


def poisson_window(x, aux=None):
    x = np.asarray(x, np.float64)
    with np.errstate(invalid='ignore'):
        t = np.where(x > 0.0, np.sqrt(WINDOW_VAR * x) + WINDOW_PAD, 0.0)
        return np.maximum(np.ceil(x - t), 0.0), np.floor(x + t)


def negbin_logpmf(x, y, r):
    def f(x, y):
        x, y = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64))
        lp = ((gammaln(y + r) - gammaln(r)) - gammaln(y + 1.0)) - r * np.log1p(x / r) + y * (np.log(x) - np.log(r + x))
        return np.where(x == 0.0, np.where(y == 0.0, 0.0, -np.inf), lp)
    return _safe(f, x, y)


def negbin_var(x, r):
    x = np.asarray(x, np.float64)
    return x + x * x / r


def negbin_window(x, r):
    x = np.asarray(x, np.float64)
    with np.errstate(invalid='ignore'):
        return np.zeros_like(x), np.floor(x + np.sqrt(80.0 * (x + x * x / r)) + 80.0 * (1.0 + x / r))


def readout(lam_d, lam_b):
    """(logpmf, noise_var, window) of the two-Poisson readout with dark and bright rates lam_d < lam_b."""
    def logpmf(x, y, aux=None):
        def f(x, y):
            x, y = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64))
            a = np.log(x) + (y * np.log(lam_b) - lam_b)
            b = np.log1p(-x) + (y * np.log(lam_d) - lam_d)
            return np.logaddexp(a, b) - gammaln(y + 1.0)
        return _safe(f, x, y)

    def noise_var(x, aux=None):
        x = np.asarray(x, np.float64)
        with np.errstate(invalid='ignore'):
            v = x * lam_b + (1.0 - x) * lam_d + x * (1.0 - x) * (lam_b - lam_d) ** 2
            return np.where((x >= 0.0) & (x <= 1.0), v, -1.0)

    def window(x, aux=None):
        x = np.asarray(x, np.float64)
        return np.zeros_like(x), np.full_like(x, np.floor(lam_b + np.sqrt(WINDOW_VAR * lam_b) + WINDOW_PAD))
    return logpmf, noise_var, window


def betabinom(phi):
    """(logpmf, noise_var, window) of the beta-binomial with alpha + beta = phi, n = aux trials."""
    def logpmf(x, y, n):
        def f(x, y):
            x, y = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64))
            a, b = x * phi, (1.0 - x) * phi
            lp = (((gammaln(n + 1.0) - gammaln(y + 1.0)) - gammaln(n - y + 1.0))
                  + (((gammaln(y + a) + gammaln(n - y + b)) - gammaln(n + phi)) - ((gammaln(a) + gammaln(b))
                                                                                    - gammaln(phi))))
            lp = np.where(x == 0.0, np.where(y == 0.0, 0.0, -np.inf), lp)
            return np.where(x == 1.0, np.where(y == n, 0.0, -np.inf), lp)
        return _safe(f, x, y)

    def noise_var(x, n):
        x = np.asarray(x, np.float64)
        return n * x * (1.0 - x) * (phi + n) / (phi + 1.0)

    def window(x, n):
        x = np.asarray(x, np.float64)
        return np.zeros_like(x), np.full_like(x, float(n))
    return logpmf, noise_var, window


def pmf(name, **kw):
    """(source, entry, noise_var, window, logpmf, noise_var_np, window_np) of a named pmf (see the module doc)."""
    if name == 'poisson':
        return (POISSON_SOURCE, 'pois_lp', 'pois_var', 'pois_win', poisson_logpmf, poisson_var, poisson_window)
    if name == 'negbin':
        return (NEGBIN_SOURCE, 'nb_lp', 'nb_var', 'nb_win', negbin_logpmf, negbin_var, negbin_window)
    if name == 'readout':
        lam_d, lam_b = kw.get('lam_d', 0.5), kw.get('lam_b', 3.0)
        return (readout_source(lam_d, lam_b), 'ro_lp', 'ro_var', 'ro_win') + readout(lam_d, lam_b)
    if name == 'betabinom':
        phi = kw.get('phi', 20.0)
        return (betabinom_source(phi), 'bb_lp', 'bb_var', 'bb_win') + betabinom(phi)
    raise ValueError(f'unknown pmf {name!r}')
