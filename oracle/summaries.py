"""numpy restatement of the posterior summaries (optbayesexpt_b200/summaries.py, csrc/obe_summary.cuh).

Exact by construction: fixed-point masses are numpy uint64 (integer sums, so their order does not matter),
the quantile target is computed with Python integers, and the histogram bins follow numpy's own rules.
"""
import math
from fractions import Fraction

import numpy as np

SCALE = 2.0 ** 62


def quantised(weights):
    """wq = rint(w * 2^62) as uint64 (round half to even, like __double2ull_rn); negative weights give 0."""
    w = np.asarray(weights, dtype=np.float64) * SCALE
    w = np.where(w > 0.0, w, 0.0)
    q = np.rint(w)
    out = np.zeros(q.shape, dtype=np.uint64)
    big = q >= 2.0 ** 64
    out[~big] = q[~big].astype(np.uint64)
    out[big] = np.uint64(2 ** 64 - 1)
    return out


def total(wq):
    """W = sum(wq) as a Python int; weights that sum to 4 or more (W >= 2^64) are refused, as on the device."""
    W = int(np.sum(wq >> np.uint64(32), dtype=np.uint64)) * 2 ** 32 + int(np.sum(wq & np.uint64(2 ** 32 - 1),
                                                                                dtype=np.uint64))
    if W >= 2 ** 64:
        raise ValueError('weights sum to 4 or more')
    return W


def target(q, W):
    """T = max(1, ceil(q W)), exact."""
    return max(1, math.ceil(Fraction(float(q)) * int(W)))


def _canon(x):
    # -0.0 and +0.0 are one value; the answer is reported as +0.0
    return np.where(x == 0.0, 0.0, x)


def quantile(x, wq, levels):
    """Smallest coordinate x* with sum(wq[x <= x*]) >= T for each level."""
    keep = wq > 0
    x = _canon(np.asarray(x, dtype=np.float64)[keep])
    w = wq[keep]
    W = total(w)
    if W == 0:
        raise ValueError('empty posterior')
    order = np.argsort(x, kind='stable')
    xs, cum = x[order], np.cumsum(w[order], dtype=np.uint64)
    out = []
    for q in np.atleast_1d(levels):
        i = int(np.searchsorted(cum, np.uint64(target(q, W)), side='left'))
        out.append(xs[i])
    return np.array(out)


def quantiles(particles, weights, levels, params=None):
    """(len(params), len(levels)) quantiles of the rows of particles (d, n) with float weights."""
    wq = quantised(weights)
    params = range(particles.shape[0]) if params is None else params
    return np.stack([quantile(particles[p], wq, levels) for p in params])


def auto_range(x, wq):
    keep = wq > 0
    return float(np.min(x[keep])), float(np.max(x[keep]))


def hist_index(x, edges):
    """np.histogram's bin of each x for uniform edges (-1: outside): computed index, then its correction."""
    nb = len(edges) - 1
    first, last = edges[0], edges[-1]
    idx = np.full(x.shape, -1, dtype=np.intp)
    keep = (x >= first) & (x <= last)
    xs = x[keep]
    f = ((xs - first) / (last - first)) * nb
    k = f.astype(np.intp)
    k[k == nb] -= 1
    k[xs < edges[k]] -= 1
    k[(xs >= edges[k + 1]) & (k != nb - 1)] += 1
    idx[keep] = k
    return idx


def dd_index(x, edges):
    """np.histogramdd's bin of each x along one axis (-1: outside): searchsorted right, last edge closed."""
    nb = len(edges) - 1
    k = np.searchsorted(edges, x, side='right')
    k[x == edges[-1]] -= 1
    k = k - 1
    k[(k < 0) | (k >= nb)] = -1
    return k


def u64_bincount(idx, wq, nb):
    """Exact uint64 sums of wq per bin (three 22-bit slices, each summed exactly in float64)."""
    keep = idx >= 0
    idx, wq = idx[keep], wq[keep]
    total = np.zeros(nb, dtype=np.uint64)
    for shift in (0, 22, 44):
        part = ((wq >> np.uint64(shift)) & np.uint64((1 << 22) - 1)).astype(np.float64)
        s = np.bincount(idx, weights=part, minlength=nb)
        total += s.astype(np.uint64) << np.uint64(shift)
    return total, np.bincount(idx, minlength=nb).astype(np.uint64)


def histogram(x, wq, edges):
    """(raw u64 mass, counts) of one row."""
    keep = wq > 0
    return u64_bincount(hist_index(np.asarray(x, dtype=np.float64)[keep], edges), wq[keep], len(edges) - 1)


def histogram2d(x, y, wq, xedges, yedges):
    keep = wq > 0
    bx, by = len(xedges) - 1, len(yedges) - 1
    ix, iy = dd_index(x[keep], xedges), dd_index(y[keep], yedges)
    flat = np.where((ix >= 0) & (iy >= 0), ix * by + iy, -1)
    raw, counts = u64_bincount(flat, wq[keep], bx * by)
    return raw.reshape(bx, by), counts.reshape(bx, by)


def mass(raw):
    return raw.astype(np.float64) * 2.0 ** -62
