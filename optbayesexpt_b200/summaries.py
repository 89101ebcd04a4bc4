"""Posterior summaries computed on the device: weighted quantiles and 1-D / 2-D marginal histograms.

``ParticlePDF.quantile`` / ``histogram`` / ``histogram2d`` (and so every engine class built on it) call the
kernels of ``csrc/obe_summary.cuh`` through the C ABI.  Only the small results come back to the host; the
cloud, its weights and the engine's state are left as they were.

Definitions (see INTEGRATION.md):
  * a particle's mass is ``wq = rint(w * 2**62)`` as an unsigned 64-bit integer, ``w`` its normalised weight as
    ``particle_weights`` returns it; particles with ``wq == 0`` take no part; the weights must sum to less than 4
    (normalised weights sum to 1), else ``sum(wq)`` would not fit in 64 bits and the call raises;
  * ``quantile``: with ``W = sum(wq)`` and ``T = max(1, ceil(q * W))`` (exact), the smallest coordinate ``x*``
    with ``sum(wq[x <= x*]) >= T``;
  * ``histogram`` / ``histogram2d``: numpy's edges and bin rule, mass ``sum(wq) * 2**-62`` per bin.

This module holds the argument checks and the edge computation, so they can be exercised without a GPU.
"""
import ctypes as C
import numbers

import numpy as np

from . import _lib

MAX_Q = 16
MAX_BINS = 4096
MAX_BINS2D = 65536
MASS_SCALE = 2.0 ** -62


def _index(value, n_dims, what='parameter index'):
    if isinstance(value, (bool, np.bool_)) or not isinstance(value, numbers.Integral):
        raise TypeError(f'{what} must be an integer, got {value!r}')
    value = int(value)
    if not 0 <= value < n_dims:
        raise ValueError(f'{what} {value} out of range for {n_dims} parameters')
    return value


def param_list(params, n_dims):
    """The parameter rows a summary covers: all of them for None, else an int or a sequence of ints."""
    if params is None:
        return list(range(n_dims))
    if isinstance(params, numbers.Integral) and not isinstance(params, (bool, np.bool_)):
        params = [params]
    params = [_index(p, n_dims) for p in params]
    if not 1 <= len(params) <= _lib.MAX_PARAMS:
        raise ValueError(f'params must name 1..{_lib.MAX_PARAMS} parameters')
    return params


def quantile_levels(q):
    """q as a float64 vector of 1..16 levels in [0, 1]."""
    levels = np.atleast_1d(np.asarray(q, dtype=np.float64))
    if levels.ndim != 1 or not 1 <= levels.shape[0] <= MAX_Q:
        raise ValueError(f'q must be a scalar or a sequence of 1..{MAX_Q} levels')
    if not np.all((levels >= 0.0) & (levels <= 1.0)):      # NaN fails too
        raise ValueError('quantile levels must lie in [0, 1]')
    return np.ascontiguousarray(levels)


def _bin_count(bins, limit):
    if isinstance(bins, (bool, np.bool_)) or not isinstance(bins, numbers.Integral):
        raise TypeError(f'bins must be an integer, got {bins!r}')
    bins = int(bins)
    if not 1 <= bins <= limit:
        raise ValueError(f'bins must be 1..{limit}, got {bins}')
    return bins


def hist_bins(bins):
    return _bin_count(bins, MAX_BINS)


def hist_bins2d(bins):
    """An int or a pair -> (bins_x, bins_y) with bins_x * bins_y <= 65536."""
    if isinstance(bins, numbers.Integral) and not isinstance(bins, (bool, np.bool_)):
        bx = by = bins
    else:
        try:
            bx, by = bins
        except (TypeError, ValueError):
            raise TypeError('bins must be an integer or a pair of integers') from None
    bx, by = _bin_count(bx, MAX_BINS2D), _bin_count(by, MAX_BINS2D)
    if bx * by > MAX_BINS2D:
        raise ValueError(f'bins_x * bins_y must be at most {MAX_BINS2D}, got {bx} * {by}')
    return bx, by


def edges_for(lo, hi, bins):
    """np.histogram's edges for the range (lo, hi): its checks, its widening of an empty range, its linspace."""
    return np.histogram_bin_edges(np.empty(0), bins=bins, range=(float(lo), float(hi)))


def hist_ranges(range, n):
    """None, one (lo, hi) pair for every row, or n pairs -> list of n (lo, hi) or None."""
    if range is None:
        return None
    arr = np.asarray(range, dtype=np.float64)
    if arr.shape == (2,):
        return [tuple(arr)] * n
    if arr.shape == (n, 2):
        return [tuple(r) for r in arr]
    raise ValueError(f'range must be (lo, hi) or {n} such pairs')


def mass_from_fixed(raw):
    """u64 fixed-point sums -> float64 mass."""
    return raw.astype(np.float64) * MASS_SCALE


class SummaryMixin:
    """The three summary methods of ParticlePDF (the engine supplies _buf, _cs, _stream, _check, _lib)."""

    def _summary_scratch(self, nbytes):
        buf = getattr(self, '_summary_buf', None)
        if buf is None or buf.numel() < nbytes or buf.device != self._buf.device:
            buf = self._summary_buf = self._torch.empty(int(nbytes), dtype=self._torch.uint8,
                                                        device=self._buf.device)
        return C.c_void_p(buf.data_ptr())

    def _summary_range(self, params):
        lo = np.empty(len(params))
        hi = np.empty(len(params))
        scratch = self._summary_scratch(self._lib.obe_histogram_scratch_bytes(len(params), 1))
        self._check(self._lib.obe_summary_range(self._cs(), _lib.iarr(params), len(params), scratch, _lib.dptr(lo),
                                                _lib.dptr(hi), self._stream()))
        return lo, hi

    def quantile(self, q, params=None):
        """Weighted quantiles of each requested parameter's marginal, shape (len(params), len(q)).

        The result for level q is the smallest particle coordinate x* whose cumulative weight reaches
        max(1, ceil(q W)) in 2**-62 fixed-point units, so q = 0 / 1 give the minimum / maximum of the
        particles with weight.  Computed on the device; the engine's state is not changed."""
        if self._pending_cycle:
            self._settle()
        levels = quantile_levels(q)
        params = param_list(params, self.n_dims)
        out = np.empty(len(params) * len(levels))
        scratch = self._summary_scratch(self._lib.obe_quantile_scratch_bytes(len(params), len(levels)))
        self._check(self._lib.obe_quantile(self._cs(), _lib.iarr(params), len(params), _lib.dptr(levels),
                                           len(levels), scratch, _lib.dptr(out), self._stream()))
        return out.reshape(len(params), len(levels))

    def histogram(self, bins, range=None, params=None, return_counts=False):
        """Weighted 1-D marginal histograms: (mass (len(params), bins), edges (len(params), bins + 1)).

        Edges and bin membership are np.histogram's; with range=None each parameter's range is the min / max of
        its particles with weight.  ``range`` is one (lo, hi) for all parameters or one per parameter.  With
        return_counts the unweighted particle count per bin (uint64) comes third."""
        if self._pending_cycle:
            self._settle()
        bins = hist_bins(bins)
        params = param_list(params, self.n_dims)
        ranges = hist_ranges(range, len(params))
        if ranges is None:
            lo, hi = self._summary_range(params)
            ranges = list(zip(lo, hi))
        edges = np.ascontiguousarray(np.stack([edges_for(a, b, bins) for a, b in ranges]))
        raw = np.empty((len(params), bins), dtype=np.uint64)
        counts = np.empty((len(params), bins), dtype=np.uint64)
        scratch = self._summary_scratch(self._lib.obe_histogram_scratch_bytes(len(params), bins))
        self._check(self._lib.obe_histogram(self._cs(), _lib.iarr(params), len(params), _lib.dptr(edges), bins,
                                            scratch, raw.ctypes.data_as(C.POINTER(C.c_uint64)),
                                            counts.ctypes.data_as(C.POINTER(C.c_uint64)), self._stream()))
        mass = mass_from_fixed(raw)
        return (mass, edges, counts) if return_counts else (mass, edges)

    def histogram2d(self, i, j, bins, range=None, return_counts=False):
        """Joint weighted histogram of parameters i and j, shaped like np.histogram2d: (mass (bx, by), xedges,
        yedges).  bins: an int or a pair, bx * by <= 65536; range: None or [[xmin, xmax], [ymin, ymax]]."""
        if self._pending_cycle:
            self._settle()
        i, j = _index(i, self.n_dims), _index(j, self.n_dims)
        bx, by = hist_bins2d(bins)
        if range is None:
            lo, hi = self._summary_range([i, j])
            ranges = list(zip(lo, hi))
        elif np.asarray(range, dtype=np.float64).shape == (2, 2):
            ranges = hist_ranges(range, 2)
        else:
            raise ValueError('range must be [[xmin, xmax], [ymin, ymax]]')
        xedges = np.ascontiguousarray(edges_for(ranges[0][0], ranges[0][1], bx))
        yedges = np.ascontiguousarray(edges_for(ranges[1][0], ranges[1][1], by))
        raw = np.empty((bx, by), dtype=np.uint64)
        counts = np.empty((bx, by), dtype=np.uint64)
        scratch = self._summary_scratch(self._lib.obe_histogram2d_scratch_bytes(bx, by))
        self._check(self._lib.obe_histogram2d(self._cs(), i, j, _lib.dptr(xedges), bx, _lib.dptr(yedges), by,
                                              scratch, raw.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              counts.ctypes.data_as(C.POINTER(C.c_uint64)), self._stream()))
        mass = mass_from_fixed(raw)
        return (mass, xedges, yedges, counts) if return_counts else (mass, xedges, yedges)
