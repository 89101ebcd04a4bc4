"""Restatement of the batched simulator's count sampler (csrc/obe_device.cuh: obe_poisson_draw, obe_binomial_draw) and
of the batched count record, for the tests.

Draw c of instance b in cycle t takes its uniforms from Philox4x32-10 with ctr = (b, t, 0x60000000 | c, attempt) and
key = the simulator seed; attempt j gives u = u53(x0, x1) and v = u53(x2, x3).  Below a mean of 10 (Poisson lam < 10,
binomial n min(p, 1 - p) < 10) the count is the inversion of u through the pmf recurrence; at or above it, Hormann's
transformed rejection (PTRS for Poisson, BTRS for binomial with p > 1/2 by symmetry), one attempt per Philox call, at
most 64 attempts (NaN after that).  Every operation is the device's, in its order and without contraction, so the counts
agree bit for bit except where a decision depends on the last bits of exp / log1p / log / lgamma.  Each draw therefore
also returns its decision margin: the distance of u from the inversion's CDF values, or of the acceptance test from its
boundary relative to the size of its two sides (inf where no such decision was taken).
"""
import numpy as np
from scipy.special import gammaln

from oracle.obe_oracle import philox4x32_10

COUNT_CTR = 0x60000000
COUNT_TRIES = 64
MEAN_SWITCH = 10.0
MAX_TRIALS = 2.0 ** 31


def count_uniforms(seed, inst, cycle, channel, attempt):
    """(u, v): the two 53-bit uniforms of ``attempt`` for the instances ``inst`` (uint32 array)."""
    x = philox4x32_10(np.asarray(inst, dtype=np.uint32), np.uint32(cycle), np.uint32(COUNT_CTR | channel),
                      np.uint32(attempt), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)

    def u53(lo, hi):
        v = (hi.astype(np.uint64) << np.uint64(32)) | lo.astype(np.uint64)
        return ((v >> np.uint64(11)).astype(np.float64) + 0.5) * (2.0 ** -53)
    return u53(x[0], x[1]), u53(x[2], x[3])


def _test_margin(lhs, rhs):
    """Distance of an acceptance test lhs <= rhs from its boundary, relative to the size of its two sides."""
    return np.abs(lhs - rhs) / np.maximum(1.0, np.maximum(np.abs(lhs), np.abs(rhs)))


def _inversion(u, p0, step, kmax):
    """k = the first count whose CDF reaches u, with pmf(0) = p0 and pmf(k) = pmf(k-1) * step(k); the walk stops at
    kmax or when the pmf underflows.  Returns (k, margin)."""
    k = np.zeros_like(u)
    p = p0.copy()
    F = p0.copy()
    Fprev = np.full_like(u, -np.inf)
    live = (u > F) & (p > 0) & (k < kmax)
    while np.any(live):
        k = np.where(live, k + 1.0, k)
        p = np.where(live, p * step(np.where(live, k, 1.0)), p)
        Fprev = np.where(live, F, Fprev)
        F = np.where(live, F + p, F)
        live = live & (u > F) & (p > 0) & (k < kmax)
    return k, np.minimum(np.abs(F - u), np.abs(u - Fprev))


def poisson_counts(lam, seed, inst, cycle, channel=0):
    """(k, margin) of the Poisson draws with means ``lam`` (one per instance in ``inst``)."""
    lam = np.asarray(lam, dtype=np.float64) * np.ones(np.shape(inst))
    inst = np.asarray(inst, dtype=np.uint32)
    k = np.full(lam.shape, np.nan)
    margin = np.full(lam.shape, np.inf)
    valid = (lam >= 0.0) & (lam <= np.finfo(np.float64).max)
    small = valid & (lam < MEAN_SWITCH)
    if np.any(small):
        u, _ = count_uniforms(seed, inst[small], cycle, channel, 0)
        ls = lam[small]
        k[small], margin[small] = _inversion(u, np.exp(-ls), lambda kk: ls / kk, np.inf)
    big = np.flatnonzero(valid & ~small)
    if big.size:
        lb = lam[big]
        with np.errstate(all='ignore'):
            slam = np.sqrt(lb)
            loglam = np.log(lb)
            b = 0.931 + 2.53 * slam
            a = -0.059 + 0.02483 * b
            invalpha = 1.1239 + 1.1328 / (b - 3.4)
            vr = 0.9277 - 3.6224 / (b - 2.0)
        out = np.full(big.size, np.nan)
        mg = np.full(big.size, np.inf)
        todo = np.ones(big.size, dtype=bool)
        for j in range(COUNT_TRIES):
            i = np.flatnonzero(todo)
            if i.size == 0:
                break
            u, v = count_uniforms(seed, inst[big[i]], cycle, channel, j)
            U = u - 0.5
            us = 0.5 - np.abs(U)
            kk = np.floor((((2.0 * a[i]) / us + b[i]) * U + lb[i]) + 0.43)
            box = (us >= 0.07) & (v <= vr[i])
            rej = ~box & ((kk < 0) | ((us < 0.013) & (v > us)))
            test = ~box & ~rej
            with np.errstate(all='ignore'):
                lhs = (np.log(v) + np.log(invalpha[i])) - np.log(a[i] / (us * us) + b[i])
                kl = kk * loglam[i]
                lg = gammaln(kk + 1.0)
                rhs = (-lb[i] + kl) - lg
                mg[i] = np.where(test, np.minimum(mg[i], _test_margin(lhs, rhs)), mg[i])
            acc = box | (test & (lhs <= rhs))
            out[i[acc]] = kk[acc]
            todo[i[acc]] = False
        k[big], margin[big] = out, mg
    return k, margin


def binomial_counts(n, p, seed, inst, cycle, channel=0):
    """(k, margin) of the binomial draws of ``n`` trials with success probabilities ``p``."""
    shape = np.shape(inst)
    n = np.asarray(n, dtype=np.float64) * np.ones(shape)
    p = np.asarray(p, dtype=np.float64) * np.ones(shape)
    inst = np.asarray(inst, dtype=np.uint32)
    k = np.full(shape, np.nan)
    margin = np.full(shape, np.inf)
    valid = (p >= 0.0) & (p <= 1.0) & (n >= 0.0) & (n <= MAX_TRIALS) & (n == np.floor(n))
    flip = p > 0.5
    q = np.where(flip, 1.0 - p, p)
    small = valid & (n * q < MEAN_SWITCH)
    res = np.full(shape, np.nan)
    if np.any(small):
        u, _ = count_uniforms(seed, inst[small], cycle, channel, 0)
        qs, ns = q[small], n[small]
        with np.errstate(all='ignore'):
            r = qs / (1.0 - qs)
            p0 = np.exp(ns * np.log1p(-qs))
        res[small], margin[small] = _inversion(u, p0, lambda kk: (r * ((ns - kk) + 1.0)) / kk, ns)
    big = np.flatnonzero(valid & ~small)
    if big.size:
        qb, nb = q[big], n[big]
        qq = 1.0 - qb
        spq = np.sqrt((nb * qb) * qq)
        b = 1.15 + 2.53 * spq
        a = (-0.0873 + 0.0248 * b) + 0.01 * qb
        c = nb * qb + 0.5
        alpha = (2.83 + 5.1 / b) * spq
        vr = 0.92 - 4.2 / b
        m = np.floor((nb + 1.0) * qb)
        lpq = np.log(qb / qq)
        h = gammaln(m + 1.0) + gammaln((nb - m) + 1.0)
        out = np.full(big.size, np.nan)
        mg = np.full(big.size, np.inf)
        todo = np.ones(big.size, dtype=bool)
        for j in range(COUNT_TRIES):
            i = np.flatnonzero(todo)
            if i.size == 0:
                break
            u, v = count_uniforms(seed, inst[big[i]], cycle, channel, j)
            U = u - 0.5
            us = 0.5 - np.abs(U)
            kk = np.floor(((2.0 * a[i]) / us + b[i]) * U + c[i])
            inside = (kk >= 0) & (kk <= nb[i])
            box = inside & (us >= 0.07) & (v <= vr[i])
            test = inside & ~box
            with np.errstate(all='ignore'):
                lhs = np.log((v * alpha[i]) / (a[i] / (us * us) + b[i]))
                lg = gammaln(kk + 1.0) + gammaln((nb[i] - kk) + 1.0)
                tl = (kk - m[i]) * lpq[i]
                rhs = (h[i] - lg) + tl
                mg[i] = np.where(test, np.minimum(mg[i], _test_margin(lhs, rhs)), mg[i])
            acc = box | (test & (lhs <= rhs))
            out[i[acc]] = kk[acc]
            todo[i[acc]] = False
        res[big], margin[big] = out, mg
    k = np.where(flip, n - res, res)
    return k, margin


def count_record(counts, aux, likelihood):
    """The batched count record of one instance as the likelihood oracles take it: (y_meas, aux, lconst) per channel,
    lconst the per-record log-factorial constants the batched update computes on the device (lgamma(k + 1) for
    Poisson, lgamma(n + 1) - lgamma(k + 1) - lgamma(n - k + 1) for binomial, 0 for a user likelihood).  The
    constants match the terms of loglik_poisson / loglik_binomial, which are the likelihoods of this record."""
    k = np.atleast_1d(np.asarray(counts, dtype=np.float64))
    a = np.broadcast_to(np.atleast_1d(np.asarray(aux, dtype=np.float64)), k.shape)
    if likelihood == 'poisson':
        lconst = gammaln(k + 1.0)
    elif likelihood == 'binomial':
        lconst = (gammaln(a + 1.0) - gammaln(k + 1.0)) - gammaln((a - k) + 1.0)
    else:
        lconst = np.zeros_like(k)
    return k, a, lconst
