"""Particle cloud sharded over the GPUs of one node: one process per GPU (torch.distributed).

Particles are exchangeable, so every O(N) step is local to a shard; large setting grids are sliced for
the utility pass.  Only small vectors cross NVLink -- by peer writes into CUDA-IPC-mapped buffers with
system-scope flags (PeerLink, the default on an NCCL job) or through NCCL/gloo collectives:
  * after the update: the 64-double stats blocks of all ranks -> global normaliser, N_eff,
    mean, covariance, and the exclusive scan of shard weight totals (the inter-GPU CDF offsets);
  * the K drawn parameter sets: each shard produces the draws it owns (peer mode: stores them into
    every rank's buffer; collective mode: zeroed (d, K) buffer + one all-reduce(sum));
  * the argmax of a sliced grid: one all-gather of (value, index) pairs, lowest global index wins ties
    (grids up to 131072 settings are evaluated whole on every rank: no exchange).
Resampling needs NO particle exchange: shard g's particles own the global comb slots
[H_g, H_g+1), so shard lengths float by a fraction of a percent per resample inside a slack
capacity.  The host-side decisions are pure functions (combine_stats, shard_slot_bounds,
assign_draws, reduce_best) so they can be tested without a GPU (gloo).
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from .models import non_gaussian
from .obe_base import OptBayesExpt


# --------------------------------------------------------------------------------------------------
# pure host logic
# --------------------------------------------------------------------------------------------------
def combine_stats(gathered, d):
    """Global stats from the per-shard stats blocks, summed in rank order (identical on every rank).

    Returns a dict with totals (G,), offsets (G,), total, sumsq, sumt, m1 (d,), m2 packed, noise (4,),
    pivot (d,).  All shards must have used the same pivot."""
    g = np.asarray(gathered, dtype=np.float64)
    nm2 = d * (d + 1) // 2
    totals = g[:, _lib.ST_TOTAL].copy()
    offsets = np.zeros_like(totals)
    acc = 0.0
    for r in range(len(totals)):          # sequential: the canonical inter-GPU exclusive scan
        offsets[r] = acc
        acc = acc + totals[r]

    def rsum(cols):
        out = g[0, cols].copy()
        for r in range(1, g.shape[0]):
            out = out + g[r, cols]
        return out
    return dict(totals=totals, offsets=offsets, total=acc,
                sumsq=float(rsum([_lib.ST_SUMSQ])[0]), sumt=float(rsum([_lib.ST_SUMT])[0]),
                m1=rsum(list(range(_lib.ST_M1, _lib.ST_M1 + d))),
                m2=rsum(list(range(_lib.ST_M2, _lib.ST_M2 + nm2))),
                noise=rsum(list(range(_lib.ST_NOISE, _lib.ST_NOISE + 4))),
                pivot=g[0, _lib.ST_PIVOT:_lib.ST_PIVOT + d].copy())


def moments_from(gs, d):
    """(mean, covariance, biased variance, n_eff) from combined stats (same formulas as ParticlePDF)."""
    s = gs['sumt']
    mean = gs['pivot'] + gs['m1'] / s
    m2 = np.zeros((d, d))
    q = 0
    for j in range(d):
        for k in range(j, d):
            m2[j, k] = m2[k, j] = gs['m2'][q]
            q += 1
    cov = (m2 - np.outer(gs['m1'], gs['m1']) / s) / (s - gs['sumsq'] / s)
    var = np.diag(m2) / s - (gs['m1'] / s) ** 2
    n_eff = gs['total'] ** 2 / gs['sumsq']
    return mean, cov, var, n_eff


def shard_slot_bounds(offsets, total, u0, n_total, comb_count):
    """H_g: first global comb slot owned by shard g (H_0 = 0, H_G = n_total), monotone.
    comb_count(c, u0, n) must be the library's obe_comb_count so that neighbours agree to the bit."""
    inv_total = 1.0 / total
    bounds = [0]
    for g in range(1, len(offsets)):
        h = int(comb_count(float(offsets[g] * inv_total), float(u0), int(n_total)))
        bounds.append(min(max(h, bounds[-1]), int(n_total)))
    bounds.append(int(n_total))
    return bounds


def assign_draws(u, offsets, totals, total):
    """Owner shard and shard-local uniform of every global uniform u_k.
    Owner g: offset_g <= u*total < offset_g + total_g (last shard takes the remainder)."""
    u = np.asarray(u, dtype=np.float64)
    target = u * total
    ends = offsets + totals
    owner = np.searchsorted(ends, target, side='right')
    owner = np.minimum(owner, len(totals) - 1)
    # skip empty shards
    for i in range(len(owner)):
        while totals[owner[i]] <= 0 and owner[i] > 0:
            owner[i] -= 1
    local = (target - offsets[owner]) / np.where(totals[owner] > 0, totals[owner], 1.0)
    local = np.clip(local, 0.0, np.nextafter(1.0, 0.0))
    return owner, local


def reduce_best(pairs):
    """np.argmax over the concatenated grid from per-shard (global_index, value) pairs: the first
    maximum wins, NaN counts as the maximum (numpy semantics)."""
    best_i, best_v = -1, 0.0
    for idx, val in pairs:
        idx = int(idx)
        if idx < 0:
            continue
        if best_i < 0:
            take = True
        else:
            vn, bn = val != val, best_v != best_v
            if vn and bn:
                take = idx < best_i
            elif vn:
                take = True
            elif bn:
                take = False
            else:
                take = val > best_v or (val == best_v and idx < best_i)
        if take:
            best_i, best_v = idx, float(val)
    return best_i, best_v


REPLICATE_GRID_MAX = 131072
PEER_EXCHANGE_DEFAULT = '0'      # '1': stats and draws travel by peer writes over NVLink instead of NCCL


def setting_slice(n_settings, rank, world):
    lo = n_settings * rank // world
    hi = n_settings * (rank + 1) // world
    return lo, hi


class Comm:
    """The three small collectives, over torch.distributed (nccl on GPUs, gloo in CPU tests)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)

        self.backend = dist.get_backend(group)

    def _staged(self, t):
        # gloo moves host memory: stage device tensors through the CPU (tests on a single GPU)
        return self.backend == 'gloo' and t.is_cuda

    def allgather(self, vec):
        import torch
        src = vec.contiguous().view(-1)
        if self._staged(vec):
            src = src.cpu()
        parts = [torch.empty_like(src) for _ in range(self.world)]
        if self.backend == 'gloo':
            self.dist.all_gather(parts, src, group=self.group)
            out = torch.stack(parts)
        else:
            out = torch.empty((self.world, src.numel()), dtype=src.dtype, device=src.device)
            self.dist.all_gather_into_tensor(out.view(-1), src, group=self.group)
        return out.view((self.world,) + tuple(vec.shape)).to(vec.device)

    def alltoall_rows(self, dst, src, recv_sizes, send_sizes):
        """all-to-all-v of one contiguous row: src is cut into send_sizes (one piece per rank, in rank order), dst is
        filled with the recv_sizes pieces in rank order."""
        if self.backend == 'gloo':
            out = dst.cpu()
            self.dist.all_to_all_single(out, src.cpu().contiguous(), list(recv_sizes), list(send_sizes), group=self.group)
            dst.copy_(out)
        else:
            self.dist.all_to_all_single(dst, src, list(recv_sizes), list(send_sizes), group=self.group)

    def allreduce_sum(self, t):
        if self._staged(t):
            c = t.cpu()
            self.dist.all_reduce(c, op=self.dist.ReduceOp.SUM, group=self.group)
            t.copy_(c)
        else:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t


class PeerLink:
    """The ranks' exchange buffers, mapped into this process through CUDA IPC (one process per GPU on one node;
    NVLink peer access is enabled lazily by the driver).  Built collectively: every rank must construct it."""

    def __init__(self, comm, lib, device):
        """Collective and exception-free: every rank runs the same two all-gathers whatever fails locally;
        ``self.ok`` says whether ALL ranks mapped ALL buffers (otherwise nobody may use the link)."""
        import torch
        self.lib, self.rank, self.world = lib, comm.rank, comm.world
        self._own, self._opened, self.error = None, [], None
        self.ptrs = (C.c_void_p * self.world)()
        handle = C.create_string_buffer(64)
        try:
            own = C.c_void_p()
            _lib.check(lib.obe_peer_alloc(C.byref(own), handle))
            self._own = own
        except Exception as exc:              # noqa: BLE001
            self.error = exc
        mine = torch.tensor(list(handle.raw), dtype=torch.uint8, device=device)
        handles = comm.allgather(mine).cpu().numpy()
        if self.error is None:
            try:
                for g in range(self.world):
                    if g == self.rank:
                        self.ptrs[g] = self._own.value
                    else:
                        p = C.c_void_p()
                        _lib.check(lib.obe_peer_open(bytes(bytearray(handles[g].tolist())), C.byref(p)))
                        self.ptrs[g] = p.value
                        self._opened.append(p)
            except Exception as exc:          # noqa: BLE001
                self.error = exc
        good = comm.allgather(torch.tensor([1.0 if self.error is None else 0.0], dtype=torch.float64, device=device))
        self.ok = bool((good > 0.5).all().item())      # also the barrier: everybody has mapped everybody
        self.epoch = [0, 0]            # stats exchanges, draw exchanges

    def next_epoch(self, kind):
        self.epoch[kind] += 1
        return self.epoch[kind]

    def close(self):
        for p in self._opened:
            self.lib.obe_peer_close(p)
        self._opened = []
        if self._own is not None:
            self.lib.obe_peer_free(self._own)
            self._own = None


# --------------------------------------------------------------------------------------------------
def gstats_from_plan(plan_host, d, world):
    """The combined-stats dict (same keys as combine_stats) from a fetched plan block."""
    g = plan_host[_lib.PLAN_GSTATS:_lib.PLAN_GSTATS + _lib.STATS_LEN]
    nm2 = d * (d + 1) // 2
    return dict(totals=plan_host[160:160 + world].copy(), offsets=plan_host[96:96 + world].copy(),
                total=float(g[_lib.ST_TOTAL]), sumsq=float(g[_lib.ST_SUMSQ]), sumt=float(g[_lib.ST_SUMT]),
                m1=g[_lib.ST_M1:_lib.ST_M1 + d].copy(), m2=g[_lib.ST_M2:_lib.ST_M2 + nm2].copy(),
                noise=g[_lib.ST_NOISE:_lib.ST_NOISE + 4].copy(), pivot=g[_lib.ST_PIVOT:_lib.ST_PIVOT + d].copy())


_SUMMARY_REFUSAL = ('{} of a sharded cloud is not implemented yet (it needs an all-reduce of the fixed-point bins '
                    'across shards); gather the cloud or use an unsharded engine')


class ShardedOptBayesExpt(OptBayesExpt):
    """OptBayesExpt over a cloud sharded across the ranks of a process group.

    ``parameter_samples`` is THIS rank's shard (d, n_local); ``setting_values`` is the full grid on
    every rank.  All ranks must pass the same ``seed`` (the comb offset u0 and the K uniforms are
    drawn from identically seeded Generators so that every rank takes the same decisions).

    After every update the stats blocks are all-gathered and ``k_shard_plan`` turns them, on the
    device, into the shard plan (global normaliser and moments, Cholesky factor, CDF offsets, comb
    slot bounds of every shard): ``run_cycle_async`` enqueues update -> all-gather -> plan ->
    resample -> draws -> all-reduce -> utility with no host synchronisation at all; the
    reference-shaped ``pdf_update``/``opt_setting`` fetch the plan block only to take the
    resample decision and to return the argmax."""

    _drift_refusal = ('ShardedOptBayesExpt does not take drift: its normals would have to be keyed by the global '
                      'particle slot to keep the cloud independent of the number of ranks')

    def __init__(self, measurement_model, setting_values, parameter_samples, constants, group=None,
                 slack=0.25, seed=0, peer_exchange=None, **kwargs):
        import torch
        if kwargs.get('drift') is not None:           # (before the process group is touched)
            raise ValueError(self._drift_refusal)
        if non_gaussian(measurement_model, kwargs.get('likelihood_model')):
            raise ValueError('ShardedOptBayesExpt supports the Gaussian likelihood only; use OptBayesExpt for '
                             'likelihood_model=\'poisson\' | \'binomial\' | cuda_likelihood(...)')
        self._comm = Comm(group)
        if peer_exchange is None:
            # default: on for a real multi-GPU job (nccl backend), off otherwise; OBE_PEER_EXCHANGE=0/1 overrides
            default = '1' if (self._comm.backend == 'nccl' and self._comm.world > 1) else PEER_EXCHANGE_DEFAULT
            peer_exchange = os.environ.get('OBE_PEER_EXCHANGE', default) == '1'
        self._want_peer = bool(peer_exchange)
        self._peer = None
        kwargs['resampling'] = 'systematic'
        kwargs['seed'] = seed
        n_local = parameter_samples.shape[-1]
        self._capacity = int(n_local * (1.0 + slack)) + 2 * _lib.TILE     # shard lengths float
        self._gstats = None
        self._plan_valid = False
        self._n_local = None
        OptBayesExpt.__init__(self, measurement_model, setting_values, parameter_samples, constants, **kwargs)
        dev = self._buf.device
        self._buf.enable_device_count()
        self._alt = self._buf.empty_like()
        counts = self._comm.allgather(torch.tensor([self._n_local], dtype=torch.int64, device=dev))
        self.n_total = int(counts.sum().item())
        self._caps = self._comm.allgather(torch.tensor([self._buf.ld], dtype=torch.int64, device=dev)).cpu().numpy().reshape(-1)
        self._plan = torch.zeros(_lib.PLAN_LEN, dtype=torch.float64, device=dev)
        self._check(self._lib.obe_set_uniform_total(self._cs(), self.n_total, self._stream()))
        n_set = len(self.setting_indices)
        # The utility kernel is latency-bound (one thread per setting, ~30 us) up to ~1e5 settings: below that
        # every rank evaluates the whole grid -- same draws, same settings, so the same argmax everywhere --
        # and the selection needs no collective at all.  Larger grids are sliced over the ranks.
        self._replicate_grid = n_set <= REPLICATE_GRID_MAX
        if self._replicate_grid:
            self._s_lo, self._s_hi = 0, n_set
        else:
            self._s_lo, self._s_hi = setting_slice(n_set, self._comm.rank, self._comm.world)
        piv = torch.from_numpy(self._pivot.copy()).to(dev)     # a common pivot: rank 0's estimate
        self._pivot = self._comm.allgather(piv)[0].cpu().numpy()
        self._section = 0          # 0: draw with the plan's current-weight totals, 1: post-resample
        if self._want_peer and self._comm.world <= 16:
            # collective and all-or-nothing: if the IPC mapping fails on any rank, every rank stays on NCCL
            link = PeerLink(self._comm, self._lib, dev)
            if link.ok:
                self._peer = link
            else:
                link.close()
                if self._comm.rank == 0:
                    import warnings
                    warnings.warn(f'peer exchange unavailable ({link.error}); using NCCL collectives', RuntimeWarning)
        self._make_plan()

    def close(self):
        """Unmap the peers' exchange buffers and free the local one.  Call it on every rank, after a barrier: a
        peer that is still running a cycle would store into freed memory.  (Not done implicitly on deletion for
        that reason; process exit releases everything.)"""
        if getattr(self, '_peer', None) is not None:
            self._torch.cuda.synchronize()
            self._peer.close()
            self._peer = None

    # ---- the live shard length lives on the device
    @property
    def n_particles(self):
        if self._n_local is None:
            self._n_local = int(self._buf.n_dev.item())
        return self._n_local

    @n_particles.setter
    def n_particles(self, value):
        self._n_local = int(value)

    def _invalidate(self, particles=False, weights=True):
        OptBayesExpt._invalidate(self, particles, weights)
        if weights:
            self._gstats = None
            self._plan_valid = False

    # ---- plan
    def _make_plan(self):
        """all-gather the stats blocks -> k_shard_plan (device).  Asynchronous."""
        self._u0 = float(self.rng.random())                 # identical on every rank
        if self._peer is not None:
            # stats exchange fused into the plan kernel: peer writes over NVLink + flags, no collective
            self._check(self._lib.obe_shard_plan_peer(
                self._peer.ptrs, self._comm.rank, self._comm.world, self._peer.next_epoch(0), self.n_dims, self._u0,
                self.n_total, float(self.tuning_parameters['a_param']), 1 if self._weights_lazy else 0,
                self._cs(), self._cs(self._alt), C.c_void_p(self._plan.data_ptr()), self._stream()))
            gathered = None
        else:
            gathered = self._comm.allgather(self._buf.stats)
            self._check(self._lib.obe_shard_plan(C.c_void_p(gathered.data_ptr()), self._comm.rank, self._comm.world,
                                                 self.n_dims, self._u0, self.n_total,
                                                 float(self.tuning_parameters['a_param']),
                                                 1 if self._weights_lazy else 0,
                                                 self._cs(), self._cs(self._alt), C.c_void_p(self._plan.data_ptr()),
                                                 self._stream()))
        self._keep = gathered
        self._plan_valid = True
        self._section = 0
        self._gstats = None

    def _fetch_plan(self):
        """Bring the plan block to the host (synchronises): global stats, counts, overflow flag."""
        if not self._plan_valid or not self._moments_valid:
            if not self._moments_valid:
                ni = self._noise_index
                self._check(self._lib.obe_refresh(self._cs(), 0, 0, _lib.iarr(ni), 0 if ni is None else len(ni),
                                                  _lib.darr(self._pivot, _lib.MAX_PARAMS), 0, self._stream()))
                self._moments_valid = True
            self._make_plan()
        if self._gstats is None:
            ph = self._plan.cpu().numpy()
            if ph[_lib.PLAN_OVERFLOW] == 2.0:
                raise RuntimeError('peer exchange timed out: a rank died or the ranks fell out of step')
            # (checked against every rank's capacity, so that all ranks raise together and nobody walks into the
            # next collective alone; the device-side word only knows the local buffer)
            counts = ph[_lib.PLAN_COUNTS:_lib.PLAN_COUNTS + self._comm.world]
            if ph[_lib.PLAN_OVERFLOW] != 0.0 or np.any(counts > self._caps):
                raise RuntimeError('a shard outgrew its buffer capacity in a resample; raise `slack` '
                                   '(or call rebalance() before the lengths drift that far)')
            self._plan_host = ph
            self._gstats = gstats_from_plan(ph, self.n_dims, self._comm.world)
            self._gmom = moments_from(self._gstats, self.n_dims)
            self._stats = ph[_lib.PLAN_GSTATS:_lib.PLAN_GSTATS + _lib.STATS_LEN].copy()
        return self._gstats

    def _after_update(self):
        self._invalidate()
        self._weights_uniform = False
        self._weights_lazy = True
        self._moments_valid = True
        self._make_plan()
        self._fetch_plan()
        self._pivot = self._gmom[0].copy()
        if self.tuning_parameters['auto_resample']:
            self.resample_test()

    def _ensure_moments(self):
        self._fetch_plan()
        return self._stats

    def mean(self):
        self._fetch_plan()
        return self._gmom[0].copy()

    def covariance(self):
        self._fetch_plan()
        return self._gmom[1].copy()

    def std(self):
        self._fetch_plan()
        return np.sqrt(np.maximum(self._gmom[2], 0.0))

    def n_eff(self):
        self._fetch_plan()
        return float(self._gmom[3])

    # The inherited summaries would answer for this rank's shard alone.  The sharded version is one integer
    # all-reduce of the fixed-point bins per pass (DESIGN.md §7); until it exists they refuse.
    def quantile(self, q, params=None):
        raise NotImplementedError(_SUMMARY_REFUSAL.format('quantile'))

    def histogram(self, bins, range=None, params=None, return_counts=False):
        raise NotImplementedError(_SUMMARY_REFUSAL.format('histogram'))

    def histogram2d(self, i, j, bins, range=None, return_counts=False):
        raise NotImplementedError(_SUMMARY_REFUSAL.format('histogram2d'))

    def resample_test(self):
        import warnings
        n_eff = self.n_eff()
        if n_eff < 0.1 * self.n_total:
            warnings.warn(f"\nParticle filter rejected > 90 % of particles. N_eff = {n_eff:.2f}. "
                          "Particle impoverishment may lead to errors.", RuntimeWarning)
            self._do_resample()
            self.just_resampled = True
        elif n_eff / self.n_total < self.tuning_parameters['resample_threshold']:
            self._do_resample()
            self.just_resampled = True
        else:
            self.just_resampled = False

    # ---- resample: every shard keeps its own offspring; all parameters come from the device plan
    def resample(self):
        if not self._plan_valid or self._section != 0:
            self._plan_valid = False if self._section != 0 else self._plan_valid
            self._fetch_plan()
        self._epoch += 1
        self._check(self._lib.obe_resample_systematic_planned(
            self._cs(), self._cs(self._alt), C.c_void_p(self._plan.data_ptr()), self.n_total, self._philox_seed,
            self._epoch, float(self.tuning_parameters['a_param']), 1 if self.tuning_parameters['scale'] else 0,
            self._stream()))
        self._buf, self._alt = self._alt, self._buf
        self._cloud_version += 1
        self._n_local = None
        OptBayesExpt._invalidate(self, particles=True)
        self._gstats = None
        self._stats = None
        self._moments_valid = False
        self._weights_uniform = True
        self._weights_lazy = False
        self._section = 1           # the plan stays valid for draws: its post-resample totals apply

    # ---- rebalancing (SURVEY hard part 10): shard lengths drift by a fraction of a percent per resample
    def rebalance(self, force=False, threshold=0.9):
        """Equalise the shard lengths with one all-to-all-v per particle row.  Collective (every rank must call it) and
        synchronising.  Shards are contiguous pieces of the global cloud in rank order, so the cloud's order -- and
        with it every later result -- is unchanged; only the cut points move back to n_total*g/G.  Without ``force``
        nothing moves unless some shard has grown beyond ``threshold`` of its buffer capacity (the decision is taken
        from the all-gathered lengths and capacities, identically on every rank).  Returns True if particles moved.

        A SINGLE resample that concentrates more than the slack allows on one shard still overflows (the plan flags
        it and the next host look raises): counts can only be balanced after the offspring exist."""
        import torch
        comm, dev = self._comm, self._buf.device
        G, r = comm.world, comm.rank
        info = comm.allgather(torch.tensor([float(self.n_particles), float(self._buf.ld)], dtype=torch.float64,
                                           device=dev)).cpu().numpy()
        counts, caps = info[:, 0].astype(np.int64), info[:, 1].astype(np.int64)
        if not force and not np.any(counts > threshold * caps):
            return False
        n = int(counts.sum())
        starts = np.concatenate([[0], np.cumsum(counts)])
        targets = np.array([n * g // G for g in range(G + 1)], dtype=np.int64)
        if np.any(np.diff(targets) > caps):
            raise RuntimeError('rebalance: an equal share does not fit a shard buffer; raise `slack`')

        def overlap(a0, a1, b0, b1):
            return int(max(0, min(a1, b1) - max(a0, b0)))
        send = [overlap(starts[r], starts[r + 1], targets[p], targets[p + 1]) for p in range(G)]
        recv = [overlap(starts[p], starts[p + 1], targets[r], targets[r + 1]) for p in range(G)]
        c_old, c_new = int(counts[r]), int(targets[r + 1] - targets[r])
        uniform = bool(self._weights_uniform)
        if not uniform:
            self._check(self._lib.obe_materialize_weights(self._cs(), self._stream()))
        torch.cuda.synchronize()
        for j in range(self.n_dims):
            comm.alltoall_rows(self._alt.particles[j, :c_new], self._buf.particles[j, :c_old], recv, send)
        if not uniform:
            comm.alltoall_rows(self._alt.weights[:c_new], self._buf.weights[:c_old], recv, send)
            self._alt.stats.copy_(self._buf.stats)             # the normaliser INVS travels with the weights
        self._buf, self._alt = self._alt, self._buf
        self._buf.n_dev.fill_(c_new)
        self._alt.n_dev.fill_(c_new)
        self._n_local = c_new
        self._cloud_version += 1
        OptBayesExpt._invalidate(self, particles=True)
        self._stats = None
        if uniform:
            self._check(self._lib.obe_set_uniform_total(self._cs(), self.n_total, self._stream()))
            self._weights_lazy = False
            self._moments_valid = False
        else:
            ni = self._noise_index
            self._check(self._lib.obe_refresh(self._cs(), 0, 0, _lib.iarr(ni), 0 if ni is None else len(ni),
                                              _lib.darr(self._pivot, _lib.MAX_PARAMS), 0, self._stream()))
            self._moments_valid = True
        self._gstats = None
        self._plan_valid = False
        self._make_plan()
        return True

    @property
    def shard_counts(self):
        """Lengths of all shards (synchronises)."""
        import torch
        return self._comm.allgather(self._buf.n_dev).cpu().numpy().reshape(-1)

    # ---- K draws through the sharded CDF: owners write, everyone else adds zeros
    def _randdraw_dev(self, n_draws):
        import torch
        if not self._plan_valid:
            self._fetch_plan()
        u = self.rng.random(n_draws)                        # identical on every rank
        draws = torch.empty((self.n_dims, n_draws), dtype=torch.float64, device=self._buf.device)
        if self._peer is not None and n_draws <= 128 and n_draws * self.n_dims <= 1024:
            # owners write their draws into every rank's buffer; one small kernel waits and collects
            self._check(self._lib.obe_draw_planned_peer(
                self._cs(), _lib.dptr(u), int(n_draws), self._peer.ptrs, self._comm.rank, self._comm.world,
                self._peer.next_epoch(1), C.c_void_p(self._plan.data_ptr()), self._section,
                C.c_void_p(draws.data_ptr()), self._stream()))
            return draws
        self._check(self._lib.obe_draw_planned(self._cs(), _lib.dptr(u), int(n_draws), C.c_void_p(draws.data_ptr()),
                                               C.c_void_p(self._plan.data_ptr()), self._section, self._stream()))
        self._comm.allreduce_sum(draws)
        return draws

    def _pick_draws(self, u, draws, side_raw):
        """Early select over the sharded cloud: every rank produces the offspring it owns.  Peer mode: the owners store
        into every rank's buffer and a one-CTA kernel collects; collective mode: zeros elsewhere + all-reduce, both on
        the selection stream."""
        if self._peer is not None and len(u) * self.n_dims <= 1024:
            self._check(self._lib.obe_resample_pick(_lib.dptr(u), int(len(u)), C.c_void_p(draws.data_ptr()),
                                                    self._peer.ptrs, self._comm.rank, self._comm.world,
                                                    self._peer.next_epoch(1), side_raw))
            return
        self._check(self._lib.obe_resample_pick(_lib.dptr(u), int(len(u)), C.c_void_p(draws.data_ptr()), None, 0, 0, 0,
                                                side_raw))
        with self._torch.cuda.stream(self._side_stream()[0]):
            self._comm.allreduce_sum(draws)

    # ---- utility over this rank's slice of the grid
    def _utility_dev_run(self, draws=None, side=None):
        if draws is None:
            draws = self._randdraw_dev(self.N_DRAWS)
        n_loc = self._s_hi - self._s_lo
        stats_ptr = None
        if self._noise_from_stats():
            # weighted mean of sigma^2 from the GLOBAL noise sums the shard plan combined (no host round-trip)
            if not self._plan_valid or self._section != 0:
                self._fetch_plan()
            var_noise = None
            stats_ptr = C.c_void_p(self._plan.data_ptr() + 8 * _lib.PLAN_GSTATS)
        else:
            var_noise = _lib.darr(np.asarray(self.yvar_noise_model(), dtype=np.float64).reshape(-1),
                                  _lib.MAX_CHANNELS)
        cost = self.cost_estimate()
        cost_ptr = None
        if not (np.isscalar(cost) and float(cost) == 1.0):
            import torch
            cost_arr = np.array(np.broadcast_to(np.asarray(cost, dtype=np.float64), (len(self.setting_indices),)))
            if side is not None:
                with torch.cuda.stream(side):
                    self._cost_dev = torch.from_numpy(cost_arr[self._s_lo:self._s_hi].copy()).to(self._buf.device)
            else:
                self._cost_dev = torch.from_numpy(cost_arr[self._s_lo:self._s_hi].copy()).to(self._buf.device)
            cost_ptr = C.c_void_p(self._cost_dev.data_ptr())
        settings_ptr = C.c_void_p(self._settings_dev.data_ptr() + 8 * self._s_lo)
        util_ptr = C.c_void_p(self._utility_dev.data_ptr() + 8 * self._s_lo)
        self._check(self._lib.obe_utility(self._model, C.c_void_p(draws.data_ptr()), int(self.N_DRAWS), settings_ptr,
                                          self._lds, n_loc, self._cons_arr, var_noise, stats_ptr, cost_ptr,
                                          self._utility_code, 1 if self.utility_log_form else 0,
                                          self._kld_noise_ptr(), util_ptr,
                                          C.c_void_p(self._best_dev.data_ptr()),
                                          C.c_void_p(self._select_scratch.data_ptr()), self._stream()))

    def _kld_noise_ptr(self):
        # every rank must add the same noise: draw it from the instance Generator (identically seeded)
        from . import obe_base
        saved, obe_base.rng = obe_base.rng, self.rng
        try:
            return OptBayesExpt._kld_noise_ptr(self)
        finally:
            obe_base.rng = saved

    def opt_setting(self):
        import torch
        if self._select_ready:
            self._select_ready = False
        else:
            self._utility_dev_run()
            self._best_copied = False
        if self._replicate_grid:
            if self._best_copied:               # the cycle entry delivers the argmax into the pinned block
                self._best_copied = False
                self._wait_cycle()
                best = int(self._cy_best_np[0])
            else:
                self._best_host.copy_(self._best_dev, non_blocking=True)
                self._check(self._lib.obe_stream_sync(self._stream()))
                best = int(self._best_host_np[0])
            self.last_setting_index = best
            return tuple(self.allsettings[:, best])
        self._best_copied = False
        pairs = self._comm.allgather(self._best_dev).cpu()
        vals = pairs[:, 1].contiguous().view(torch.float64).numpy()
        idxs = pairs[:, 0].numpy()
        lows = [setting_slice(len(self.setting_indices), r, self._comm.world)[0] for r in range(self._comm.world)]
        best, _ = reduce_best([(int(idxs[r]) + lows[r] if idxs[r] >= 0 else -1, float(vals[r]))
                               for r in range(self._comm.world)])
        self.last_setting_index = best
        return tuple(self.allsettings[:, best])

    def utility(self):
        import torch
        if self._select_ready:
            self._select_ready = False
        else:
            self._utility_dev_run()
        n_set = len(self.setting_indices)
        world = self._comm.world
        if self._replicate_grid:
            return self._utility_dev[:n_set].cpu().numpy()
        width = max(setting_slice(n_set, r, world)[1] - setting_slice(n_set, r, world)[0] for r in range(world))
        buf = torch.zeros(width, dtype=torch.float64, device=self._buf.device)
        buf[:self._s_hi - self._s_lo] = self._utility_dev[self._s_lo:self._s_hi]
        allu = self._comm.allgather(buf).cpu().numpy()
        out = np.empty(n_set)
        for r in range(world):
            lo, hi = setting_slice(n_set, r, world)
            out[lo:hi] = allu[r, :hi - lo]
        return out

    def random_setting(self):
        """Uniformly random setting (obe_base.py:791-805), drawn from the instance Generator: identically seeded on
        every rank, so all ranks measure at the same setting (the module-level Generator of the base class is not)."""
        settingindex = int(self.rng.choice(self.setting_indices))
        self.last_setting_index = settingindex
        return self.allsettings[:, settingindex]

    def good_setting(self, pickiness=None):
        import torch
        if pickiness is None:
            pickiness = self.pickiness
        full = torch.from_numpy(self.utility()).to(self._buf.device)
        self._utility_dev.copy_(full)
        u = float(self.rng.random())
        self._check(self._lib.obe_pick(C.c_void_p(self._utility_dev.data_ptr()), len(self.setting_indices),
                                       float(pickiness), u, C.c_void_p(self._pick_dev.data_ptr()),
                                       C.c_void_p(self._select_scratch.data_ptr()), self._stream()))
        goodindex = int(self._pick_dev.item())
        self.last_setting_index = goodindex
        return tuple(self.allsettings[:, goodindex])

    def _apply_constraint_masks(self, mask_le=0, mask_lt=0):
        """weight <- 0 where the masked parameters are not positive, on every shard, then a new plan (global
        normaliser and noise sums of the constrained cloud)."""
        ni = self._noise_index
        self._check(self._lib.obe_refresh(self._cs(), mask_le, mask_lt, _lib.iarr(ni), 0 if ni is None else len(ni),
                                          _lib.darr(self._pivot, _lib.MAX_PARAMS), 1, self._stream()))
        self._invalidate()
        self._weights_uniform = False
        self._weights_lazy = True
        self._moments_valid = True
        self._make_plan()

    def run_cycle_async(self, measurement_record, resample=True, select=True):
        """Sharded cycle with NO host synchronisation: update -> all-gather(stats) -> device plan ->
        planned resample -> owner-written draws -> all-reduce -> utility over this rank's grid slice."""
        if (resample and self._peer is not None and self._replicate_grid and self._cycle_c_ok(resample, select)
                and not self._noise_from_stats() and self._constraint_masks() == (0, 0)
                and self.N_DRAWS * self.n_dims <= 1024):
            return self._run_cycle_c(measurement_record, resample, select)
        OptBayesExpt.run_cycle_async(self, measurement_record, resample=False, select=False)
        self._make_plan()
        self.resample_select_async(resample, select)

    def _async_stats_source(self, resample):
        return self._plan[_lib.PLAN_GSTATS:_lib.PLAN_GSTATS + _lib.STATS_LEN]      # the combined (global) block

    def _async_stats_ptr(self, resample):
        return self._plan.data_ptr() + 8 * _lib.PLAN_GSTATS

    def _device_test_ok(self):
        return False            # the resample test of a sharded cloud needs the combined stats of all ranks

    def _n_total_for_test(self):
        return self.n_total

    def _pdf_update_async(self, measurement_record, resample):
        if not resample:        # (the unsharded entry would skip the stats exchange: keep the synchronous path)
            self.async_update, saved = False, self.async_update
            try:
                return self.pdf_update(measurement_record)
            finally:
                self.async_update = saved
        return OptBayesExpt._pdf_update_async(self, measurement_record, resample)

    def _run_cycle_c(self, measurement_record, resample, select):
        """The sharded cycle through obe_cycle: update -> stats exchange + shard plan -> plan -> [pick + exchange of the
        draws + utility] || [streaming resample], one C call.  Also used for the bare update (resample=select=False)
        by the step-wise path, where it is the single-cloud entry."""
        if not resample:
            return OptBayesExpt._run_cycle_c(self, measurement_record, resample, select)
        cy = self._cycle_struct()
        self._fill_cycle_update(cy, measurement_record, resample)
        if self.split_cycle:                                # the update kernel first, the rest of the struct while it runs
            cy.phase = 1
            self._check(self._lib.obe_cycle(C.byref(cy)))
            cy.phase = 2
        self._fill_cycle_rest(cy, resample, select)
        self._u0 = float(self.rng.random())                 # identical on every rank
        cy.u0 = self._u0
        cy.plan_dev = self._plan.data_ptr()
        cy.peer_bufs = C.cast(self._peer.ptrs, C.POINTER(C.c_void_p))
        cy.rank, cy.world = self._comm.rank, self._comm.world
        cy.epoch_stats = self._peer.next_epoch(0)
        cy.n_total = self.n_total
        if select:
            cy.epoch_draws = self._peer.next_epoch(1)
            self._cy_u[:cy.k] = self.rng.random(cy.k)
        try:
            self._check(self._lib.obe_cycle(C.byref(cy)))
        finally:
            cy.plan_dev = None                              # the bare-update use of the struct is unsharded
        # host bookkeeping of the update, _make_plan() and resample()
        OptBayesExpt._invalidate(self)
        self._keep = None
        self._epoch += 1
        self._buf, self._alt = self._alt, self._buf
        self._cloud_version += 1
        self._n_local = None
        OptBayesExpt._invalidate(self, particles=True)
        self._gstats = None
        self._stats = None
        self._plan_valid = True
        self._moments_valid = False
        self._weights_uniform = True
        self._weights_lazy = False
        self._section = 1
        self.just_resampled = True

    def resample_select_async(self, resample=True, select=True):
        if resample and select and self._early_select_ok():
            self._resample_with_select()
            self._select_ready = False
            self.just_resampled = True
            return
        if resample:
            self.resample()
            self.just_resampled = True
            self.enforce_parameter_constraints()
        if select:
            self._utility_dev_run()


class ShardedOptBayesExptNoiseParameter(ShardedOptBayesExpt):
    """OptBayesExptNoiseParameter (obe_noiseparam.py) over a sharded cloud: sigma is a particle coordinate, the
    noise variance of the utility is the GLOBAL weighted mean of sigma^2 (combined in the shard plan), and the
    positivity constraint is applied on every shard after a resample."""

    def __init__(self, measurement_model, setting_values, parameter_samples, constants, noise_parameter_index=None,
                 **kwargs):
        ShardedOptBayesExpt.__init__(self, measurement_model, setting_values, parameter_samples, constants, **kwargs)
        idx = np.atleast_1d(noise_parameter_index)
        if noise_parameter_index is None or len(idx) != self.n_channels:
            raise RuntimeError(f'noise_parameter_index is not compatible with {self.n_channels} measurement channels')
        self.noise_parameter_index = idx.astype(int)
        self._noise_index = [int(i) for i in self.noise_parameter_index]
        # the noise sums were not part of the first stats pass
        self._moments_valid = False
        self._plan_valid = False
        self._fetch_plan()

    def _likelihood_spec(self, measurement_record):
        y_meas = np.atleast_1d(np.asarray(measurement_record[1], dtype=np.float64))
        n_lik = min(self.n_channels, len(y_meas))
        return y_meas[:n_lik], None, self._noise_index[:n_lik], n_lik

    def _noise_from_stats(self):
        return True

    def enforce_parameter_constraints(self):
        mask = 0
        for i in self._noise_index:
            mask |= 1 << i
        self._apply_constraint_masks(mask_le=mask)

    def yvar_noise_model(self):
        gs = self._fetch_plan()
        c = self.n_channels
        return (gs['noise'][:c] / gs['sumt']).reshape((c, 1))
