"""ParticlePDF with the cloud resident in HBM.

Mirror of the reference's ``optbayesexpt/particlepdf.py`` (v1.2.0): same constructor, methods,
attributes and error behaviour, but ``particles`` (d, N) and the weights live on the GPU as fp64
torch tensors and every O(N) step is a hand-written sm_100a kernel reached through the C ABI of
libobe_b200.so.  There is no CPU path.

Differences a user can see (all deliberate, see DESIGN.md):
  * ``particles`` / ``particle_weights`` return READ-ONLY numpy mirrors downloaded on demand
    (assign a new array to change them; in-place edits would silently miss the device copy, so
    they raise instead).  ``particles_dev`` / ``weights_dev`` give the torch tensors, zero-copy.
  * ``quantile`` / ``histogram`` / ``histogram2d`` summarise the posterior on the device
    (summaries.py); only their small results reach the host.
  * ``resampling='systematic'`` (default) uses the fused systematic-comb kernel with Philox
    normals on the device; ``resampling='multinomial'`` reproduces the reference's
    ``Generator.choice`` + ``multivariate_normal`` exactly, consuming ``self.rng`` in the same
    order (N uniforms, then N*d normals).
"""
import ctypes as C
import warnings

import numpy as np

from . import _lib
from .models import ParticleBuffers
from .summaries import SummaryMixin


class ParticlePDF(SummaryMixin):
    """Weighted-particle probability distribution (particlepdf.py:12-145)."""

    def __init__(self, prior, a_param=0.98, resample_threshold=0.5, auto_resample=True, scale=True,
                 use_jit=True, resampling='systematic', device=None, seed=None):
        import torch
        self._torch = torch
        self._lib = _lib.require_device()
        #: dict: resampling knobs, live-mutable as in the reference (particlepdf.py:96-99)
        self.tuning_parameters = {'a_param': a_param, 'resample_threshold': resample_threshold,
                                  'auto_resample': auto_resample, 'scale': scale}
        if resampling not in ('systematic', 'multinomial', 'multinomial_device'):
            raise ValueError("resampling must be 'systematic', 'multinomial' or 'multinomial_device'")
        self.resampling = resampling
        self.just_resampled = False
        try:
            self.rng = np.random.default_rng(seed)
        except AttributeError:  # pragma: no cover
            self.rng = np.random
        self._philox_seed = int(np.random.default_rng(seed).integers(0, 2 ** 63 - 1))
        self._epoch = 0
        self._cloud_version = 0        # bumped whenever the particle coordinates change
        self._device = device
        self._install(prior)
        self._check(self._lib.obe_set_uniform(self._cs(), self._stream()))
        self._weights_uniform = True

    # ------------------------------------------------------------------------------------------
    # plumbing
    # ------------------------------------------------------------------------------------------
    # A cycle whose resample test runs on the device (OptBayesExpt._pdf_update_device_test) leaves the outcome --
    # which of the two buffers holds the cloud -- unknown to the host until the stream has been synchronised.  Every
    # path to the cloud goes through ``_buf`` / ``_alt`` / ``just_resampled``: looking at any of them settles the
    # pending cycle first.
    _pending_cycle = False

    def _settle(self):
        """Nothing is pending on a plain ParticlePDF (OptBayesExpt overrides this)."""
        self._pending_cycle = False

    @property
    def _buf(self):
        if self._pending_cycle:
            self._settle()
        return self._buf_live

    @_buf.setter
    def _buf(self, value):
        self._buf_live = value

    @property
    def _alt(self):
        if self._pending_cycle:
            self._settle()
        return self._buf_alt

    @_alt.setter
    def _alt(self, value):
        self._buf_alt = value

    @property
    def just_resampled(self):
        """True if the last update resampled (particlepdf.py:120-126)."""
        if self._pending_cycle:
            self._settle()
        return self._just_resampled

    @just_resampled.setter
    def just_resampled(self, value):
        self._just_resampled = value

    def _install(self, samples):
        self._buf = ParticleBuffers(samples, self._device, capacity=getattr(self, '_capacity', None))
        self._dev_index = self._buf.device.index
        self._stream_override = None      # raw stream handle the C calls go to instead of torch's current stream
        self._alt = None
        self.n_particles = self._buf.n
        self.n_dims = self._buf.d
        self._particle_indices = np.arange(self.n_particles, dtype='int')
        self._host_particles = None
        self._host_weights = None
        self._stats = None          # host copy of the stats block, valid for the current cloud
        self._moments_valid = False
        self._noise_index = None    # set by OptBayesExptNoiseParameter
        self._weights_lazy = False  # True: device weights are un-normalised, INVS = 1/total
        # pivot for the shifted moment accumulators: a point near the mean
        p = self._buf.particles[:, :self.n_particles]
        self._pivot = p[:, :min(self.n_particles, 65536)].mean(dim=1).cpu().numpy().astype(np.float64)

    def _stream(self):
        over = self._stream_override
        if over is not None:
            return over
        return _lib.raw_stream(self._torch, self._dev_index)

    def _cs(self, buf=None):
        return C.byref((buf or self._buf).struct())

    @staticmethod
    def _check(rc):
        _lib.check(rc)

    def _invalidate(self, particles=False, weights=True):
        if particles:
            self._host_particles = None
        if weights:
            self._host_weights = None

    def _fetch_stats(self):
        pin = getattr(self, '_stats_pin', None)
        if pin is None:                       # pinned landing buffer: the D2H copy is a real async DMA
            pin = self._stats_pin = self._torch.zeros(_lib.STATS_LEN, dtype=self._torch.float64).pin_memory()
            self._stats_pin_np = pin.numpy()
            self._stats_pin_ptr = C.cast(pin.data_ptr(), C.POINTER(C.c_double))
        self._check(self._lib.obe_fetch_stats(self._cs(), self._stats_pin_ptr, self._stream()))
        self._stats = self._stats_pin_np.copy()
        return self._stats

    def _refresh(self, mask_le=0, mask_lt=0, renormalise=0):
        """Tile sums + CDF prefix + moments from the current device weights."""
        if self._pending_cycle:
            self._settle()
        ni = self._noise_index
        self._check(self._lib.obe_refresh(self._cs(), mask_le, mask_lt, _lib.iarr(ni),
                                          0 if ni is None else len(ni), _lib.darr(self._pivot, _lib.MAX_PARAMS),
                                          renormalise, self._stream()))
        st = self._fetch_stats()
        # a far-off pivot costs accuracy: redo once around the mean just found
        mean = self._mean_from(st)
        var = self._var_from(st)
        shift2 = (mean - self._pivot) ** 2
        self._pivot = mean
        if np.any(shift2 > 1e4 * np.maximum(var, 1e-300)):
            self._check(self._lib.obe_refresh(self._cs(), 0, 0, _lib.iarr(ni), 0 if ni is None else len(ni),
                                              _lib.darr(self._pivot, _lib.MAX_PARAMS),
                                              renormalise if not (mask_le | mask_lt) else 1, self._stream()))
            st = self._fetch_stats()
        self._moments_valid = True
        self._weights_uniform = False
        return st

    def _ensure_moments(self):
        if self._pending_cycle:
            self._settle()
        if not self._moments_valid or self._stats is None:
            self._refresh(renormalise=1 if self._weights_lazy else 0)
        return self._stats

    @staticmethod
    def _n_eff_from(st):
        # 1/sum(w^2) with w = t * INVS  (particlepdf.py:243-244)
        return 1.0 / (st[_lib.ST_SUMSQ] * st[_lib.ST_INVS] ** 2)

    def _mean_from(self, st):
        d = self.n_dims
        return st[_lib.ST_PIVOT:_lib.ST_PIVOT + d] + st[_lib.ST_M1:_lib.ST_M1 + d] / st[_lib.ST_SUMT]

    def _m2_matrix(self, st):
        d = self.n_dims
        m2 = np.zeros((d, d))
        q = _lib.ST_M2
        for j in range(d):
            for k in range(j, d):
                m2[j, k] = m2[k, j] = st[q]
                q += 1
        return m2

    def _var_from(self, st):
        d = self.n_dims
        s = st[_lib.ST_SUMT]
        m1 = st[_lib.ST_M1:_lib.ST_M1 + d] / s
        return np.diag(self._m2_matrix(st)) / s - m1 * m1

    # ------------------------------------------------------------------------------------------
    # numpy-facing state
    # ------------------------------------------------------------------------------------------
    @property
    def particles(self):
        """(n_dims, n_particles) float64, read-only host mirror (particlepdf.py:101-105)."""
        if self._pending_cycle:
            self._settle()
        if self._host_particles is None:
            arr = self._buf.particles[:, :self.n_particles].cpu().numpy()
            arr.setflags(write=False)
            self._host_particles = arr
        return self._host_particles

    @particles.setter
    def particles(self, value):
        if self._pending_cycle:
            self._settle()
        value = np.atleast_2d(np.asarray(value, dtype=np.float64))
        if value.shape != (self.n_dims, self.n_particles):
            raise ValueError('particles has the wrong shape; use set_pdf() to change the geometry')
        self._buf.particles[:, :self.n_particles].copy_(self._torch.from_numpy(np.ascontiguousarray(value)))
        self._host_particles = None
        self._moments_valid = False
        self._cloud_version = getattr(self, '_cloud_version', 0) + 1

    @property
    def particle_weights(self):
        """(n_particles,) normalised weights, read-only host mirror (particlepdf.py:119-121)."""
        if self._pending_cycle:
            self._settle()
        if self._host_weights is None:
            out = self._torch.empty(self.n_particles, dtype=self._torch.float64, device=self._buf.device)
            self._check(self._lib.obe_normalized_weights(self._cs(), C.c_void_p(out.data_ptr()), self._stream()))
            arr = out.cpu().numpy()
            arr.setflags(write=False)
            self._host_weights = arr
        return self._host_weights

    @particle_weights.setter
    def particle_weights(self, value):
        if self._pending_cycle:
            self._settle()
        # stored as given, like the reference (tests/test_particlepdf.py:128,142,149 assign directly)
        value = np.asarray(value, dtype=np.float64).reshape(-1)
        if value.shape[0] != self.n_particles:
            raise ValueError('Length of weights does not match the number of particles.')
        self._buf.weights[:self.n_particles].copy_(self._torch.from_numpy(np.ascontiguousarray(value)))
        self._buf.stats[62:63].zero_()          # OBE_ST_UNIFORM: the weight row is explicit
        self._host_weights = None
        self._stats = None
        self._moments_valid = False
        self._weights_lazy = False
        self._refresh(renormalise=0)

    @property
    def particles_dev(self):
        """torch view (n_dims, n_particles) of the device cloud, zero-copy."""
        if self._pending_cycle:
            self._settle()
        return self._buf.particles[:, :self.n_particles]

    @property
    def weights_dev(self):
        """torch view of the UN-normalised device weights; multiply by ``weight_scale``.  (After a
        systematic resample the weights are implicit on the device; this materialises them.)"""
        if self._pending_cycle:
            self._settle()
        self._check(self._lib.obe_materialize_weights(self._cs(), self._stream()))
        return self._buf.weights[:self.n_particles]

    @property
    def weight_scale(self):
        if self._pending_cycle:
            self._settle()
        return float(self._buf.stats[_lib.ST_INVS].item())

    def set_pdf(self, samples, weights=None):
        """Re-initialise the distribution (particlepdf.py:147-171)."""
        if self._pending_cycle:
            self._settle()
        self._install(samples)
        self._cloud_version = getattr(self, '_cloud_version', 0) + 1
        if weights is None:
            self._check(self._lib.obe_set_uniform(self._cs(), self._stream()))
            self._weights_uniform = True
        else:
            if len(weights) != self.n_particles:
                raise ValueError('Length of weights does not match the number of particles.')
            w = np.asarray(weights, dtype=np.float64)
            self.particle_weights = w / np.sum(w)

    # ------------------------------------------------------------------------------------------
    # moments (particlepdf.py:173-214)
    # ------------------------------------------------------------------------------------------
    def mean(self):
        """Weighted mean, size n_dims (particlepdf.py:182-183)."""
        if self._pending_cycle:
            self._settle()
        return self._mean_from(self._ensure_moments()).copy()

    def covariance(self):
        """np.cov(particles, aweights=w): (n_dims, n_dims) (particlepdf.py:194-198)."""
        if self._pending_cycle:
            self._settle()
        st = self._ensure_moments()
        d = self.n_dims
        s = st[_lib.ST_SUMT]
        m1 = st[_lib.ST_M1:_lib.ST_M1 + d]
        cov = (self._m2_matrix(st) - np.outer(m1, m1) / s) / (s - st[_lib.ST_SUMSQ] / s)
        return cov.reshape((d, d))

    def std(self):
        """sqrt(sum w x^2 - (sum w x)^2) per parameter (particlepdf.py:209-214); evaluated from the
        pivot-shifted accumulators, so without the reference's cancellation error."""
        if self._pending_cycle:
            self._settle()
        return np.sqrt(np.maximum(self._var_from(self._ensure_moments()), 0.0))

    def n_eff(self):
        if self._pending_cycle:
            self._settle()
        return float(self._n_eff_from(self._ensure_moments()))

    # ------------------------------------------------------------------------------------------
    # inference (particlepdf.py:216-258)
    # ------------------------------------------------------------------------------------------
    def bayesian_update(self, likelihood):
        """weights <- normalised(weights * likelihood), then the resample test."""
        if self._pending_cycle:
            self._settle()
        lik = np.asarray(likelihood, dtype=np.float64).reshape(-1)
        if lik.shape[0] != self.n_particles:
            raise ValueError('likelihood length does not match the number of particles')
        ldev = self._torch.zeros(self._buf.ld, dtype=self._torch.float64, device=self._buf.device)
        ldev[:self.n_particles].copy_(self._torch.from_numpy(np.ascontiguousarray(lik)))
        self._check(self._lib.obe_update_from_likelihood(self._cs(), C.c_void_p(ldev.data_ptr()),
                                                         _lib.darr(self._pivot, _lib.MAX_PARAMS), self._stream()))
        self._after_update()

    def _after_update(self):
        self._invalidate()
        self._weights_uniform = False
        self._weights_lazy = True
        st = self._fetch_stats()
        self._moments_valid = True
        self._pivot = self._mean_from(st)
        if self.tuning_parameters['auto_resample']:
            self.resample_test()

    def resample_test(self):
        """Resample if N_eff/N is below the threshold; sets just_resampled (particlepdf.py:236-258)."""
        if self._pending_cycle:
            self._settle()
        n_eff = self._n_eff_from(self._ensure_moments())
        if n_eff < 0.1 * self.n_particles:
            warnings.warn("\nParticle filter rejected > 90 % of particles. "
                          f"N_eff = {n_eff:.2f}. "
                          "Particle impoverishment may lead to errors.", RuntimeWarning)
            self._do_resample()
            self.just_resampled = True
        elif n_eff / self.n_particles < self.tuning_parameters['resample_threshold']:
            self._do_resample()
            self.just_resampled = True
        else:
            self.just_resampled = False

    def _do_resample(self):
        """The resample the test decided on (a hook: OptBayesExpt may start the selection with it)."""
        self.resample()

    # ------------------------------------------------------------------------------------------
    # resampling (particlepdf.py:260-345)
    # ------------------------------------------------------------------------------------------
    def resample(self):
        """Weighted re-draw of the cloud + Liu-West jitter (particlepdf.py:260-310)."""
        if self._pending_cycle:
            self._settle()
        torch = self._torch
        if self._alt is None:
            self._alt = self._buf.empty_like()
        a_param = float(self.tuning_parameters['a_param'])
        scale = 1 if self.tuning_parameters['scale'] else 0
        n, d = self.n_particles, self.n_dims
        self._epoch += 1
        if self.resampling == 'multinomial':
            # the reference's order of Generator consumption: N uniforms, [cov, mean], N*d normals
            u = torch.from_numpy(self.rng.random(n)).to(self._buf.device)
            covar = self.covariance()
            center = self.mean()
            newcovar = (1 - a_param ** 2) * covar
            # Generator.multivariate_normal(method='svd'): x = z @ (u * sqrt(s)).T
            (uu, ss, _) = np.linalg.svd(newcovar)
            factor = np.ascontiguousarray((uu * np.sqrt(ss)).T)
            z = torch.from_numpy(self.rng.standard_normal(n * d)).to(self._buf.device)
            cdf = torch.empty(n, dtype=torch.float64, device=self._buf.device)
            idx = torch.empty(n, dtype=torch.int64, device=self._buf.device)
            self._check(self._lib.obe_cdf(self._cs(), C.c_void_p(cdf.data_ptr()), self._stream()))
            self._check(self._lib.obe_search(self._cs(), C.c_void_p(cdf.data_ptr()), C.c_void_p(u.data_ptr()),
                                             n, C.c_void_p(idx.data_ptr()), self._stream()))
            self._check(self._lib.obe_gather_jitter(self._cs(), self._cs(self._alt), C.c_void_p(idx.data_ptr()),
                                                    _lib.darr(factor.reshape(-1)), _lib.darr(center),
                                                    C.c_void_p(z.data_ptr()), 0, 0, a_param, scale, self._stream()))
            self._last_ancestors = idx
        elif self.resampling == 'multinomial_device':
            # the reference's ALGORITHM (N i.i.d. uniforms -> cumsum/searchsorted -> gather -> jitter,
            # particlepdf.py:286-310) with the randomness made on the device: uniforms from torch's CUDA
            # generator, normals from the Philox stream, Cholesky factor from the device moments.  No host
            # round trip; this is the like-for-like arm of the bench (same algorithm as the CPU reference).
            if not self._moments_valid:
                self._ensure_moments()
            gen = getattr(self, '_torch_gen', None)
            if gen is None:
                gen = self._torch_gen = torch.Generator(device=self._buf.device)
                gen.manual_seed(self._philox_seed & 0x7fffffffffffffff)
            mb = getattr(self, '_multinomial_bufs', None)
            if mb is None or mb[0].numel() != n:
                mb = self._multinomial_bufs = (torch.empty(n, dtype=torch.float64, device=self._buf.device),
                                               torch.empty(n, dtype=torch.float64, device=self._buf.device),
                                               torch.empty(n, dtype=torch.int64, device=self._buf.device))
            u, cdf, idx = mb
            torch.rand(n, generator=gen, dtype=torch.float64, device=self._buf.device, out=u)
            self._check(self._lib.obe_cdf(self._cs(), C.c_void_p(cdf.data_ptr()), self._stream()))
            self._check(self._lib.obe_search(self._cs(), C.c_void_p(cdf.data_ptr()), C.c_void_p(u.data_ptr()),
                                             n, C.c_void_p(idx.data_ptr()), self._stream()))
            self._check(self._lib.obe_gather_jitter(self._cs(), self._cs(self._alt), C.c_void_p(idx.data_ptr()),
                                                    None, None, None, self._philox_seed, self._epoch, a_param, scale,
                                                    self._stream()))
            self._last_ancestors = idx
        else:
            if not self._moments_valid:
                self._ensure_moments()
            u0 = float(self.rng.random())
            self._check(self._lib.obe_resample_systematic(self._cs(), self._cs(self._alt), u0, None, None,
                                                          self._philox_seed, self._epoch, a_param, scale,
                                                          None, None, self._stream()))
            self._last_ancestors = None
        self._buf, self._alt = self._alt, self._buf
        self._cloud_version += 1
        self._invalidate(particles=True)
        self._stats = None
        self._moments_valid = False
        self._weights_uniform = True
        self._weights_lazy = False

    def randdraw(self, n_draws=1):
        """(n_dims, n_draws) weighted random draws (particlepdf.py:312-345)."""
        if self._pending_cycle:
            self._settle()
        return self._randdraw_dev(n_draws).cpu().numpy()

    def _randdraw_dev(self, n_draws, out=None):
        if self._pending_cycle:
            self._settle()
        u = self.rng.random(n_draws)
        draws = out if out is not None else self._torch.empty((self.n_dims, n_draws), dtype=self._torch.float64,
                                                               device=self._buf.device)
        self._check(self._lib.obe_draw(self._cs(), _lib.dptr(u), int(n_draws), C.c_void_p(draws.data_ptr()),
                                       None, self._stream()))
        return draws

    @staticmethod
    def _normalized_product(weight_array, likelihood_array):
        """Kept for API parity (particlepdf.py:347-360); the device path is obe_update*."""
        raise NotImplementedError('the normalised product runs inside the fused update kernel')
