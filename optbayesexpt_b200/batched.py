"""B independent OptBayesExpt engines as ONE batched engine (BASELINE config c5: 4096 lock-in
instances x 1e4 particles).  The reference's idiom for this is ``multiprocessing.Pool.map`` over
independent runs (demos/fit_vs_obe/fit_vs_obe_makedata.py:319-321); here every phase of the cycle is
one launch over all instances and the whole closed loop stays on the device:

    idx = beng.opt_setting()        # K draws + utility + argmax of every instance   (obe_base.py:733-756)
    beng.pdf_update(y)              # fused update with each instance's own record   (obe_base.py:340-399)
                                    # + systematic resample of the instances that need it

Same model functors, same kernels' arithmetic, same constraint/cost/noise-parameter options as the
single engines; instance b reproduces a single engine that is fed the same uniforms
(tests/test_gpu_batched.py).

``drift`` gives every instance time-varying parameters, as ``OptBayesExpt(drift=...)`` does: at the end of every
update each particle takes a Gaussian random-walk step ``x <- x + F z`` with ``F F^T = Q`` (``optbayesexpt_b200.drift``).
``set_simulator(..., drift=...)`` lets the simulated experiment's true parameters take the same kind of step after
every simulated measurement, so a closed loop of drifting instruments runs on the device.

``likelihood_model``, ``design_noise`` and ``design_aux`` mean what they mean for ``OptBayesExpt``: the update of every
instance uses a Poisson, binomial or ``cuda_likelihood`` measurement likelihood, and ``design_noise='likelihood'``
divides each instance's utility by the likelihood's own noise variance.  ``set_simulator`` then draws counts on the
device (Poisson, or binomial with ``trials``), so a design study of counting measurements runs thousands of seeds in
one closed loop::

    beng = BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 241),), priors, (0.3,),
                               likelihood_model='poisson', design_noise='likelihood')
    beng.set_simulator(truths)                       # (B, 3) true parameters; counts ~ Poisson(model)
    for _ in range(150):
        beng.closed_loop_cycle()                     # no host round trip
"""
import ctypes as C

import numpy as np

from . import _lib
from .drift import batched_drift_factors
from .models import DeviceModel, builtin
from .obe_base import design_aux_array, resolve_likelihood


class BatchedOptBayesExpt:
    """``drift``: the random-walk step every instance's cloud takes at the end of every update (after the resample
    of the instances that resampled), or None (the default: static parameters).  It takes every form of
    ``OptBayesExpt``'s ``drift`` -- a standard deviation, ``n_dims`` of them or an ``(n_dims, n_dims)`` covariance
    ``Q`` -- applied to all instances, or an ``(n_instances, n_dims, n_dims)`` array with one covariance per instance
    (per-instance standard deviations as diagonal covariances).  It is also a property: ``beng.drift = Q * dt`` takes
    effect at the next update, in stream order and without a host synchronisation; ``beng.drift = None`` stops the
    steps.  The weights are never changed, and a step that would leave the region of the constraint masks (such as
    a positive noise parameter) is not taken.  The summaries and the next design therefore describe the parameters
    at the next measurement.  The normals are Philox normals keyed by the engine seed, the instance, the particle
    slot and the engine's count of drift steps, so no step reuses another's numbers.

    ``likelihood_model`` ('poisson', 'binomial' or a ``cuda_likelihood``; None keeps the model's own, Gaussian by
    default), ``design_noise`` ('fixed' or 'likelihood') and ``design_aux`` are ``OptBayesExpt``'s and apply to every
    instance: instance b reproduces a single ``OptBayesExpt`` with the same likelihood fed the same counts.  With a
    count likelihood ``pdf_update(counts, aux)`` takes the record's third element as its second argument (ignored for
    Poisson, the trials of a binomial, the aux of a ``cuda_likelihood``), a noise parameter is refused, and a binomial
    ``design_aux`` with ``design_noise='likelihood'`` must be an integer >= 1.  Only the variance utility is
    implemented for batched engines."""

    def __init__(self, measurement_model, setting_values, parameter_samples, constants, n_draws=30, choke=None,
                 default_noise_std=1.0, noise_parameter_index=None, constraint_le=(), constraint_lt=(),
                 cost_of_changing_setting=None, a_param=0.98, resample_threshold=0.5, auto_resample=True,
                 scale=True, seed=0, utility_method='variance_approx', device=None, drift=None, likelihood_model=None,
                 design_noise='fixed', design_aux=1):
        import torch
        self._torch = torch
        shape = tuple(parameter_samples.shape) if hasattr(parameter_samples, 'shape') else np.shape(parameter_samples)
        # (the cloud's shape, drift and the likelihood are checked before the device is)
        if len(shape) != 3:
            raise ValueError(f'parameter_samples must have shape (n_instances, n_dims, n_particles), got {shape}: every '
                             'instance has a cloud of its own, whatever its likelihood (Gaussian, Poisson, binomial '
                             'or cuda_likelihood); one (n_dims, n_particles) cloud is an OptBayesExpt')
        drift_factors = batched_drift_factors(drift, shape[0], shape[1])
        if isinstance(measurement_model, str):
            measurement_model = builtin(measurement_model)
        if not isinstance(measurement_model, DeviceModel):
            raise TypeError('measurement_model must be a DeviceModel; there is no CPU fallback')
        if utility_method not in ('variance_approx',):
            raise NotImplementedError('batched engines implement the variance utility')
        measurement_model, self._design_lik = resolve_likelihood(measurement_model, likelihood_model, design_noise,
                                                                 design_aux, utility_method)
        #: 'gaussian', 'poisson', 'binomial' or a CudaLikelihood
        self.likelihood_model = measurement_model.likelihood
        #: 'fixed' or 'likelihood': the noise variance of the utility
        self.design_noise = design_noise
        if self.likelihood_model != 'gaussian' and noise_parameter_index is not None:
            raise ValueError('a noise parameter is the sigma of the Gaussian likelihood: '
                             f'{type(self).__name__} takes no other likelihood_model')
        self.n_channels = measurement_model.n_channels
        self.design_aux = design_aux
        self._lib = _lib.require_device()
        self.model_function = measurement_model
        from .models import resolve_device
        dev = resolve_device(device)
        self._dev = dev
        if isinstance(parameter_samples, torch.Tensor):
            src = parameter_samples.to(dtype=torch.float64, device=dev)
        else:
            src = torch.from_numpy(np.ascontiguousarray(np.asarray(parameter_samples, dtype=np.float64))).to(dev)
        B, d, n = src.shape
        self.n_instances, self.n_dims, self.n_particles = int(B), int(d), int(n)
        T = (n + _lib.TILE - 1) // _lib.TILE
        if T > 64:
            raise ValueError('batched engines hold at most 64 tiles (131072 particles) per instance')
        self._tiles, self._np = T, T * _lib.TILE
        ld = B * self._np
        f64 = dict(dtype=torch.float64, device=dev)
        self._p = [torch.zeros((d, ld), **f64), torch.zeros((d, ld), **f64)]
        self._p[0].view(d, B, self._np)[:, :, :n].copy_(src.permute(1, 0, 2))
        self._w = [torch.zeros(ld, **f64), torch.zeros(ld, **f64)]
        self._cur = torch.zeros(B, dtype=torch.int32, device=dev)
        self._tile_sums = torch.zeros(B * T, **f64)
        self._prefix = torch.zeros(B * (T + 1), **f64)
        self._stats = torch.zeros((B, _lib.STATS_LEN), **f64)
        self._pivot = torch.zeros((B, 8), **f64)
        self._record = torch.zeros((B, 12), **f64)
        self._last_idx = torch.zeros(B, dtype=torch.int64, device=dev)
        self._best_val = torch.zeros(B, **f64)
        self._flag = torch.zeros(B, dtype=torch.int32, device=dev)
        self._list = torch.zeros(B, dtype=torch.int32, device=dev)
        self._n_list = torch.zeros(1, dtype=torch.int32, device=dev)
        self._epoch = torch.zeros(B, dtype=torch.int32, device=dev)
        self._batch = _lib.Batch((C.c_void_p * 2)(self._p[0].data_ptr(), self._p[1].data_ptr()),
                                 (C.c_void_p * 2)(self._w[0].data_ptr(), self._w[1].data_ptr()),
                                 self._cur.data_ptr(), self._tile_sums.data_ptr(), self._prefix.data_ptr(),
                                 self._stats.data_ptr(), self._pivot.data_ptr(), self._record.data_ptr(),
                                 self._last_idx.data_ptr(), self._best_val.data_ptr(), self._flag.data_ptr(),
                                 self._list.data_ptr(), self._n_list.data_ptr(), self._epoch.data_ptr(),
                                 B, n, self._np, ld, d, T)
        self._model = measurement_model.handle(d)
        # setting grid (obe_base.py:174-180)
        self.allsettings = np.array([s.flatten() for s in
                                     np.meshgrid(*[np.asarray(v, dtype=np.float64) for v in setting_values],
                                                 indexing='ij')])
        n_set = self.allsettings.shape[1]
        self.setting_indices = np.arange(n_set, dtype=int)
        self._lds = n_set + (n_set & 1)
        self._settings_dev = torch.zeros((self.allsettings.shape[0], self._lds), **f64)
        self._settings_dev[:, :n_set].copy_(torch.from_numpy(np.ascontiguousarray(self.allsettings)))
        self.cons = constants
        self._cons_arr = _lib.darr(list(constants)[:_lib.MAX_CONSTANTS], _lib.MAX_CONSTANTS)
        self.N_DRAWS = int(n_draws)
        self.choke = choke
        self.default_noise_std = np.ones((self.n_channels, 1)) * default_noise_std
        self.noise_parameter_index = None
        self._noise_index = None
        if noise_parameter_index is not None:
            idx = np.atleast_1d(noise_parameter_index).astype(int)
            if len(idx) != self.n_channels:
                raise RuntimeError(f'noise_parameter_index is not compatible with {self.n_channels} measurement channels')
            self.noise_parameter_index = idx
            self._noise_index = [int(i) for i in idx]
        self._mask_le = sum(1 << int(j) for j in constraint_le)
        self._mask_lt = sum(1 << int(j) for j in constraint_lt)
        if self._noise_index is not None and not (self._mask_le | self._mask_lt):
            self._mask_le = sum(1 << j for j in set(self._noise_index))       # obe_noiseparam.py:57-79
        self.cost_of_changing_setting = cost_of_changing_setting
        self.tuning_parameters = {'a_param': a_param, 'resample_threshold': resample_threshold,
                                  'auto_resample': auto_resample, 'scale': scale}
        self.utility_log_form = False
        self._seed_uniform = int(seed)
        self._seed_normal = int(np.random.default_rng(seed).integers(0, 2 ** 62))
        self.cycle = 0
        self._utility_dev = None
        self._check(self._lib.obe_batch_init(self._bs(), _lib.iarr(self._noise_index),
                                             0 if self._noise_index is None else len(self._noise_index),
                                             self._stream()))
        self._drift_step = 0              # drift steps taken: the step word of their normals
        self._install_drift(drift, drift_factors)

    # ---- plumbing
    def _stream(self):
        return _lib.raw_stream(self._torch)

    def _bs(self):
        return C.byref(self._batch)

    @staticmethod
    def _check(rc):
        _lib.check(rc)

    def _to_device(self, a):
        """A new float64 device tensor holding ``a``, copied in stream order without a host synchronisation."""
        host = self._torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).pin_memory()
        return host.to(self._dev, non_blocking=True)

    def _factor_args(self, factors):
        """(factor_host, factor_dev tensor) of the C drift entries: a shared F by value, per-instance F on the device."""
        if factors is None:
            return None, None
        if factors.ndim == 2:
            return _lib.darr(factors.reshape(-1)), None
        return None, self._to_device(factors)

    @staticmethod
    def _ptr(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    # ---- time-varying parameters
    @property
    def drift(self):
        """The random-walk step of every instance's cloud per update (see the class docstring), or None."""
        return self._drift

    @drift.setter
    def drift(self, value):
        self._install_drift(value, batched_drift_factors(value, self.n_instances, self.n_dims))

    def _install_drift(self, value, factors):
        self._drift = value
        self._drift_arr, self._drift_dev = self._factor_args(factors)

    def _apply_drift(self):
        """One random-walk step of every instance's live cloud (obe_batch_drift); its moments follow on the device."""
        self._drift_step += 1
        ni = self._noise_index
        self._check(self._lib.obe_batch_drift(self._bs(), self._drift_arr, self._ptr(self._drift_dev), self._mask_le,
                                              self._mask_lt, _lib.iarr(ni), 0 if ni is None else len(ni),
                                              self._seed_normal, self._drift_step & 0xffffffff, self._stream()))

    # ---- design half
    @property
    def design_aux(self):
        """Per-channel aux of the likelihood-aware utility (``design_noise='likelihood'``): the planned trials of the
        next binomial measurement, the ``aux`` of a cuda_likelihood's ``noise_var``.  It travels by value in every
        selection launch, so reassigning it between cycles needs no synchronisation."""
        return self._design_aux

    @design_aux.setter
    def design_aux(self, value):
        arr = design_aux_array(value, self._design_lik, self.likelihood_model, self.n_channels)
        if self._design_lik and self.likelihood_model == 'binomial' and not np.all(arr == np.floor(arr)):
            raise ValueError(f'a binomial design_aux is the planned number of trials, an integer >= 1, got {value!r}')
        self._design_aux = value
        self._design_aux_arr = arr

    def opt_setting(self, want_utility=False, sync=True):
        """argmax-utility setting of every instance -> (indices (B,), settings (s, B))."""
        torch = self._torch
        util_ptr = None
        if want_utility:
            if self._utility_dev is None:
                self._utility_dev = torch.zeros((self.n_instances, len(self.setting_indices)), dtype=torch.float64,
                                                device=self._dev)
            util_ptr = C.c_void_p(self._utility_dev.data_ptr())
        var_noise = None
        if self._design_lik:
            var_noise = _lib.darr(self._design_aux_arr, _lib.MAX_CHANNELS)
        elif self._noise_index is None:
            var_noise = _lib.darr((self.default_noise_std ** 2).reshape(-1), _lib.MAX_CHANNELS)
        cost = float(self.cost_of_changing_setting) if self.cost_of_changing_setting is not None else 0.0
        self._check(self._lib.obe_batch_select(self._model, self._bs(), C.c_void_p(self._settings_dev.data_ptr()),
                                               self._lds, len(self.setting_indices), self._cons_arr, self.N_DRAWS,
                                               var_noise, cost, self._seed_uniform, self.cycle, 0,
                                               1 if self.utility_log_form else 0, util_ptr, self._stream()))
        if not sync:
            return None
        idx = self._last_idx.cpu().numpy()
        return idx, self.allsettings[:, idx]

    @property
    def last_setting_index(self):
        return self._last_idx.cpu().numpy()

    def utility(self):
        self.opt_setting(want_utility=True, sync=False)
        return self._utility_dev.cpu().numpy()

    # ---- inference half
    def pdf_update(self, y_meas, sigma=None, settings=None, force_resample=False):
        """Bayesian update of every instance from its own measurement, then the resample of the
        instances whose N_eff dropped below the threshold.  y_meas (B, C); sigma (B, C) or scalar for
        known-sigma models; settings (B, s) or None to use each instance's last chosen setting.
        With a non-Gaussian likelihood y_meas holds the counts (the measured values of a cuda_likelihood) and
        ``sigma`` the record's third element: ignored for Poisson, ``n_trials`` for binomial, the aux of a
        cuda_likelihood (a scalar, (B,) or (B, C)); the records are checked before anything reaches the device."""
        torch = self._torch
        B = self.n_instances
        rec = np.zeros((B, 12))
        if self.likelihood_model != 'gaussian':
            y, aux = count_record(self.likelihood_model, y_meas, sigma, B, self.n_channels)
            n_lik = y.shape[1]
            rec[:, 4:4 + n_lik] = y
            rec[:, 8:8 + n_lik] = aux
        else:
            y = np.asarray(y_meas, dtype=np.float64).reshape(B, -1)
            n_lik = min(self.n_channels, y.shape[1])
            rec[:, 4:4 + n_lik] = y[:, :n_lik]
            if self._noise_index is None:
                if sigma is None:
                    raise ValueError('sigma is required: this engine has no noise_parameter_index (known-sigma model)')
                sg = np.asarray(sigma, dtype=np.float64)
                if sg.ndim == 1 and sg.shape[0] == B:
                    sg = sg.reshape(B, 1)
                rec[:, 8:8 + n_lik] = np.broadcast_to(sg, (B, n_lik))
        if settings is not None:
            st = np.asarray(settings, dtype=np.float64).reshape(B, -1)
            rec[:, :st.shape[1]] = st
        self._record.copy_(torch.from_numpy(rec))
        self._update_from_record(0 if settings is not None else 1, n_lik, force_resample)

    def _update_from_record(self, use_last, n_lik, force_resample):
        auto = bool(self.tuning_parameters['auto_resample'])
        self._check(self._lib.obe_batch_update(self._model, self._bs(), C.c_void_p(self._settings_dev.data_ptr()),
                                               self._lds, use_last, self._cons_arr,
                                               _lib.iarr(self._noise_index), n_lik, 0 if self.choke is None else 1,
                                               0.0 if self.choke is None else float(self.choke),
                                               float(self.tuning_parameters['resample_threshold']) if auto else -1.0,
                                               1 if force_resample else 0, self._stream()))
        if auto or force_resample:
            self._check(self._lib.obe_batch_resample(self._bs(), float(self.tuning_parameters['a_param']),
                                                     1 if self.tuning_parameters['scale'] else 0, self._seed_normal,
                                                     self._seed_uniform, self.cycle, self.N_DRAWS, self._mask_le,
                                                     self._mask_lt, _lib.iarr(self._noise_index),
                                                     0 if self._noise_index is None else len(self._noise_index),
                                                     self._stream()))
        if self._drift is not None:
            self._apply_drift()
        self.cycle += 1

    # ---- on-device MeasurementSimulator (obe_utils.py:8-53), SURVEY 8(f) row 4
    def set_simulator(self, true_params, noise_level=None, seed=12345, drift=None, trials=None):
        """Install the simulated experiment of every instance: ``true_params`` (B, n_model_params) (or one
        set for all), ``noise_level`` a scalar, one value per channel, or (B,) per instance.

        With a count likelihood the simulator draws counts on the device instead of adding Gaussian noise: Poisson
        counts with mean the model output (no ``noise_level``: passing one raises), or binomial counts of ``trials``
        trials (required: a scalar, one per channel, or (B,) per instance; integers in [0, 2^31]) with success
        probability the model output; the trials become the record's third element.  A cuda_likelihood has no
        sampler and raises.  An instance whose model output is invalid for the likelihood gets a NaN count.

        ``drift``: the true parameters of every instance take one Gaussian random-walk step on the device after each
        simulated measurement, so measurement t sees the truth after t steps (``simulator_truth()`` returns the
        current one).  It takes the forms of the engine's ``drift`` over the model's ``n_model_params``; None (the
        default) keeps the truths fixed.  No constraint applies to the truth."""
        torch = self._torch
        B = self.n_instances
        npm = self.model_function.n_model_params
        noise_level = simulator_noise(self.model_function.likelihood, noise_level, trials)
        sim_factors = batched_drift_factors(drift, B, npm)
        tp = np.asarray(true_params, dtype=np.float64)
        if tp.ndim == 1:
            tp = np.broadcast_to(tp[:npm], (B, npm))
        if tp.shape[0] != B or tp.shape[1] < npm:
            raise ValueError(f'true_params must have shape ({B}, >= {npm})')
        self._sim_true = torch.from_numpy(np.ascontiguousarray(tp[:, :npm].T)).to(self._dev)       # (npm, B) SoA
        nl = np.atleast_1d(np.asarray(noise_level, dtype=np.float64))
        self._sim_noise_dev = None
        self._sim_noise = None
        if nl.shape == (B,) and B != self.n_channels and B != 1:
            self._sim_noise_dev = torch.from_numpy(np.ascontiguousarray(nl)).to(self._dev)
        else:
            self._sim_noise = _lib.darr(np.broadcast_to(nl, (self.n_channels,)), _lib.MAX_CHANNELS)
        self._sim_seed = int(seed)
        self._sim_drift_arr, self._sim_drift_dev = self._factor_args(sim_factors)
        self._sim_drift = drift
        self._truth_step = 0

    def simulator_truth(self):
        """(B, n_model_params): the simulator's current true parameters of every instance."""
        if getattr(self, '_sim_true', None) is None:
            raise RuntimeError('call set_simulator(true_params, noise_level) first')
        return self._sim_true.T.cpu().numpy()

    def simulate_measurement(self):
        """Instance b measures at the setting it chose last; the record rows are written on the device.
        Returns the device record tensor (B, 12): [0:4) setting, [4:8) y, [8:12) sigma (a binomial's trials)."""
        if getattr(self, '_sim_true', None) is None:
            raise RuntimeError('call set_simulator(true_params, noise_level) first')
        self._check(self._lib.obe_batch_simulate(
            self._model, self._bs(), C.c_void_p(self._settings_dev.data_ptr()), self._lds,
            C.c_void_p(self._sim_true.data_ptr()), self.n_instances, self._cons_arr, self._sim_noise,
            None if self._sim_noise_dev is None else C.c_void_p(self._sim_noise_dev.data_ptr()),
            self._sim_seed, self.cycle, 1 if self._noise_index is None else 0, self._stream()))
        if self._sim_drift is not None:
            self._truth_step += 1
            self._check(self._lib.obe_batch_truth_drift(
                C.c_void_p(self._sim_true.data_ptr()), self.n_instances, self.n_instances,
                self.model_function.n_model_params, self._sim_drift_arr, self._ptr(self._sim_drift_dev),
                self._sim_seed, self._truth_step & 0xffffffff, self._stream()))
        return self._record

    def closed_loop_cycle(self, force_resample=False):
        """opt_setting -> simulated measurement -> pdf_update of every instance, without any host
        round trip (no synchronisation, no H2D/D2H): the fit_vs_obe study's inner loop
        (demos/fit_vs_obe/fit_vs_obe_makedata.py:149-194) for all runs at once.  With a ``drift`` the cloud steps at
        the end of the update, and with a simulator ``drift`` the truth steps after the simulated measurement."""
        self.opt_setting(sync=False)
        self.simulate_measurement()
        self._update_from_record(1, self.n_channels, force_resample)

    @property
    def just_resampled(self):
        """(B,) bool: which instances the last pdf_update resampled."""
        return self._flag.cpu().numpy().astype(bool)

    # ---- moments (particlepdf.py:173-214), per instance
    def _stats_host(self):
        return self._stats.cpu().numpy()

    def mean(self):
        st = self._stats_host()
        d = self.n_dims
        return st[:, _lib.ST_PIVOT:_lib.ST_PIVOT + d] + st[:, _lib.ST_M1:_lib.ST_M1 + d] / st[:, [_lib.ST_SUMT]]

    def std(self):
        st = self._stats_host()
        d = self.n_dims
        s = st[:, [_lib.ST_SUMT]]
        m1 = st[:, _lib.ST_M1:_lib.ST_M1 + d] / s
        diag = np.zeros((self.n_instances, d))
        q = _lib.ST_M2
        for j in range(d):
            diag[:, j] = st[:, q]
            q += d - j
        return np.sqrt(np.maximum(diag / s - m1 * m1, 0.0))

    def covariance(self):
        st = self._stats_host()
        d = self.n_dims
        out = np.zeros((self.n_instances, d, d))
        s = st[:, _lib.ST_SUMT]
        q = _lib.ST_M2
        for j in range(d):
            for k in range(j, d):
                c = (st[:, q] - st[:, _lib.ST_M1 + j] * st[:, _lib.ST_M1 + k] / s) / (s - st[:, _lib.ST_SUMSQ] / s)
                out[:, j, k] = out[:, k, j] = c
                q += 1
        return out

    def n_eff(self):
        st = self._stats_host()
        return st[:, _lib.ST_TOTAL] ** 2 / st[:, _lib.ST_SUMSQ]

    # ---- per-instance views (tests, inspection)
    def particles(self, b):
        cb = int(self._cur[b].item())
        lo = b * self._np
        return self._p[cb][:, lo:lo + self.n_particles].cpu().numpy()

    def particle_weights(self, b):
        cb = int(self._cur[b].item())
        lo = b * self._np
        w = self._w[cb][lo:lo + self.n_particles].cpu().numpy()
        return w * float(self._stats[b, _lib.ST_INVS].item())


def simulator_noise(likelihood, noise_level, trials):
    """The per-channel / per-instance value the simulator reads (the Gaussian noise level, the binomial trials, 0 for
    Poisson) of ``set_simulator``'s arguments; raises ValueError for an argument the likelihood does not take."""
    if likelihood == 'gaussian':
        if noise_level is None:
            raise ValueError('the Gaussian simulator needs noise_level')
        if trials is not None:
            raise ValueError('trials applies to a binomial likelihood; the Gaussian simulator takes noise_level')
        return noise_level
    if not isinstance(likelihood, str):
        raise ValueError('a cuda_likelihood has no sampler: simulate its measurements on the host and pass them to '
                         'pdf_update')
    if noise_level is not None:
        raise ValueError(f'a {likelihood} simulator draws its own noise and takes no noise_level'
                         + (' (pass trials=)' if likelihood == 'binomial' else ''))
    if likelihood == 'poisson':
        if trials is not None:
            raise ValueError('trials applies to a binomial likelihood')
        return 0.0
    if trials is None:
        raise ValueError('a binomial simulator needs trials: a scalar, one per channel, or one per instance')
    n = np.asarray(trials, dtype=np.float64)
    if not (np.all(np.isfinite(n)) and np.all(n >= 0) and np.all(n <= 2.0 ** 31) and np.all(n == np.floor(n))):
        raise ValueError(f'trials must be integers in [0, 2^31], got {trials!r}')
    return n


def count_record(likelihood, y_meas, aux, n_instances, n_channels):
    """(y (B, n_lik), third element (B, n_lik)) of the batched records of a non-Gaussian likelihood, checked as the
    single engine checks one record: Poisson counts finite non-negative integers (aux ignored), binomial integers
    0 <= k <= n_trials with ``aux`` the trials, a cuda_likelihood's values and aux as given (aux required).  ``aux``
    is a scalar, (B,) or (B, C).  Raises ValueError."""
    y = np.asarray(y_meas, dtype=np.float64).reshape(n_instances, -1)
    n_lik = min(n_channels, y.shape[1])
    y = y[:, :n_lik]
    if likelihood == 'poisson':
        if not (np.all(np.isfinite(y)) and np.all(y >= 0) and np.all(y == np.floor(y))):
            raise ValueError('Poisson counts must be finite non-negative integers')
        return y, np.zeros_like(y)
    if aux is None:
        raise ValueError('a binomial record needs n_trials' if likelihood == 'binomial'
                         else 'a cuda_likelihood record needs its aux')
    a = np.asarray(aux, dtype=np.float64)
    if a.ndim == 1 and a.shape[0] == n_instances:
        a = a.reshape(n_instances, 1)
    a = np.array(np.broadcast_to(a if a.ndim < 2 else a[:, :n_lik], (n_instances, n_lik)))
    if likelihood == 'binomial':
        if not (np.all(np.isfinite(y)) and np.all(np.isfinite(a)) and np.all(y >= 0) and np.all(y <= a)
                and np.all(y == np.floor(y)) and np.all(a == np.floor(a))):
            raise ValueError('binomial records need integers 0 <= k <= n_trials')
    return y, a
