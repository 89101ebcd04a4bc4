"""OptBayesExpt on the GPU: the experiment-design engine of the reference's
``optbayesexpt/obe_base.py`` (v1.2.0) with the same constructor, methods and attributes.

``pdf_update`` is one fused kernel pass over the resident cloud (model -> Gaussian likelihood
-> weight product -> tile sums, N_eff and moments) plus a tiny prefix kernel; ``opt_setting`` /
``good_setting`` draw ``N_DRAWS`` particles through the tile-level CDF, evaluate them over the
whole setting grid and pick the argmax (or a pickiness-weighted draw) on the device.  Only the
measurement record goes to the GPU each cycle, and only the stats block (64 doubles) and the
chosen index come back.
"""
import ctypes as C
import math

import numpy as np

from . import _lib
from .drift import drift_factor
from .models import DESIGN_NOISES, CudaLikelihood, DeviceModel, builtin
from .particlepdf import ParticlePDF

DEFAULT_N_DRAWS = 30
rng = np.random.default_rng()


class LazyDeviceArray:
    """numpy-convertible handle returned by pdf_update: materialises (D2H) only when looked at."""

    def __init__(self, getter):
        self._getter = getter

    def __array__(self, dtype=None, copy=None):
        arr = self._getter()
        return arr if dtype is None else arr.astype(dtype)

    def __getitem__(self, item):
        return self._getter()[item]

    def __len__(self):
        return len(self._getter())

    @property
    def shape(self):
        return self._getter().shape

    def tolist(self):
        return self._getter().tolist()

    def __repr__(self):
        return f'LazyDeviceArray({self._getter()!r})'


def _information_gain_aux_problem(aux):
    """Why the binomial trial counts ``aux`` cannot be the information gain's (None if they can)."""
    a = np.asarray(aux, dtype=np.float64).reshape(-1)
    if not (np.all(np.isfinite(a)) and np.all(a >= 1.0) and np.all(a == np.floor(a))):
        return ("utility_method='information_gain' with a binomial likelihood needs design_aux, the planned number of "
                f'trials, to be an integer >= 1, got {aux!r}')
    return None


def _information_gain_problem(likelihood, design_lik, n_channels, aux):
    """Why an engine cannot run the information-gain utility (None if it can)."""
    user_window = isinstance(likelihood, CudaLikelihood) and likelihood.window is not None
    if not (user_window or (isinstance(likelihood, str) and likelihood in ('poisson', 'binomial'))):
        return ("utility_method='information_gain' needs likelihood_model='poisson' or 'binomial', or a "
                'cuda_likelihood with a window (the sum over counts needs a known support), got '
                f'{likelihood!r}')
    if not design_lik:
        return "utility_method='information_gain' needs design_noise='likelihood'"
    if n_channels != 1:
        return f"utility_method='information_gain' supports single-channel models, got {n_channels} channels"
    if likelihood == 'binomial':
        if aux is None:
            return ("utility_method='information_gain' with a binomial likelihood needs design_aux, the planned "
                    'number of trials')
        return _information_gain_aux_problem(aux)
    return None


def resolve_likelihood(measurement_model, likelihood_model, design_noise, design_aux, utility_method):
    """(model variant, likelihood-aware design?) of an engine built with ``likelihood_model`` / ``design_noise`` /
    ``design_aux`` (see :class:`OptBayesExpt`); raises ValueError for a combination no engine runs."""
    if likelihood_model is not None:
        measurement_model = measurement_model.with_likelihood(likelihood_model)
    if design_noise not in DESIGN_NOISES:
        raise ValueError(f'design_noise must be one of {list(DESIGN_NOISES)}, got {design_noise!r}')
    # the likelihood-aware utility kernel runs only for a non-Gaussian likelihood
    design_lik = design_noise == 'likelihood' and measurement_model.likelihood != 'gaussian'
    if design_lik:
        if utility_method == 'full_kld_utility':
            raise ValueError("design_noise='likelihood' does not apply to full_kld_utility: its noise samples "
                             'are Gaussian draws')
        if measurement_model.likelihood == 'binomial' and design_aux is None:
            raise ValueError("design_noise='likelihood' with a binomial likelihood needs design_aux, the planned "
                             'number of trials of the next measurement')
        measurement_model = measurement_model.with_likelihood(measurement_model.likelihood, 'likelihood')
    elif measurement_model.design_noise != 'fixed':
        measurement_model = measurement_model.with_likelihood(measurement_model.likelihood)
    return measurement_model, design_lik


def design_aux_array(value, design_lik, likelihood, n_channels):
    """The per-channel array of a ``design_aux`` value (see :class:`OptBayesExpt`); raises ValueError."""
    if value is None:
        if design_lik and likelihood == 'binomial':
            raise ValueError("design_noise='likelihood' with a binomial likelihood needs design_aux")
        return np.ones(n_channels)
    arr = np.asarray(value, dtype=np.float64).reshape(-1)
    if arr.size == 1:
        arr = np.full(n_channels, arr[0])
    if arr.size != n_channels:
        raise ValueError(f'design_aux needs a scalar or {n_channels} values, got {arr.size}')
    if not (np.all(np.isfinite(arr)) and np.all(arr > 0)):
        raise ValueError(f'design_aux must be finite and > 0, got {value!r}')
    return arr


class OptBayesExpt(ParticlePDF):
    """Sequential Bayesian experiment design (obe_base.py:21-272).

    ``measurement_model`` must be a :class:`~optbayesexpt_b200.models.DeviceModel` (or the name
    of a built-in): a Python callable cannot run inside a kernel and there is no CPU path.

    ``likelihood_model`` selects the measurement likelihood of the update (the reference's
    ``likelihood`` method, obe_base.py:418-461), evaluated inside the update kernel:

    - ``'gaussian'`` (the default): records ``(setting, y_meas, sigma)``;
    - ``'poisson'``: records ``(setting, counts)`` or ``(setting, counts, ignored)``, the model output is the
      expected count;
    - ``'binomial'``: records ``(setting, k, n_trials)``, the model output is the success probability;
    - :func:`~optbayesexpt_b200.models.cuda_likelihood`: a log-likelihood in CUDA, records
      ``(setting, y_meas, aux)``.

    ``design_noise`` selects the noise variance the utility divides the spread of the model curves by:

    - ``'fixed'`` (the default): ``yvar_noise_model()``, the same at every setting; for counting data
      ``default_noise_std`` then sets the noise scale of the utility (e.g. about sqrt of a typical count);
    - ``'likelihood'``: the likelihood's own noise variance at each setting, averaged over the drawn parameter
      sets -- the expected count for Poisson, p (1 - p) / n for binomial with ``n = design_aux`` the planned trials
      of the next measurement (required), the ``noise_var`` function of a ``cuda_likelihood`` (required) at
      ``aux = design_aux`` (default 1).  A setting where some draw's model output is impossible for the likelihood
      gets utility 0.  On a Gaussian engine this is the fixed variance by definition.  Not with
      ``full_kld_utility``, whose noise samples are Gaussian.

    ``design_aux`` is a scalar or one value per channel, finite and > 0, and may be reassigned between cycles.
    Overriding ``likelihood`` in Python raises ``TypeError``: it could not run inside the kernel.

    ``utility_method='information_gain'`` ranks settings by the mutual information between the parameters and the
    next count, in nats, for the parameters uniform over the K drawn sets:
    ``I(s) = (1/K) sum_k sum_y p_k(y) log(p_k(y) / pbar(y))``, summed exactly over the counts the K draws make
    possible (see :meth:`utility_information_gain`).  It needs ``likelihood_model='poisson'`` or ``'binomial'``, or
    a ``cuda_likelihood`` with a ``window`` (its entry is then a normalised log-pmf, called with ``aux =
    design_aux``), ``design_noise='likelihood'``, a single-channel model and, for binomial, an integer
    ``design_aux >= 1`` (the planned trials).  ``utility_log_form`` does not apply to it and is ignored;
    ``cost_estimate()`` divides it.

    ``drift`` makes the parameters time-varying: after every update (and after the resample, if one ran) each
    particle takes one Gaussian random-walk step ``x <- x + F z``, ``z ~ N(0, I)``, ``F F^T = Q``, on the device.
    ``drift`` is the per-parameter standard deviation of one step (a scalar or ``n_dims`` values) or its
    ``(n_dims, n_dims)`` covariance ``Q`` (symmetric positive semidefinite; zero variance keeps a parameter fixed
    bit for bit), ``None`` (the default) for static parameters.  It may be reassigned between cycles, e.g.
    ``eng.drift = Q_per_unit_time * dt_next`` for irregular time steps.  A step that would leave the region of the
    engine's constraints (the positive noise parameters of OptBayesExptNoiseParameter) is not taken.  The weights
    are not changed.  The normals are Philox normals keyed by the engine seed, the particle slot and the drift step,
    also with ``resampling='multinomial'``.  See :meth:`pdf_update` for what the summaries describe.
    """
    #: why a subclass does not take ``drift`` (None: it does)
    _drift_refusal = None

    def __init__(self, measurement_model, setting_values, parameter_samples, constants,
                 n_draws=DEFAULT_N_DRAWS, choke=None, use_jit=True, utility_method='variance_approx',
                 selection_method='optimal', pickiness=15, default_noise_std=1.0, likelihood_model=None,
                 design_noise='fixed', design_aux=None, drift=None, **kwargs):
        if drift is not None and self._drift_refusal:
            raise ValueError(self._drift_refusal)
        if isinstance(measurement_model, str):
            measurement_model = builtin(measurement_model)
        if not isinstance(measurement_model, DeviceModel):
            raise TypeError('measurement_model must be a DeviceModel (optbayesexpt_b200.models.builtin(...) or '
                            'cuda_source(...)): a Python callable cannot run on the GPU and there is no CPU fallback')
        if type(self).likelihood is not OptBayesExpt.likelihood:
            raise TypeError(f'{type(self).__name__} overrides likelihood() in Python, which the update kernel cannot '
                            'run: pass likelihood_model=\'poisson\' | \'binomial\' | '
                            'optbayesexpt_b200.cuda_likelihood(source, entry) instead')
        measurement_model, self._design_lik = resolve_likelihood(measurement_model, likelihood_model, design_noise,
                                                                 design_aux, utility_method)
        #: 'fixed' or 'likelihood': the noise variance of the utility (see the class documentation)
        self.design_noise = design_noise
        if utility_method == 'information_gain':
            problem = _information_gain_problem(measurement_model.likelihood, self._design_lik,
                                                measurement_model.n_channels, design_aux)
            if problem:
                raise ValueError(problem)
        #: 'gaussian', 'poisson', 'binomial' or a CudaLikelihood
        self.likelihood_model = measurement_model.likelihood
        if self.likelihood_model != 'gaussian':
            self._likelihood_spec = self._counting_spec if isinstance(self.likelihood_model, str) else self._aux_spec
        ParticlePDF.__init__(self, parameter_samples, use_jit=use_jit, **kwargs)
        torch = self._torch
        self.model_function = measurement_model
        self._model_function = measurement_model
        self._model = measurement_model.handle(self.n_dims)
        self.setting_values = setting_values
        # obe_base.py:174-180: all setting combinations, first knob slowest
        self.allsettings = np.array([s.flatten() for s in
                                     np.meshgrid(*[np.asarray(v, dtype=np.float64) for v in setting_values],
                                                 indexing='ij')])
        if self.allsettings.shape[0] != measurement_model.n_settings:
            raise ValueError(f'model takes {measurement_model.n_settings} settings, got {self.allsettings.shape[0]}')
        self.setting_indices = np.arange(len(self.allsettings[0]), dtype=int)
        n_set = len(self.setting_indices)
        self._lds = n_set + (n_set & 1)
        self._settings_dev = torch.zeros((self.allsettings.shape[0], self._lds), dtype=torch.float64,
                                         device=self._buf.device)
        self._settings_dev[:, :n_set].copy_(torch.from_numpy(np.ascontiguousarray(self.allsettings)))
        self.cons = constants
        if len(tuple(constants)) < measurement_model.n_constants:
            raise ValueError(f'model takes {measurement_model.n_constants} constants')
        self._cons_arr = _lib.darr(list(constants)[:_lib.MAX_CONSTANTS], _lib.MAX_CONSTANTS)
        self.choke = choke
        self.N_DRAWS = n_draws
        self.pickiness = pickiness
        self.measurement_results = []
        self.last_setting_index = 0
        self.n_channels = measurement_model.n_channels
        self.utility_y_space = np.array([])   # never materialised on the device path
        self.default_noise_std = np.ones((self.n_channels, 1)) * default_noise_std
        self._utility_code = 4 if utility_method == 'information_gain' else None   # (read by the design_aux setter)
        self.design_aux = design_aux

        utilitymethods = ['variance_approx', 'pseudo_utility', 'full_kld_utility', 'max_min', 'information_gain']
        if utility_method == 'variance_approx':
            self._utility_code = 0
        elif utility_method == 'max_min':
            self._utility_code = 1
        elif utility_method == 'pseudo_utility':
            self._utility_code = 2
        elif utility_method == 'full_kld_utility':
            self._utility_code = 3
            if self.n_channels != 1:
                raise ValueError('full_kld_utility supports single-channel models (the reference broadcast '
                                 'of obe_base.py:719-720 only works for one channel)')
        elif utility_method == 'information_gain':
            self._utility_code = 4
        else:
            raise SyntaxError(f'Unknown utility method, {utility_method}. '
                              f'Valid utility methods are: {utilitymethods}')
        self.utility_method = utility_method
        #: use log(1 + var/sigma^2) instead of the linear form of obe_base.py:654 (the information gain ignores it)
        self.utility_log_form = False

        selection_methods = ['optimal', 'good', 'random']
        if selection_method == 'optimal':
            self.get_setting = self.opt_setting
        elif selection_method == 'good':
            self.get_setting = self.good_setting
        elif selection_method == 'random':
            self.get_setting = self.random_setting
        else:
            raise SyntaxError(f'Unknown selection_method, {selection_method}. '
                              f'Valid selection methods are: {selection_methods}')

        self._utility_dev = torch.zeros(n_set, dtype=torch.float64, device=self._buf.device)
        self._best_dev = torch.zeros(2, dtype=torch.int64, device=self._buf.device)
        self._pick_dev = torch.zeros(1, dtype=torch.int64, device=self._buf.device)
        self._select_scratch = torch.zeros(int(self._lib.obe_select_scratch_bytes(n_set)), dtype=torch.uint8,
                                           device=self._buf.device)
        self._cost_dev = None
        self._best_host = torch.zeros(2, dtype=torch.int64).pin_memory()
        self._best_host_np = self._best_host.numpy()
        # reusable by-value argument arrays (a small-cloud cycle is host-bound: no allocations per call)
        self._a_setting = _lib.ArgArray(_lib.MAX_SETTINGS)
        self._a_y = _lib.ArgArray(_lib.MAX_CHANNELS)
        self._a_sigma = _lib.ArgArray(_lib.MAX_CHANNELS)
        self._a_pivot = _lib.ArgArray(_lib.MAX_PARAMS)
        self._a_u = None
        self._var_noise_cache = None
        #: early select: when a systematic resample is followed by the selection (run_cycle_async, or pdf_update
        #: with ``eager_select``), the K draws are taken from the resample PLAN (offspring slot floor(u*N)) before
        #: the cloud is streamed, and the utility pass overlaps the resample on a second stream
        self.early_select = True
        #: pdf_update: a resample also starts the selection the next opt_setting()/good_setting() will ask for
        #: (the K uniforms are drawn from ``self.rng`` at that moment instead of inside opt_setting)
        self.eager_select = False
        #: pdf_update does not wait for the stats block when the resample decision does not depend on it
        #: (auto_resample off, or resample_threshold > 1): one C call, no synchronisation; the pivot of the moment
        #: accumulators and the impoverishment warning then lag one update behind
        self.async_update = False
        #: with ``eager_select`` and ``async_update`` both on, a pdf_update whose resample decision DOES depend on
        #: N_eff (the normal case) leaves the test to the device: one C call, the outcome arrives with the argmax at
        #: the one synchronisation of the cycle (opt_setting / good_setting / just_resampled / any look at the cloud)
        self.device_resample_test = True
        #: ... and that call is split in two: the update kernel is enqueued first, the resample / selection half of
        #: the argument struct is filled in (and the uniforms drawn) while it runs
        self.split_cycle = True
        #: early select runs the selection on a second stream beside the streaming resample from this many particles on;
        #: below, the same early order goes to the main stream.  Measured: two streams win even at 1e4 particles (65 vs
        #: 72 us per forced c1 cycle, 115 vs 124 us at c3), so the default is 0
        self.two_stream_min_particles = 0
        self._select_ready = False
        self._side = None                 # (torch stream object, raw handle) of the selection stream
        # pinned landing block of the cycle entry: [0:64] the update's stats block, [64:66] (argmax index, value)
        # and [66] the completion word the utility kernel raises once the pair has landed
        self._cy_pin = torch.zeros(_lib.STATS_LEN + 4, dtype=torch.float64).pin_memory()
        self._cy_pin_np = self._cy_pin.numpy()
        self._cy_stats_np = self._cy_pin_np[:_lib.STATS_LEN]
        self._cy_best_np = self._cy_pin_np[_lib.STATS_LEN:_lib.STATS_LEN + 2].view(np.int64)
        self._cy_seq_np = self._cy_pin_np[_lib.STATS_LEN + 2:_lib.STATS_LEN + 3].view(np.uint64)
        self._cy_seq = 0                  # number of the last cycle that was asked to deliver its results
        self._cy_seq_seen = 0             # ... and of the last one whose results were seen on the host
        #: wait for a cycle's results by polling the completion word instead of synchronising the stream: trailing
        #: gated-off launches and the stream-synchronisation wake-up leave the critical path (3 us per small-cloud
        #: cycle); falls back to a stream synchronisation after `poll_spins` looks (~4 ms).  Kernels still in flight
        #: behind the word (the streaming resample of a resampling cycle) are ordered before everything enqueued later
        self.poll_results = True
        self.poll_spins = 40000
        self._cy_polls = False            # the last delivering cycle ran a selection (which raises the word)
        self._cy_copy_out = False         # the next cycle call also copies stats + argmax into the pinned block
        self._best_copied = False         # the argmax of the prepared selection is on its way to _cy_best_np
        self._async_pending = False
        self._dt_cache = None
        self._drift_epoch = 0             # drift steps taken: the epoch word of their normals
        self.drift = drift

    # ------------------------------------------------------------------------------------------
    # time-varying parameters
    # ------------------------------------------------------------------------------------------
    @property
    def drift(self):
        """Standard deviations or covariance of one random-walk step of the parameters per update (None: static)."""
        return self._drift

    @drift.setter
    def drift(self, value):
        if value is not None and self._drift_refusal:
            raise ValueError(self._drift_refusal)
        factor = drift_factor(value, self.n_dims)
        self._drift = value
        self._drift_F = factor
        self._drift_arr = None if factor is None else _lib.darr(factor.reshape(-1), _lib.MAX_PARAMS * _lib.MAX_PARAMS)
        self._dt_cache = None

    def _apply_drift(self, pivot):
        """One random-walk step of the live cloud (obe_drift); its moments are then valid on the device."""
        self._drift_epoch += 1
        ni = self._noise_index
        le, lt = self._constraint_masks()
        self._check(self._lib.obe_drift(self._cs(), self._drift_arr, le, lt, self._noise_iarr(ni),
                                        0 if ni is None else len(ni), _lib.darr(pivot, _lib.MAX_PARAMS),
                                        self._philox_seed, self._drift_epoch & 0xffffffff, None, self._stream()))
        self._after_drift()

    def _after_drift(self):
        self._invalidate(particles=True)
        self._cloud_version += 1
        self._stats = None
        self._moments_valid = True

    # -- the reference rebinds `parameters` to `particles` in pdf_update (obe_base.py:185,395);
    #    here it is a live alias, which removes the stale-alias quirk after resample()/set_pdf()
    @property
    def parameters(self):
        return self.particles

    def _invalidate(self, particles=False, weights=True):
        ParticlePDF._invalidate(self, particles, weights)
        self._select_ready = False        # a prefetched selection belongs to the cloud it was drawn from

    def set_n_draws(self, n_draws=None):
        """obe_base.py:274-296."""
        self._select_ready = False
        if n_draws == 'default':
            self.N_DRAWS = DEFAULT_N_DRAWS
        elif n_draws:
            self.N_DRAWS = n_draws
        return self.N_DRAWS

    def set_pdf(self, samples, weights=None):
        if self._pending_cycle:
            self._settle()
        self._select_ready = False
        noise_index = self._noise_index
        ParticlePDF.set_pdf(self, samples, weights)
        self._noise_index = noise_index
        self._model = self.model_function.handle(self.n_dims)
        if self._drift is not None:
            self.drift = self._drift          # (checks the shape against the new cloud)

    # ------------------------------------------------------------------------------------------
    # model evaluation in both orientations (obe_base.py:298-338)
    # ------------------------------------------------------------------------------------------
    def eval_over_all_parameters(self, onesettingset):
        if self._pending_cycle:
            self._settle()
        y = self._eval_parameters_dev(onesettingset)
        return y[:, :self.n_particles].cpu().numpy()

    def eval_over_all_parameters_dev(self, onesettingset):
        """The model over all particles at one setting, left on the device: pass the result as
        ``pdf_update(record, y_model_data=...)`` to overlap the model pass with the instrument's measurement
        (obe_base.py:374-385) without a host round trip."""
        return self._eval_parameters_dev(onesettingset)

    def prefetch_model(self, onesettingset):
        """Start the model pass for the setting the instrument is about to measure (obe_base.py:374-385: "the
        model evaluation can be done while waiting for measurement results").  Enqueued on a side stream, so it
        overlaps whatever else the device is doing; the next ``pdf_update`` for the same setting picks the result up
        (unless the cloud was resampled or replaced in between) instead of evaluating the model in its own pass."""
        if self._pending_cycle:
            self._settle()
        torch = self._torch
        side = getattr(self, '_prefetch_stream', None)
        if side is None:
            side = self._prefetch_stream = torch.cuda.Stream(device=self._buf.device)
        key = tuple(float(v) for v in np.atleast_1d(onesettingset))
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            y = self._eval_parameters_dev(onesettingset)
        done = torch.cuda.Event()
        done.record(side)
        self._prefetched = (key, y, done, self._cloud_version)

    def _take_prefetched(self, onesetting):
        pre = getattr(self, '_prefetched', None)
        self._prefetched = None
        if pre is None:
            return None
        key, y, done, version = pre
        if version != self._cloud_version or key != tuple(float(v) for v in np.atleast_1d(onesetting)):
            return None
        self._torch.cuda.current_stream().wait_event(done)
        return y

    def _eval_parameters_dev(self, onesettingset):
        y = self._torch.empty((self.n_channels, self._buf.ld), dtype=self._torch.float64, device=self._buf.device)
        self._check(self._lib.obe_eval_parameters(self._model, self._cs(),
                                                  _lib.darr(np.atleast_1d(onesettingset), _lib.MAX_SETTINGS),
                                                  self._cons_arr, C.c_void_p(y.data_ptr()), self._buf.ld,
                                                  self._stream()))
        return y

    def eval_over_all_settings(self, oneparamset):
        n_set = len(self.setting_indices)
        y = self._torch.empty((self.n_channels, self._lds), dtype=self._torch.float64, device=self._buf.device)
        self._check(self._lib.obe_eval_settings(self._model, C.c_void_p(self._settings_dev.data_ptr()), self._lds,
                                                n_set, _lib.darr(np.atleast_1d(oneparamset), _lib.MAX_PARAMS),
                                                self._cons_arr, C.c_void_p(y.data_ptr()), self._lds, self._stream()))
        return y[:, :n_set].cpu().numpy()

    # ------------------------------------------------------------------------------------------
    # inference half (obe_base.py:340-461)
    # ------------------------------------------------------------------------------------------
    def _likelihood_spec(self, measurement_record):
        """(y_meas[C], sigma[C] | None, noise_index | None, n_lik) -- the zip() of
        obe_base.py:453-455 truncates to the shortest of (channels, y_meas, sigma)."""
        onesetting, y_meas, sigma = measurement_record[0], measurement_record[1], measurement_record[2]
        if type(y_meas) is float and type(sigma) is float:       # the common single-channel record, without numpy
            return (y_meas,), (sigma,), None, 1
        y_meas = np.atleast_1d(np.asarray(y_meas, dtype=np.float64))
        sigma = np.atleast_1d(np.asarray(sigma, dtype=np.float64))
        n_lik = min(self.n_channels, len(y_meas), len(sigma))
        return y_meas[:n_lik], sigma[:n_lik], None, n_lik

    def _counting_spec(self, measurement_record):
        """Poisson (setting, counts[, ignored]) / binomial (setting, k, n_trials) records: (k[C], n_trials[C] |
        None, None, n_lik), checked here so that a bad record raises before anything is enqueued."""
        k = measurement_record[1]
        if type(k) is float:                     # the common single-channel record, without numpy
            if self.likelihood_model == 'poisson':
                n = k
            else:
                n = measurement_record[2] if len(measurement_record) > 2 else None
            if type(n) is float and 0.0 <= k <= n < math.inf and k == math.floor(k) and n == math.floor(n):
                return (k,), (None if self.likelihood_model == 'poisson' else (n,)), None, 1
        k = np.atleast_1d(np.asarray(measurement_record[1], dtype=np.float64))
        n_lik = min(self.n_channels, len(k))
        if self.likelihood_model == 'poisson':
            k = k[:n_lik]
            if not (np.all(np.isfinite(k)) and np.all(k >= 0) and np.all(k == np.floor(k))):
                raise ValueError(f'Poisson counts must be finite non-negative integers, got {k}')
            return k, None, None, n_lik
        if len(measurement_record) < 3:
            raise ValueError('a binomial record is (setting, k, n_trials)')
        n = np.atleast_1d(np.asarray(measurement_record[2], dtype=np.float64))
        n_lik = min(n_lik, len(n))
        k, n = k[:n_lik], n[:n_lik]
        if not (np.all(np.isfinite(k)) and np.all(np.isfinite(n)) and np.all(k >= 0) and np.all(k <= n)
                and np.all(k == np.floor(k)) and np.all(n == np.floor(n))):
            raise ValueError(f'binomial records need integers 0 <= k <= n_trials, got k={k}, n_trials={n}')
        return k, n, None, n_lik

    def _aux_spec(self, measurement_record):
        """cuda_likelihood records (setting, y_meas, aux): (y_meas[C], aux[C], None, n_lik)."""
        if len(measurement_record) < 3:
            raise ValueError('a cuda_likelihood record is (setting, y_meas, aux)')
        y_meas = np.atleast_1d(np.asarray(measurement_record[1], dtype=np.float64))
        aux = np.atleast_1d(np.asarray(measurement_record[2], dtype=np.float64))
        n_lik = min(self.n_channels, len(y_meas), len(aux))
        return y_meas[:n_lik], aux[:n_lik], None, n_lik

    def pdf_update(self, measurement_record, y_model_data=None):
        """Bayesian update of the cloud from one measurement (obe_base.py:340-399).

        Returns ``(particles, particle_weights)`` as lazy, numpy-convertible handles: nothing is
        copied off the GPU unless the caller looks at them.

        With a ``drift`` the random-walk step is the last thing the update does, on every path: after it the cloud
        and therefore ``mean()``, ``std()``, ``covariance()``, ``quantile()``, ``histogram()``, ``randdraw()`` and
        the draws of the next ``opt_setting()`` are one step ahead -- the predictive distribution of the parameters
        at the next measurement, not the posterior at this one.
        """
        if self._pending_cycle:
            self._settle()
        if self.async_update and y_model_data is None and getattr(self, '_prefetched', None) is None:
            decision = self._resample_decision_known()
            if decision is not None and self._cycle_c_ok(decision, bool(self.eager_select)):
                return self._pdf_update_async(measurement_record, decision)
            if decision is None and self._device_test_ok():
                return self._pdf_update_device_test(measurement_record)
        onesetting = measurement_record[0]
        y_meas, sigma, noise_index, n_lik = self._likelihood_spec(measurement_record)
        use_choke = 0 if self.choke is None else 1
        choke = 0.0 if self.choke is None else float(self.choke)
        update_pivot = self._pivot
        pivot = self._a_pivot.fill(self._pivot)
        if y_model_data is None and getattr(self, '_prefetched', None) is not None:
            y_model_data = self._take_prefetched(onesetting)
        if y_model_data is None:
            self._check(self._lib.obe_update(self._model, self._cs(), self._a_setting.fill(onesetting), self._cons_arr,
                                             self._a_y.fill(y_meas),
                                             None if sigma is None else self._a_sigma.fill(sigma),
                                             self._noise_iarr(noise_index), n_lik, use_choke, choke, pivot,
                                             self._stream()))
        else:
            torch = self._torch
            if isinstance(y_model_data, torch.Tensor) and y_model_data.is_cuda and y_model_data.dtype == torch.float64 \
                    and y_model_data.dim() == 2 and y_model_data.shape == (self.n_channels, self._buf.ld) \
                    and y_model_data.is_contiguous():
                y = y_model_data          # eval_over_all_parameters_dev: the model pass was prefetched on the device
            else:
                y = torch.zeros((self.n_channels, self._buf.ld), dtype=torch.float64, device=self._buf.device)
                if isinstance(y_model_data, torch.Tensor):
                    src = y_model_data.to(dtype=torch.float64, device=self._buf.device).reshape(self.n_channels, -1)
                else:
                    src = torch.as_tensor(np.ascontiguousarray(
                        np.asarray(y_model_data, dtype=np.float64).reshape(self.n_channels, -1)))
                y[:, :self.n_particles].copy_(src[:, :self.n_particles])
            self._check(self._lib.obe_update_from_y_model(self._model, self._cs(), C.c_void_p(y.data_ptr()),
                                                          self._buf.ld, self.n_channels,
                                                          _lib.darr(y_meas, _lib.MAX_CHANNELS),
                                                          None if sigma is None else _lib.darr(sigma, _lib.MAX_CHANNELS),
                                                          _lib.iarr(noise_index), n_lik, use_choke, choke, pivot,
                                                          self._stream()))
        self._after_update()
        if self.just_resampled:
            self.enforce_parameter_constraints()
        if self._drift_F is not None:
            # (moments around the update's pivot, and the next pivot from the step's moments: what the cycle entry
            # does, so that every path computes the same bits)
            self._apply_drift(update_pivot)
            mean = self._mean_from(self._fetch_stats())
            if np.all(np.isfinite(mean)):
                self._pivot = mean
        return (LazyDeviceArray(lambda: self.particles), LazyDeviceArray(lambda: self.particle_weights))

    # ---- pdf_update without a host synchronisation ------------------------------------------------
    def _resample_decision_known(self):
        """True / False when the resample test of particlepdf.py:236-258 does not depend on N_eff (auto_resample
        off, or a threshold above 1: N_eff / N <= 1 always), None when the host has to look at N_eff."""
        tp = self.tuning_parameters
        if not tp['auto_resample']:
            return False
        if tp['resample_threshold'] > 1.0:
            return True
        return None

    def _pdf_update_async(self, measurement_record, resample):
        """pdf_update as ONE C call and no synchronisation (``async_update``): the resample decision is known
        beforehand, so nothing has to come back before the kernels are enqueued.  The stats block follows in an
        asynchronous copy and is adopted by the NEXT update (pivot of the moment accumulators; the particle
        impoverishment warning of particlepdf.py:245-250 is therefore issued one update late)."""
        self._adopt_async_stats()
        select = bool(self.eager_select)
        self._cy_copy_out = True
        try:
            self.run_cycle_async(measurement_record, resample=resample, select=select)
        finally:
            copied, self._cy_copy_out = not self._cy_copy_out, False     # (the C entry consumed the request)
        self._select_ready = select
        self.just_resampled = bool(resample)
        if copied:
            self._async_pending, self._best_copied = 'cycle', select
        else:
            self._post_async_stats(resample)
        if resample and self._constraint_masks() == (0, 0):
            self.enforce_parameter_constraints()          # (mask constraints were applied inside the cycle)
        return (LazyDeviceArray(lambda: self.particles), LazyDeviceArray(lambda: self.particle_weights))

    def _async_stats_source(self, resample):
        """Device block holding the stats of the update that just ran (the resample swapped the buffers), or of the
        drift step that followed it on the live cloud."""
        if self._drift_F is not None:
            return self._buf.stats
        return (self._alt if resample else self._buf).stats

    def _post_async_stats(self, resample):
        torch = self._torch
        pin = getattr(self, '_async_pin', None)
        if pin is None:
            pin = self._async_pin = torch.zeros(_lib.STATS_LEN, dtype=torch.float64).pin_memory()
            self._async_pin_np = pin.numpy()
            self._async_ev = torch.cuda.Event()
        pin.copy_(self._async_stats_source(resample), non_blocking=True)
        self._async_ev.record()
        self._async_pending = True

    def _adopt_async_stats(self):
        pending, self._async_pending = self._async_pending, False
        if not pending:
            return
        if pending == 'cycle':                  # delivered by obe_cycle itself
            self._wait_cycle()                  # (already seen in a closed loop: opt_setting waited for this cycle)
            st = self._cy_stats_np.copy()
        else:
            self._async_ev.synchronize()        # (already complete in a closed loop: opt_setting synchronised since)
            st = self._async_pin_np.copy()
        self._adopt_stats(st)

    def _wait_cycle(self):
        """Block until the results of the last delivering cycle (stats block, argmax pair) are on the host: poll the
        completion word the utility kernel raises, or synchronise the stream."""
        seq = self._cy_seq
        if self._cy_seq_seen == seq:
            return
        # (no completion word without a selection; kernels on an override stream are not ordered with torch's copies,
        # so the host must not run ahead of them)
        if self.poll_results and self._cy_polls and self._stream_override is None:
            flag = self._cy_seq_np
            for _ in range(self.poll_spins):
                if flag[0] == seq:
                    self._cy_seq_seen = seq
                    return
        self._check(self._lib.obe_stream_sync(self._stream()))
        self._cy_seq_seen = seq

    def _adopt_stats(self, st):
        """Pivot of the next update's moment accumulators and the impoverishment warning, from a stats block."""
        # (plain floats: the same IEEE operations as _mean_from / _n_eff_from without the numpy call overhead -- this
        # runs between the synchronisation of a cycle and the launch of the next one)
        v = st.tolist()
        sumt, d = v[_lib.ST_SUMT], self.n_dims
        if sumt != 0.0:
            mean = [v[_lib.ST_PIVOT + j] + v[_lib.ST_M1 + j] / sumt for j in range(d)]
            if math.isfinite(sum(mean)):
                self._pivot = np.array(mean)
        invs, ssq = v[_lib.ST_INVS], v[_lib.ST_SUMSQ]
        den = ssq * (invs * invs)
        n_eff = 1.0 / den if den != 0.0 else math.inf
        if n_eff < 0.1 * self._n_total_for_test():
            import warnings
            warnings.warn("\nParticle filter rejected > 90 % of particles. "
                          f"N_eff = {n_eff:.2f}. "
                          "Particle impoverishment may lead to errors.", RuntimeWarning)

    def _n_total_for_test(self):
        return self.n_particles

    def _async_stats_ptr(self, resample):
        """Device address of the stats block the cycle entry copies out (None: the updated cloud's own block)."""
        return None

    # ---- pdf_update with the resample test on the device ------------------------------------------
    def _device_test_ok(self):
        tp = self.tuning_parameters
        # the answer only changes with these switches: one tuple compare per update instead of seven method calls
        key = (self.device_resample_test, self.eager_select, self.resampling, tp['resample_threshold'], self.early_select,
               self.use_cycle_entry, self.N_DRAWS, self._utility_code, self._stream_override, self._drift_F is None)
        cached = self._dt_cache
        if cached is not None and cached[0] == key:
            return cached[1]
        # (with a drift the cycle draws from the drifted cloud instead of the resample plan, under the same conditions)
        ok = bool(self.device_resample_test and self.eager_select and self.resampling == 'systematic'
                  and 0.0 <= tp['resample_threshold'] <= 1.0 and self._constraint_masks() == (0, 0)
                  and not self._noise_from_stats() and self._early_select_possible() and self._cycle_c_ok(True, True))
        # (a subclass with its own cost model can change its mind between calls: do not cache for it)
        if type(self).cost_estimate is OptBayesExpt.cost_estimate:
            self._dt_cache = (key, ok)
        return ok

    def _pdf_update_device_test(self, measurement_record):
        """pdf_update + the selection of the next opt_setting() as ONE C call whose resample test
        (particlepdf.py:236-258) runs on the device: obe_cycle(resample=2).  The host learns whether the cloud was
        resampled when it synchronises for the argmax; until then the cycle is pending and any look at the cloud
        (``_buf``), ``just_resampled`` or the selection settles it first.  ``self.rng`` is consumed as in the
        synchronous path when a resample fires (u0, then the K uniforms); when it does not, the u0 drawn for it
        is simply unused."""
        self._settle()
        self._adopt_async_stats()
        cy = self._cycle_struct()
        self._cy_copy_out = True
        lib, ref = self._lib, C.byref(cy)
        # phase 1: the update kernel goes to the device before the host has filled in the other half of the struct
        self._fill_cycle_update(cy, measurement_record, True)
        cy.resample = 2
        cy.resample_threshold = float(self.tuning_parameters['resample_threshold'])
        split = self.split_cycle
        if split:
            cy.phase = 1
            self._check(lib.obe_cycle(ref))
        # phase 2: gated resample half + selection, enqueued while the update runs
        self._fill_cycle_rest(cy, True, True)
        cy.side_stream = None
        cy.u0 = float(self.rng.random())
        self._cy_u[:cy.k] = self.rng.random(cy.k)
        cy.phase = 2 if split else 0
        try:
            self._check(lib.obe_cycle(ref))
        except Exception:
            if split:                           # the update of phase 1 is already on the device: account for it
                self._invalidate(particles=True)
                self._stats = None
                self._moments_valid, self._weights_lazy = True, True
            raise
        self._invalidate(particles=True)
        self._stats = None
        self._last_ancestors = None
        self._pending_cycle = True
        self._select_ready = True
        self._best_copied = True
        return (LazyDeviceArray(lambda: self.particles), LazyDeviceArray(lambda: self.particle_weights))

    def _settle(self):
        """Wait for a pending device-decided cycle and do the host bookkeeping of its outcome."""
        if not self._pending_cycle:
            return False
        self._pending_cycle = False
        self._wait_cycle()
        st = self._cy_stats_np.copy()
        fired = bool(st[_lib.ST_FIRED] != 0.0)
        ready, copied = self._select_ready, self._best_copied
        self._after_cycle_c(fired)
        self._select_ready, self._best_copied = ready, copied     # (the prepared selection belongs to this outcome)
        self._just_resampled = fired
        if not fired or self._cy.drift:
            self._stats = st                    # the live cloud's stats block, already on the host
        self._adopt_stats(st)
        return True

    def _noise_iarr(self, noise_index):
        """ctypes int array of the noise-parameter rows (cached: it never changes for an engine)."""
        if noise_index is None:
            return None
        key = tuple(noise_index)
        cached = getattr(self, '_noise_iarr_cache', None)
        if cached is None or cached[0] != key:
            cached = self._noise_iarr_cache = (key, _lib.iarr(noise_index))
        return cached[1]

    def run_cycle_async(self, measurement_record, resample=True, select=True):
        """One full cycle -- pdf_update, (forced) systematic resample, utility + argmax -- enqueued
        on the current stream with NO host synchronisation: the resample decision is the
        caller's, the chosen index stays in ``best_index_dev``.  For pipelined / benchmark use;
        ``pdf_update`` + ``opt_setting`` is the synchronous, reference-shaped API."""
        if self._pending_cycle:
            self._settle()
        if self._cycle_c_ok(resample, select):
            return self._run_cycle_c(measurement_record, resample, select)
        onesetting = measurement_record[0]
        y_meas, sigma, noise_index, n_lik = self._likelihood_spec(measurement_record)
        self._check(self._lib.obe_update(self._model, self._cs(),
                                         _lib.darr(np.atleast_1d(onesetting), _lib.MAX_SETTINGS), self._cons_arr,
                                         _lib.darr(y_meas, _lib.MAX_CHANNELS),
                                         None if sigma is None else _lib.darr(sigma, _lib.MAX_CHANNELS),
                                         _lib.iarr(noise_index), n_lik, 0 if self.choke is None else 1,
                                         0.0 if self.choke is None else float(self.choke),
                                         _lib.darr(self._pivot, _lib.MAX_PARAMS), self._stream()))
        self._invalidate()
        self._stats = None
        self._moments_valid = True      # on the device: the resample kernel reads them there
        self._weights_lazy = True
        self.resample_select_async(resample, select)

    # ---- the whole cycle as ONE C call (obe_cycle): no Python between the launches ---------------
    #: run_cycle_async goes through obe_cycle when the engine's configuration allows it
    use_cycle_entry = True

    def _cycle_c_ok(self, resample, select):
        if not self.use_cycle_entry or (resample and self.resampling != 'systematic'):
            return False
        if select and (self._utility_code == 3 or not (1 <= self.N_DRAWS <= _lib.MAX_DRAWS)):
            return False
        if select:
            cost = self.cost_estimate()
            if not (np.isscalar(cost) and float(cost) == 1.0):
                return False
        return True

    def _cycle_struct(self):
        cy = getattr(self, '_cy', None)
        if cy is None:
            cy = self._cy = _lib.Cycle()
            cy.model = self._model
            cy.constants = C.cast(self._cons_arr, C.POINTER(C.c_double))
            cy.settings_dev = self._settings_dev.data_ptr()
            cy.lds = self._lds
            cy.n_settings = len(self.setting_indices)
            cy.utility_dev = self._utility_dev.data_ptr()
            cy.best_dev = self._best_dev.data_ptr()
            cy.select_scratch_dev = self._select_scratch.data_ptr()

            def view(field, count):         # the by-value arrays of the struct as numpy views: one slice store each
                return np.frombuffer(cy, dtype=np.float64, count=count, offset=getattr(_lib.Cycle, field).offset)
            self._cy_u = view('u', 128)
            self._cy_setting, self._cy_y = view('setting', _lib.MAX_SETTINGS), view('y_meas', _lib.MAX_CHANNELS)
            self._cy_sigma, self._cy_pivot = view('sigma', _lib.MAX_CHANNELS), view('pivot', _lib.MAX_PARAMS)
            self._cy_vn = view('var_noise', _lib.MAX_CHANNELS)
            self._cy_ni = np.frombuffer(cy, dtype=np.int32, count=_lib.MAX_CHANNELS,
                                        offset=_lib.Cycle.noise_index.offset)
        return cy

    def _fill_cycle(self, cy, measurement_record, resample, select):
        """The per-cycle fields of the obe_cycle_t; consumes self.rng in the order resample() / opt_setting() do."""
        self._fill_cycle_update(cy, measurement_record, resample)
        self._fill_cycle_rest(cy, resample, select)

    def _fill_cycle_update(self, cy, measurement_record, resample):
        """What the update kernel needs: the record, the pivot, the live cloud, the stream, the copy-out block."""
        y_meas, sigma, noise_index, n_lik = self._likelihood_spec(measurement_record)
        cy.model = self._model
        st = np.atleast_1d(measurement_record[0])
        self._cy_setting[:min(len(st), _lib.MAX_SETTINGS)] = st[:_lib.MAX_SETTINGS]
        self._cy_y[:len(y_meas)] = y_meas
        cy.has_sigma = 0 if sigma is None else 1
        if sigma is not None:
            self._cy_sigma[:len(sigma)] = sigma
        cy.has_noise_index = 0 if noise_index is None else 1
        ni = self._noise_index
        if noise_index is not None:
            self._cy_ni[:len(noise_index)] = noise_index
        elif ni is not None:
            self._cy_ni[:len(ni)] = ni
        cy.n_noise = 0 if ni is None else len(ni)
        cy.n_lik_channels = n_lik
        choke = self.choke
        cy.use_choke = 0 if choke is None else 1
        cy.choke = 0.0 if choke is None else float(choke)
        self._cy_pivot[:self.n_dims] = self._pivot
        cy.cloud = self._buf.ptr()
        cy.resample = 1 if resample else 0
        cy.stream = self._stream().value
        if self._cy_copy_out:
            self._cy_copy_out = False
            base = self._cy_pin.data_ptr()
            cy.stats_host, cy.best_host = base, base + 8 * _lib.STATS_LEN
            cy.stats_src_dev = self._async_stats_ptr(resample)
            self._cy_seq += 1
            self._cy_polls = False        # (set by _fill_cycle_rest when the cycle selects)
            cy.seq, cy.seq_host = self._cy_seq, base + 8 * (_lib.STATS_LEN + 2)
        else:
            cy.stats_host = cy.best_host = cy.stats_src_dev = cy.seq_host = None
        cy.phase = 0

    def _fill_cycle_rest(self, cy, resample, select):
        """The resample and selection halves of the struct."""
        buf = self._buf
        if resample:
            alt = self._alt
            if alt is None:
                alt = self._alt = buf.empty_like()
            cy.alt = alt.ptr()
            tp = self.tuning_parameters
            cy.scale = 1 if tp['scale'] else 0
            cy.a_param = float(tp['a_param'])
            cy.seed = self._philox_seed
            cy.epoch = self._epoch + 1
            cy.mask_le, cy.mask_lt = self._constraint_masks()
        cy.select = 1 if select else 0
        cy.noise_from_stats = 1 if self._noise_from_stats() else 0
        if select:
            cy.k = int(self.N_DRAWS)
            cy.draws_dev = self._draws_buffer().data_ptr()
            cy.method = self._utility_code
            cy.log_form = 1 if self.utility_log_form else 0
            if not cy.noise_from_stats:
                vn = np.asarray(self._design_var_noise(), dtype=np.float64).reshape(-1)
                self._cy_vn[:min(len(vn), _lib.MAX_CHANNELS)] = vn[:_lib.MAX_CHANNELS]
        if self._drift_F is not None:
            self._drift_epoch += 1
            cy.drift, cy.drift_epoch, cy.seed = 1, self._drift_epoch & 0xffffffff, self._philox_seed
            cy.drift_mask_le, cy.drift_mask_lt = self._constraint_masks()
            C.memmove(C.addressof(cy) + _lib.Cycle.drift_factor.offset, self._drift_arr, C.sizeof(self._drift_arr))
        else:
            cy.drift = 0
        if self.early_select and resample and select and self._drift_F is None:
            # (small clouds: same early order on the main stream -- the fork / join cost more than the overlap hides)
            cy.side_stream = (self._side_stream()[1].value if self._n_total_for_test() >= self.two_stream_min_particles
                              else cy.stream)
        else:
            cy.side_stream = None
        # The completion word is raised by the utility kernel.  A stats block the kernels store themselves is on the
        # host before it; one that is COPIED (stats_src_dev: the combined block of a sharded cloud) is only ahead of
        # the word in the early order, where the copy is enqueued before the selection -- otherwise wait on the stream.
        if select and cy.seq_host:
            self._cy_polls = bool(cy.stats_src_dev is None or cy.side_stream)

    def _run_cycle_c(self, measurement_record, resample, select):
        if self._pending_cycle:
            self._settle()
        cy = self._cycle_struct()
        split = self.split_cycle and (resample or select)
        self._fill_cycle_update(cy, measurement_record, resample)
        if split:                               # the update kernel first, the rest of the struct while it runs
            cy.phase = 1
            self._check(self._lib.obe_cycle(C.byref(cy)))
        self._fill_cycle_rest(cy, resample, select)
        if resample:
            cy.u0 = float(self.rng.random())
        if select:
            self._cy_u[:cy.k] = self.rng.random(cy.k)
        cy.phase = 2 if split else 0
        self._check(self._lib.obe_cycle(C.byref(cy)))
        self._after_cycle_c(resample)

    def _after_cycle_c(self, resample):
        """Host bookkeeping of run_cycle_async + resample() (+ the asynchronous constraint pass)."""
        self._invalidate()
        self._stats = None
        self._moments_valid = True
        self._weights_lazy = True
        if resample:
            self._epoch += 1
            self._last_ancestors = None
            self._buf, self._alt = self._alt, self._buf
            self._cloud_version += 1
            self._invalidate(particles=True)
            self._moments_valid = False
            self._weights_uniform = True
            self._weights_lazy = False
            self.just_resampled = True
            if self._cy.mask_le | self._cy.mask_lt:
                self._moments_valid = True
                self._weights_uniform = False
                self._weights_lazy = True
        if self._cy.drift:
            self._after_drift()

    def resample_select_async(self, resample=True, select=True):
        """The part of run_cycle_async after the update: (forced) resample and selection, enqueued without a host
        synchronisation.  With both on and early select available the K draws come from the resample plan and the
        utility pass overlaps the resample on the selection stream."""
        if self._pending_cycle:
            self._settle()
        if resample:
            if self.resampling == 'multinomial':
                raise ValueError('run_cycle_async needs a device-side resampler (systematic or multinomial_device)')
            if select and self._early_select_ok():
                self._resample_with_select()
                self._select_ready = False          # (the result is the caller's: best_index_dev)
                self.just_resampled = True
                return
            self.resample()
            self.just_resampled = True
            self._enforce_constraints_async()
        if self._drift_F is not None:
            self._apply_drift(self._pivot)
        if select:
            self._utility_dev_run()

    # ---- early select -------------------------------------------------------------------------
    def _early_select_ok(self):
        """Can the selection be taken from the resample plan?  Not with a drift, whose step comes after the
        resample; otherwise see _early_select_possible."""
        return self._drift_F is None and self._early_select_possible()

    def _early_select_possible(self):
        """Needs the one-kernel systematic resample, offspring that keep their uniform weights (no constraint mask), a
        utility that reads nothing the resample changes (no noise parameter), and no host-side upload inside the
        utility call (full KLD noise)."""
        if not self.early_select or self.resampling != 'systematic' or self._utility_code == 3:
            return False
        if not (1 <= self.N_DRAWS <= _lib.MAX_DRAWS) or self._noise_from_stats():
            return False
        return self._constraint_masks() == (0, 0)

    def _side_stream(self):
        side = self._side
        if side is None:
            st = self._torch.cuda.Stream(device=self._buf.device, priority=-1)
            side = self._side = (st, C.c_void_p(st.cuda_stream))
        return side

    def _pick_draws(self, u, draws, side_raw):
        """K offspring of the parked resample -> draws (d, K), on the selection stream."""
        self._check(self._lib.obe_resample_pick(_lib.dptr(u), int(len(u)), C.c_void_p(draws.data_ptr()), None, 0, 0, 0,
                                                side_raw))

    def _resample_with_select(self):
        """resample() with the following selection started from its plan: plan kernel -> [selection stream: pick the
        K draws, utility, argmax] || [main stream: stream the cloud] -> join.  No host synchronisation."""
        lib = self._lib
        main = self._stream()
        side_obj, side = self._side_stream()
        lib.obe_resample_defer(1)
        try:
            self.resample()                          # plan kernel only: the streaming kernel is parked
        except Exception:
            lib.obe_resample_defer(0)
            raise
        self._check(lib.obe_stream_fork(main, side))
        dd = self._draws_buffer()
        u = self.rng.random(self.N_DRAWS)
        self._pick_draws(u, dd, side)
        self._stream_override = side
        try:
            self._utility_dev_run(draws=dd, side=side_obj)
        finally:
            self._stream_override = None
        # (the streaming kernel leaves a few CTA slots free -- resample_reserve_ctas -- through which the selection
        # kernels run while it streams; it is persistent and would otherwise keep them out until it ends)
        self._check(lib.obe_resample_emit(main))
        self._check(lib.obe_stream_join(main, side))
        self._select_ready = True

    def _do_resample(self):
        if self.eager_select and self._early_select_ok():
            self._resample_with_select()
        else:
            self.resample()

    @property
    def best_index_dev(self):
        """Device tensor: [argmax index, bit pattern of its utility] of the last utility pass."""
        return self._best_dev

    def enforce_parameter_constraints(self):
        """Stub, as in the reference (obe_base.py:401-416).  Device-side constraints are data:
        see ``_apply_constraint_masks``."""
        if self._pending_cycle:
            self._settle()
        pass

    def _apply_constraint_masks(self, mask_le=0, mask_lt=0, sync=True):
        """weight <- 0 where x_j <= 0 (mask_le bit j) or x_j < 0 (mask_lt bit j), renormalise.
        ``sync=False`` only enqueues the masking pass (run_cycle_async): the stats stay on the device."""
        if sync:
            self._refresh(mask_le=mask_le, mask_lt=mask_lt, renormalise=1)
        else:
            ni = self._noise_index
            self._check(self._lib.obe_refresh(self._cs(), mask_le, mask_lt, _lib.iarr(ni), 0 if ni is None else len(ni),
                                              _lib.darr(self._pivot, _lib.MAX_PARAMS), 1, self._stream()))
            self._stats = None
            self._moments_valid = True      # on the device
            self._weights_uniform = False
        self._weights_lazy = True
        self._invalidate()

    def _constraint_masks(self):
        """(mask_le, mask_lt) of the constraint enforce_parameter_constraints applies; (0, 0): none."""
        return 0, 0

    def _enforce_constraints_async(self):
        """enforce_parameter_constraints without a host synchronisation (the masks are data)."""
        le, lt = self._constraint_masks()
        if le | lt:
            self._apply_constraint_masks(mask_le=le, mask_lt=lt, sync=False)

    def likelihood(self, y_model, measurement_record):
        """Likelihood of the record for every particle (obe_base.py:418-461), on the device, with the
        ``likelihood_model`` of the engine (choke included)."""
        torch = self._torch
        y_meas, sigma, noise_index, n_lik = self._likelihood_spec(measurement_record)
        tmp = self._buf.empty_like(share_particles=True)
        tmp.weights.fill_(1.0)
        tmp.stats[_lib.ST_INVS] = 1.0
        y = torch.zeros((self.n_channels, self._buf.ld), dtype=torch.float64, device=self._buf.device)
        y[:, :self.n_particles].copy_(torch.as_tensor(
            np.ascontiguousarray(np.asarray(y_model, dtype=np.float64).reshape(self.n_channels, -1))))
        use_choke = 0 if self.choke is None else 1
        self._check(self._lib.obe_update_from_y_model(self._model, C.byref(tmp.struct()), C.c_void_p(y.data_ptr()),
                                                      self._buf.ld, self.n_channels,
                                                      _lib.darr(y_meas, _lib.MAX_CHANNELS),
                                                      None if sigma is None else _lib.darr(sigma, _lib.MAX_CHANNELS),
                                                      _lib.iarr(noise_index), n_lik, use_choke,
                                                      0.0 if self.choke is None else float(self.choke),
                                                      _lib.darr(self._pivot, _lib.MAX_PARAMS), self._stream()))
        return tmp.weights[:self.n_particles].cpu().numpy()

    # ------------------------------------------------------------------------------------------
    # design half (obe_base.py:463-805)
    # ------------------------------------------------------------------------------------------
    @property
    def design_aux(self):
        """Per-channel aux of the likelihood-aware utility (``design_noise='likelihood'``): the planned trials of the
        next binomial measurement, the ``aux`` of a cuda_likelihood's ``noise_var``.  Read at every selection."""
        return self._design_aux

    @design_aux.setter
    def design_aux(self, value):
        arr = design_aux_array(value, self._design_lik, self.likelihood_model, self.n_channels)
        if getattr(self, '_utility_code', None) == 4 and self.likelihood_model == 'binomial':
            problem = _information_gain_aux_problem(arr)
            if problem:
                raise ValueError(problem)
        self._design_aux = value
        self._design_aux_arr = arr

    def _design_var_noise(self):
        """What the utility kernel divides by: the design aux for a likelihood-aware handle (whose kernel computes
        the noise variance itself), yvar_noise_model() otherwise."""
        if self._design_lik:
            return self._design_aux_arr
        return self.yvar_noise_model()

    def y_var_noise_model(self):
        return self.yvar_noise_model()

    def yvar_noise_model(self):
        """Constant noise variance per channel, (C,1) (obe_base.py:542-564)."""
        if self._pending_cycle:
            self._settle()
        return self.default_noise_std ** 2

    def cost_estimate(self):
        """1.0, or an array over settings in subclasses (obe_base.py:566-577)."""
        return 1.0

    def _noise_from_stats(self):
        return False

    def _draws_buffer(self):
        dd = getattr(self, '_draws_dev', None)
        if dd is None or dd.shape[1] != self.N_DRAWS:
            dd = self._draws_dev = self._torch.empty((self.n_dims, self.N_DRAWS), dtype=self._torch.float64,
                                                     device=self._buf.device)
        return dd

    def _utility_dev_run(self, draws=None, side=None):
        """draws -> utility over the grid -> argmax, all on the device; returns nothing.  ``draws``: already on the
        device (early select); ``side``: the torch stream the kernels go to when it is not the current one."""
        if self._pending_cycle:
            self._settle()
        torch = self._torch
        if draws is None:
            draws = self._randdraw_dev(self.N_DRAWS, out=self._draws_buffer())
        n_set = len(self.setting_indices)
        if self._noise_from_stats():
            if not self._moments_valid:     # (valid-on-device is enough: the kernel reads the stats block itself)
                self._ensure_moments()
            var_noise = None
            stats_ptr = C.c_void_p(self._buf.stats.data_ptr())
        else:
            vn = np.asarray(self._design_var_noise(), dtype=np.float64)
            key = vn.tobytes()
            cache = self._var_noise_cache
            if cache is None or cache[0] != key:
                cache = self._var_noise_cache = (key, _lib.darr(vn.reshape(-1), _lib.MAX_CHANNELS))
            var_noise = cache[1]
            stats_ptr = None
        cost = self.cost_estimate()
        cost_ptr = None
        if not (isinstance(cost, float) and cost == 1.0) and not (np.isscalar(cost) and float(cost) == 1.0):
            cost_arr = np.array(np.broadcast_to(np.asarray(cost, dtype=np.float64), (n_set,)))
            if self._cost_dev is None:
                self._cost_dev = torch.empty(n_set, dtype=torch.float64, device=self._buf.device)
            if side is not None:
                with torch.cuda.stream(side):            # the upload must precede the kernel on ITS stream
                    self._cost_dev.copy_(torch.from_numpy(np.ascontiguousarray(cost_arr)))
            else:
                self._cost_dev.copy_(torch.from_numpy(np.ascontiguousarray(cost_arr)))
            cost_ptr = C.c_void_p(self._cost_dev.data_ptr())
        self._check(self._lib.obe_utility(self._model, C.c_void_p(draws.data_ptr()), int(self.N_DRAWS),
                                          C.c_void_p(self._settings_dev.data_ptr()), self._lds, n_set, self._cons_arr,
                                          var_noise, stats_ptr, cost_ptr, self._utility_code,
                                          1 if self.utility_log_form else 0, self._kld_noise_ptr(),
                                          C.c_void_p(self._utility_dev.data_ptr()),
                                          C.c_void_p(self._best_dev.data_ptr()),
                                          C.c_void_p(self._select_scratch.data_ptr()), self._stream()))

    def _kld_noise_ptr(self):
        """full_kld_utility (obe_base.py:706-711): K*C standard normals from the module-level Generator,
        scaled by the noise model; uploaded for the kernel.  None for the other methods."""
        if self._utility_code != 3:
            return None
        nva = rng.normal(0, 1.0, self.N_DRAWS * self.n_channels)
        nvb = nva.reshape((self.n_channels, self.N_DRAWS))
        noisevalues = np.ascontiguousarray((nvb * np.sqrt(np.asarray(self.yvar_noise_model(), dtype=np.float64))).T)
        self._kld_noise_host = noisevalues
        self._kld_noise_dev = self._torch.from_numpy(noisevalues).to(self._buf.device)
        return C.c_void_p(self._kld_noise_dev.data_ptr())

    def utility(self):
        """Utility over all settings as a numpy array (obe_base.py:579-655)."""
        if self._pending_cycle:
            self._settle()
        self._utility_dev_run()
        return self._utility_dev.cpu().numpy()

    def _utility_as(self, code):
        """The utility of method `code` whatever ``utility_method`` the engine was built with."""
        if code == 3 and self.n_channels != 1:
            raise ValueError('full_kld_utility supports single-channel models')
        if code == 3 and self._design_lik:
            raise ValueError("full_kld_utility is not available with design_noise='likelihood': its noise samples "
                             'are Gaussian draws')
        if code == 4:
            problem = _information_gain_problem(self.likelihood_model, self._design_lik, self.n_channels,
                                                self._design_aux_arr)
            if problem:
                raise ValueError(problem)
        saved = self._utility_code
        self._utility_code = code
        try:
            return self.utility()
        finally:
            self._utility_code = saved

    def utility_variance(self):
        """Variance-based utility (obe_base.py:628-655)."""
        return self._utility_as(0)

    def utility_max_min(self):
        """(max - min over the draws)^2 / noise variance (obe_base.py:602-626)."""
        return self._utility_as(1)

    def utility_pseudo(self):
        """Entropy-based pseudo-variance utility (obe_base.py:657-686)."""
        return self._utility_as(2)

    def utility_full_kld(self):
        """Full Kullback-Leibler utility (obe_base.py:688-720)."""
        return self._utility_as(3)

    def utility_information_gain(self):
        """Expected information gain of the next measurement at every setting, in nats: the mutual information
        between the parameters (uniform over the K drawn sets) and the count,
        ``I(s) = (1/K) sum_k sum_y p_k(y) log(p_k(y) / pbar(y))``, ``pbar = (1/K) sum_j p_j``, in ``[0, log K]``.

        The sum over y is exact: it runs over the union of the draws' count windows, each wide enough that the
        mass it leaves out is below 1e-17, so a setting costs about K times that many pmf terms.  A setting where
        some draw's output is impossible for the likelihood gets 0, and identical draws give 0.  Divided by
        ``cost_estimate()``; ``utility_log_form`` is ignored.  For a ``cuda_likelihood`` with a ``window`` the sum
        runs over the union of the declared windows (see :func:`~optbayesexpt_b200.cuda_likelihood`).  Raises
        ``ValueError`` unless the engine has a Poisson or binomial likelihood, or a cuda_likelihood with a window,
        with ``design_noise='likelihood'``, one channel and, for binomial, an integer ``design_aux >= 1``."""
        return self._utility_as(4)

    def opt_setting(self):
        """Setting with the maximum utility (obe_base.py:733-756)."""
        synced = self._settle()
        if self._select_ready:
            self._select_ready = False          # started by the resample (eager_select): only the argmax is fetched
        else:
            self._utility_dev_run()
            self._best_copied = False
        if self._best_copied:                   # the cycle entry already put it into the pinned block
            self._best_copied = False
            if not synced:
                self._wait_cycle()
            bestindex = int(self._cy_best_np[0])
        else:
            self._best_host.copy_(self._best_dev, non_blocking=True)
            self._check(self._lib.obe_stream_sync(self._stream()))
            bestindex = int(self._best_host_np[0])
        self.last_setting_index = bestindex
        return tuple(self.allsettings[:, bestindex])

    def good_setting(self, pickiness=None):
        """Setting drawn with probability ~ utility**pickiness (obe_base.py:758-789)."""
        if pickiness is None:
            pickiness = self.pickiness
        self._settle()
        if self._select_ready:
            self._select_ready = False
        else:
            self._utility_dev_run()
        self._best_copied = False
        u = float(self.rng.random())
        self._check(self._lib.obe_pick(C.c_void_p(self._utility_dev.data_ptr()), len(self.setting_indices),
                                       float(pickiness), u, C.c_void_p(self._pick_dev.data_ptr()),
                                       C.c_void_p(self._select_scratch.data_ptr()), self._stream()))
        goodindex = int(self._pick_dev.item())
        self.last_setting_index = goodindex
        return tuple(self.allsettings[:, goodindex])

    def random_setting(self):
        """Uniformly random setting (obe_base.py:791-805)."""
        settingindex = rng.choice(self.setting_indices)
        self.last_setting_index = settingindex
        return self.allsettings[:, settingindex]
