"""Device functors for ``model_function``.

The reference takes a Python callable ``model(sets, pars, cons)`` (obe_base.py:50-66).  A Python
callable cannot run inside a CUDA kernel, so here the model is a :class:`DeviceModel`: either a
built-in functor compiled into libobe_b200.so (the demo models of the reference) or user CUDA
source compiled by NVRTC for sm_100a.  A DeviceModel is still *callable* with the reference's
``(sets, pars, cons)`` contract in both broadcast orientations -- the call runs the
``eval_over_all_*`` kernels on the GPU, so helpers such as a measurement simulator keep working.
"""
import ctypes as C

import numpy as np

from . import _lib

BUILTIN_INFO = {
    # name: (n_settings, n_model_params, n_constants, n_channels)
    'lorentzian_hwhm': (1, 3, 1, 1),   # demos/find_peak/sequentialLorentzian.py:66-75
    'lorentzian_fwhm': (1, 3, 1, 1),   # demos/numba/numbaLorentzian.py:104
    'lorentzian_4p': (1, 4, 0, 1),     # demos/find_peak/seqLor_pdfevolve.py:28
    'lorentzian_dip': (1, 3, 0, 1),    # demos/server/server_script.py:33
    'line': (1, 2, 0, 1),              # demos/line_plus_noise/line_plus_noise.py:54
    'rabi': (2, 2, 3, 1),              # demos/pipulse/pipulse.py:18-49
    'lockin_coil': (1, 3, 0, 2),       # demos/lockin/lockin_of_coil.py:63-102
}


class DeviceModel:
    """A measurement model that lives on the GPU.

    Use :func:`builtin` or :func:`cuda_source` to make one.  Handles are created per
    ``n_params`` (the number of rows of the particle cloud, which may exceed the number of
    parameters the model itself reads, e.g. a trailing noise parameter).
    """

    def __init__(self, name, n_settings, n_model_params, n_constants, n_channels, source=None, entry=None,
                 likelihood='gaussian', design_noise='fixed'):
        self.name = name
        self.n_settings = n_settings
        self.n_model_params = n_model_params
        self.n_constants = n_constants
        self.n_channels = n_channels
        self.source = source
        self.entry = entry
        #: measurement likelihood of the update kernels: 'gaussian', 'poisson', 'binomial' or a CudaLikelihood
        self.likelihood = likelihood
        #: noise variance of the utility kernel: 'fixed' (the engine's yvar_noise_model()) or 'likelihood' (the
        #: likelihood's own variance at each setting; non-Gaussian likelihoods only)
        self.design_noise = design_noise
        self._handles = {}
        self._variants = {}
        self.compile_log = ''

    def with_likelihood(self, likelihood, design_noise='fixed'):
        """The same model with another measurement likelihood ('gaussian', 'poisson', 'binomial' or
        :func:`cuda_likelihood`).  A non-Gaussian model is compiled by NVRTC on first use.

        ``design_noise='likelihood'`` gives the variant whose utility kernel divides by the likelihood's own noise
        variance (see ``OptBayesExpt(..., design_noise=)``); a Gaussian model has only the 'fixed' one."""
        if isinstance(likelihood, str):
            if likelihood not in LIKELIHOODS:
                raise ValueError(f'unknown likelihood_model {likelihood!r}; have {list(LIKELIHOODS)} or cuda_likelihood(...)')
        elif not isinstance(likelihood, CudaLikelihood):
            raise TypeError('likelihood_model must be one of '
                            f'{list(LIKELIHOODS)} or optbayesexpt_b200.cuda_likelihood(source, entry)')
        if design_noise not in DESIGN_NOISES:
            raise ValueError(f'design_noise must be one of {list(DESIGN_NOISES)}, got {design_noise!r}')
        if likelihood == 'gaussian':
            design_noise = 'fixed'                  # (the Gaussian noise variance is the fixed one by definition)
        elif design_noise == 'likelihood' and isinstance(likelihood, CudaLikelihood) and likelihood.noise_var is None:
            raise ValueError("design_noise='likelihood' with a cuda_likelihood needs its noise_var entry: "
                             'cuda_likelihood(source, entry, noise_var=...)')
        if likelihood == self.likelihood and design_noise == self.design_noise:
            return self
        key = (likelihood, design_noise)
        if key not in self._variants:               # (one NVRTC compile per variant and n_params)
            self._variants[key] = DeviceModel(self.name, self.n_settings, self.n_model_params, self.n_constants,
                                              self.n_channels, source=self.source, entry=self.entry,
                                              likelihood=likelihood, design_noise=design_noise)
        return self._variants[key]

    def handle(self, n_params):
        """obe_model_t for a cloud with ``n_params`` rows."""
        if n_params in self._handles:
            return self._handles[n_params]
        lib = _lib.load()
        if n_params < self.n_model_params:
            raise ValueError(f'model {self.name} reads {self.n_model_params} parameters, cloud has {n_params}')
        h = C.c_void_p()
        if self.likelihood != 'gaussian':
            log = C.create_string_buffer(1 << 16)
            user = isinstance(self.likelihood, CudaLikelihood)
            args = (self.name.encode() if self.source is None else None,
                    None if self.source is None else self.source.encode(),
                    None if self.source is None else self.entry.encode(),
                    self.n_settings, n_params, self.n_model_params, self.n_constants, self.n_channels,
                    b'user' if user else self.likelihood.encode(),
                    self.likelihood.source.encode() if user else None,
                    self.likelihood.entry.encode() if user else None)
            if self.design_noise == 'likelihood':
                nv = self.likelihood.noise_var.encode() if user else None
                rc = lib.obe_model_compile_likelihood_design(*args, nv, C.byref(h), log, len(log))
            else:
                rc = lib.obe_model_compile_likelihood(*args, C.byref(h), log, len(log))
            self.compile_log = log.value.decode(errors='replace')
            _lib.check(rc)
        elif self.source is None:
            _lib.check(lib.obe_model_builtin(self.name.encode(), n_params, C.byref(h)))
        else:
            log = C.create_string_buffer(1 << 16)
            rc = lib.obe_model_compile(self.source.encode(), self.entry.encode(), self.n_settings, n_params,
                                       self.n_model_params, self.n_constants, self.n_channels, C.byref(h),
                                       log, len(log))
            self.compile_log = log.value.decode(errors='replace')
            _lib.check(rc)
        self._handles[n_params] = h
        return h

    # ---- the reference's calling convention, evaluated on the device -------------------------
    def __call__(self, sets, pars, cons):
        import torch
        lib = _lib.require_device()
        sets = [np.asarray(s, dtype=np.float64) for s in sets]
        pars = [np.asarray(p, dtype=np.float64) for p in pars]
        cons = [float(c) for c in cons]
        set_n = max([s.size for s in sets] + [1])
        par_n = max([p.size for p in pars] + [1])
        set_scalar = all(s.ndim == 0 or s.size == 1 for s in sets)
        par_scalar = all(p.ndim == 0 or p.size == 1 for p in pars)
        if not (set_scalar or par_scalar):
            raise ValueError('model(sets, pars, cons): either the settings or the parameters must be scalars')
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        if par_scalar:
            # arrays of settings x one parameter set  (obe_base.py:338)
            shape = np.broadcast(*sets).shape if sets else ()
            n = int(np.prod(shape)) if shape else 1
            grid = np.stack([np.broadcast_to(s, shape).reshape(-1) for s in sets]) if sets else np.zeros((0, n))
            ld = n + (n & 1)
            sdev = torch.zeros((max(len(sets), 1), ld), dtype=torch.float64, device='cuda')
            if len(sets):
                sdev[:len(sets), :n] = torch.from_numpy(np.ascontiguousarray(grid))
            y = torch.empty((self.n_channels, ld), dtype=torch.float64, device='cuda')
            h = self.handle(max(len(pars), self.n_model_params))
            _lib.check(lib.obe_eval_settings(h, C.c_void_p(sdev.data_ptr()), ld, n,
                                             _lib.darr([p.reshape(-1)[0] for p in pars], _lib.MAX_PARAMS),
                                             _lib.darr(cons, _lib.MAX_CONSTANTS),
                                             C.c_void_p(y.data_ptr()), ld, stream))
            out = y[:, :n].cpu().numpy().reshape((self.n_channels,) + tuple(shape))
        else:
            # one setting x arrays of parameters  (obe_base.py:320)
            shape = np.broadcast(*pars).shape
            n = int(np.prod(shape))
            cloud = ParticleBuffers(np.stack([np.broadcast_to(p, shape).reshape(-1) for p in pars]))
            y = torch.empty((self.n_channels, cloud.ld), dtype=torch.float64, device='cuda')
            h = self.handle(len(pars))
            _lib.check(lib.obe_eval_parameters(h, C.byref(cloud.struct()),
                                               _lib.darr([s.reshape(-1)[0] for s in sets], _lib.MAX_SETTINGS),
                                               _lib.darr(cons, _lib.MAX_CONSTANTS),
                                               C.c_void_p(y.data_ptr()), cloud.ld, stream))
            out = y[:, :n].cpu().numpy().reshape((self.n_channels,) + tuple(shape))
        if self.n_channels == 1:
            out = out[0]
            if out.shape == ():
                return float(out)
        return out

    def __repr__(self):
        kind = 'builtin' if self.source is None else 'nvrtc'
        lik = '' if self.likelihood == 'gaussian' else f', likelihood={self.likelihood!r}'
        if self.design_noise != 'fixed':
            lik += f', design_noise={self.design_noise!r}'
        return (f'DeviceModel({self.name!r}, {kind}, settings={self.n_settings}, params={self.n_model_params}, '
                f'constants={self.n_constants}, channels={self.n_channels}{lik})')


#: the measurement likelihoods of the update kernel, by name (a user likelihood is a :func:`cuda_likelihood`)
LIKELIHOODS = ('gaussian', 'poisson', 'binomial')
#: the noise variance the utility divides by: the engine's fixed one, or the likelihood's own at each setting
DESIGN_NOISES = ('fixed', 'likelihood')


class CudaLikelihood:
    """A measurement likelihood as CUDA source: see :func:`cuda_likelihood`."""

    def __init__(self, source, entry, noise_var=None):
        self.source = source
        self.entry = entry
        self.noise_var = noise_var

    def __eq__(self, other):
        return isinstance(other, CudaLikelihood) and \
            (self.source, self.entry, self.noise_var) == (other.source, other.entry, other.noise_var)

    def __hash__(self):
        return hash((self.source, self.entry, self.noise_var))

    def __repr__(self):
        nv = '' if self.noise_var is None else f', noise_var={self.noise_var!r}'
        return f'cuda_likelihood(entry={self.entry!r}{nv})'


def non_gaussian(measurement_model, likelihood_model=None):
    """True when an engine built from these arguments would use a non-Gaussian likelihood."""
    if likelihood_model is not None:
        return likelihood_model != 'gaussian'
    return isinstance(measurement_model, DeviceModel) and measurement_model.likelihood != 'gaussian'


def cuda_likelihood(source, entry, noise_var=None):
    """User measurement likelihood for ``OptBayesExpt(..., likelihood_model=...)``, compiled by NVRTC with the model.

    ``source`` must define ``__device__ double <entry>(const double* y_model, const double* y_meas,
    const double* aux, int n_channels)`` returning the LOG-likelihood of the record for one particle:
    ``y_model`` are the model outputs, ``y_meas`` the record's second element and ``aux`` its third (a noise
    level, trial counts, anything per channel), both cut to ``n_channels`` entries.  The weight factor is
    ``exp(choke * log L)``; log L may be positive.  This replaces overriding ``likelihood`` in Python, which
    cannot run inside the update kernel.

    ``noise_var`` (optional) names a second function of ``source``, ``__device__ double <noise_var>(double y_model,
    double aux)``: the variance of one channel's measurement given its model output and the design aux.  It is
    what ``OptBayesExpt(..., design_noise='likelihood')`` divides the utility by (averaged over the draws), and
    that mode requires it.  A negative or NaN value marks the output as impossible: the setting's utility is 0.
    """
    return CudaLikelihood(source, entry, noise_var)


def builtin(name):
    """One of the reference's demo models as a pre-compiled device functor."""
    if name not in BUILTIN_INFO:
        raise KeyError(f'unknown built-in model {name!r}; have {sorted(BUILTIN_INFO)}')
    ns, npm, nc, nch = BUILTIN_INFO[name]
    return DeviceModel(name, ns, npm, nc, nch)


def cuda_source(source, entry, n_settings, n_params, n_constants=0, n_channels=1):
    """User model as CUDA source, compiled by NVRTC for sm_100a on first use.

    ``source`` must define ``__device__ void <entry>(const double* s, const double* p,
    const double* c, double* y)`` writing ``n_channels`` outputs.  The helpers of
    csrc/obe_device.cuh (``obe_add/obe_mul/obe_div`` ...) are available.
    """
    return DeviceModel(f'user:{entry}', n_settings, n_params, n_constants, n_channels, source=source, entry=entry)


def resolve_device(device=None):
    """The CUDA device an engine lives on.  The C library launches on the CURRENT device and its streams (one
    process per GPU is the design), so an explicit ``device=`` must name the current device: anything else would
    run GPU-0 kernels on GPU-1 memory.  Select the GPU with ``torch.cuda.set_device`` before building an engine."""
    import torch
    cur = torch.cuda.current_device()
    dev = torch.device(device if device is not None else f'cuda:{cur}')
    if dev.type != 'cuda':
        raise ValueError(f'optbayesexpt_b200 engines live on a CUDA device, got {dev}')
    index = cur if dev.index is None else dev.index
    if index != cur:
        raise ValueError(f'device={dev} is not the current CUDA device (cuda:{cur}): call torch.cuda.set_device({index}) '
                         'first -- the kernels are launched on the current device and its stream')
    return torch.device('cuda', index)


class ParticleBuffers:
    """Device buffers of one particle cloud + the obe_cloud_t that describes them."""

    def __init__(self, particles, device=None, capacity=None):
        import torch
        lib = _lib.require_device()
        if isinstance(particles, torch.Tensor):
            src = particles.to(dtype=torch.float64)
            d, n = src.shape
        else:
            src = np.ascontiguousarray(np.atleast_2d(np.asarray(particles, dtype=np.float64)))
            d, n = src.shape
        if not (1 <= d <= _lib.MAX_PARAMS):
            raise ValueError(f'n_dims must be 1..{_lib.MAX_PARAMS}, got {d}')
        if n < 1:
            raise ValueError('empty particle cloud')
        self.device = resolve_device(device)
        self.n, self.d = int(n), int(d)
        cap = max(int(capacity or 0), self.n)      # shards of a multi-GPU cloud change length
        self.ld = cap + (cap & 1)
        nt = int(lib.obe_num_tiles(self.ld))
        self.n_tiles = nt
        f64 = dict(dtype=torch.float64, device=self.device)
        self.particles = torch.zeros((self.d, self.ld), **f64)
        if isinstance(src, torch.Tensor):
            self.particles[:, :self.n].copy_(src)
        else:
            self.particles[:, :self.n].copy_(torch.from_numpy(src))
        self.weights = torch.zeros(self.ld, **f64)
        self.tile_sums = torch.zeros(nt, **f64)
        self.tile_prefix = torch.zeros(nt + 1, **f64)
        self.stats = torch.zeros(_lib.STATS_LEN, **f64)
        self.scratch = torch.zeros(int(lib.obe_scratch_bytes(self.ld)), dtype=torch.uint8, device=self.device)
        self._struct = None

    def empty_like(self, share_particles=False):
        """A second buffer set of the same geometry (resample is out-of-place)."""
        import torch
        other = object.__new__(ParticleBuffers)
        other.device, other.n, other.d, other.ld, other.n_tiles = self.device, self.n, self.d, self.ld, self.n_tiles
        other.particles = self.particles if share_particles else torch.zeros_like(self.particles)
        other.weights = torch.zeros_like(self.weights)
        other.tile_sums = torch.zeros_like(self.tile_sums)
        other.tile_prefix = torch.zeros_like(self.tile_prefix)
        other.stats = torch.zeros_like(self.stats)
        other.scratch = torch.zeros_like(self.scratch)
        other._struct = None
        if getattr(self, 'n_dev', None) is not None:
            other.n_dev = self.n_dev.clone()
        return other

    def enable_device_count(self):
        """Keep the live particle count in a device int64 (sharded clouds): `n` becomes a bound."""
        import torch
        self.n_dev = torch.tensor([self.n], dtype=torch.int64, device=self.device)
        self.n = self.ld            # the struct's n is now only the bound the grids are sized for
        self._struct = None

    def resize(self, n):
        """Change the live length (<= capacity); buffers are untouched."""
        if n > self.ld:
            raise ValueError(f'shard of {n} particles exceeds the buffer capacity {self.ld}')
        self.n = int(n)
        self._struct = None

    def struct(self):
        if self._struct is None:
            n_dev = getattr(self, 'n_dev', None)
            self._struct = _lib.Cloud(self.particles.data_ptr(), self.weights.data_ptr(),
                                      self.tile_sums.data_ptr(), self.tile_prefix.data_ptr(),
                                      self.stats.data_ptr(), self.scratch.data_ptr(),
                                      self.n, self.ld, self.d, 0,
                                      None if n_dev is None else n_dev.data_ptr())
            self._ptr = C.pointer(self._struct)
        return self._struct

    def ptr(self):
        """ctypes pointer to struct() (cached with it: the cycle entry takes one per buffer and call)."""
        self.struct()
        return self._ptr
