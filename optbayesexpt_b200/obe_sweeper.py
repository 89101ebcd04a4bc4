"""OptBayesExptSweeper on the GPU (reference: demos/sweeper/obe_sweeper.py, v1.2.0).

For instruments that sweep a setting: the design half proposes (start, stop) index pairs into the
first setting array, the inference half digests the array of values a sweep returned.  The point
utility never leaves the device: ``obe_sweep_utility`` integrates it along the swept setting
(cumsum), evaluates every (start, stop) pair and takes the argmax in two launches.
"""
import ctypes as C

import numpy as np

from . import _lib
from .obe_noiseparam import OptBayesExptNoiseParameter

try:
    rng = np.random.default_rng()        # module-level Generator, as in the reference (obe_sweeper.py:3-6)
except AttributeError:                   # pragma: no cover
    rng = np.random


class OptBayesExptSweeper(OptBayesExptNoiseParameter):
    """An OptBayesExpt class for instruments that sweep a parameter (obe_sweeper.py:9-85).

    Same constructor as the reference.  Attributes: ``sweep_settings``, ``start_stop_subsample`` (3),
    ``start_stop_indices`` (P, 2), ``start_stop_choice_indices``, ``start_stop_values``,
    ``cost_of_new_sweep`` (5.0).
    """

    _drift_refusal = ('OptBayesExptSweeper does not take drift: its fused multi-point update would need a transition '
                      'between the points of a sweep')

    def __init__(self, model_function, setting_values, parameter_samples, constants, noise_parameter_index,
                 **kwargs):
        if kwargs.get('drift') is not None:           # (before anything reaches the device)
            raise ValueError(self._drift_refusal)
        OptBayesExptNoiseParameter.__init__(self, model_function, setting_values, parameter_samples, constants,
                                            noise_parameter_index=noise_parameter_index, **kwargs)
        self.sweep_settings = np.asarray(setting_values[0])
        self.start_stop_subsample = 3
        self.start_stop_indices = self._generate_start_stop_indices()
        self.start_stop_choice_indices = np.arange(len(self.start_stop_indices), dtype=int)
        self.start_stop_values = self.sweep_settings[self.start_stop_indices]
        self.cost_of_new_sweep = 5.
        #: True: a sweep is digested by the multi-point kernel (one pass over the cloud per segment between
        #: resamples); False: one update launch per point, literally as the reference loops.
        self.fused_sweep = True
        self._pairs_host = None
        self._pairs_dev = None
        self._multi_w = None
        self._sigma_ref = None
        self._sweep_chunk = 16

    def _install(self, samples):
        # a new cloud (set_pdf) invalidates everything sized or scaled for the old one: the spare weight row of
        # the multi-point kernel and the noise scale taken from the last committed cloud
        OptBayesExptNoiseParameter._install(self, samples)
        self._multi_w = None
        self._sigma_ref = None

    # ---- inference half
    def pdf_update(self, measurement_record):
        """Bayesian inference on a swept measurement (obe_sweeper.py:87-101): one noise-parameter update per
        point of the sweep, the resample test after every point, exactly as in the reference.  With
        ``fused_sweep`` (default) the points between two resamples are one pass over the cloud."""
        (setting_values,), result_values = measurement_record
        if self.fused_sweep and len(setting_values) > 1:
            return self._pdf_update_fused(np.asarray(setting_values, dtype=np.float64), result_values)
        out = None
        for setting, result in zip(setting_values, result_values):
            out = OptBayesExptNoiseParameter.pdf_update(self, ((setting,), result))
        return out

    def _multi_update(self, xs, ys):
        """Launch the multi-point kernel on points (xs, ys) -> (first firing point or -1, its N_eff/n)."""
        torch = self._torch
        m = len(xs)
        rec = np.zeros((m, 12))
        rec[:, 0] = xs
        y = np.asarray(ys, dtype=np.float64).reshape(m, -1)
        n_lik = min(self.n_channels, y.shape[1])
        rec[:, 4:4 + n_lik] = y[:, :n_lik]
        dev = self._buf.device
        if self._multi_w is None:
            self._multi_w = torch.zeros(self._buf.ld, dtype=torch.float64, device=dev)
            self._multi_rec = torch.zeros((_lib.MULTI_MAX, 12), dtype=torch.float64, device=dev)
            self._multi_sums = torch.zeros((_lib.MULTI_MAX, 2), dtype=torch.float64, device=dev)
            self._multi_res = torch.zeros(2, dtype=torch.float64, device=dev)
            self._multi_res_host = torch.zeros(2, dtype=torch.float64).pin_memory()
        self._multi_rec[:m].copy_(torch.from_numpy(rec))
        # particle-independent scale of 1/sigma: the rms noise estimate of the last committed cloud
        if self._sigma_ref is None:
            self._sigma_ref = self._rms_noise(self._ensure_moments())
        scale = self._sigma_ref
        thr = 0.0
        if self.tuning_parameters['auto_resample']:
            thr = max(0.1, float(self.tuning_parameters['resample_threshold']))
        self._check(self._lib.obe_update_multi(
            self._model, self._cs(), C.c_void_p(self._multi_w.data_ptr()), C.c_void_p(self._multi_rec.data_ptr()), m,
            self._cons_arr, _lib.iarr(self._noise_index[:n_lik]), n_lik, _lib.darr(scale, _lib.MAX_CHANNELS),
            0 if self.choke is None else 1, 0.0 if self.choke is None else float(self.choke), thr,
            self.n_particles, C.c_void_p(self._multi_sums.data_ptr()), C.c_void_p(self._multi_res.data_ptr()),
            self._stream()))
        self._multi_res_host.copy_(self._multi_res, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return int(self._multi_res_host[0]), float(self._multi_res_host[1])

    def _commit_multi(self):
        """The row the multi-point kernel wrote becomes the cloud's weight row; stats, CDF prefix and moments
        are rebuilt from it (one refresh pass)."""
        self._buf.weights, self._multi_w = self._multi_w, self._buf.weights
        self._buf._struct = None
        self._buf.stats[_lib.ST_UNIFORM] = 0.0          # the weight row is explicit
        self._invalidate()
        self._stats = None
        self._weights_uniform = False
        self._weights_lazy = True
        self._moments_valid = False
        self._sigma_ref = self._rms_noise(self._refresh(renormalise=1))

    def _rms_noise(self, st):
        """sqrt of the weighted mean of sigma^2 per channel (obe_noiseparam.py:132-136), 1 where undefined."""
        scale = np.ones(_lib.MAX_CHANNELS)
        c = self.n_channels
        with np.errstate(all='ignore'):
            s2 = st[_lib.ST_NOISE:_lib.ST_NOISE + c] / st[_lib.ST_SUMT]
        ok = np.isfinite(s2) & (s2 > 0)
        scale[:c][ok] = np.sqrt(s2[ok])
        return scale

    def _pdf_update_fused(self, xs, ys):
        """Segments of the sweep between resamples, each one multi-point launch.  A launch that ran past the
        point where the resample test fires is wasted work (it is redone up to that point), so the number of
        points per launch follows the distance between resamples seen so far."""
        import warnings
        ys = list(ys)
        i, m_total = 0, len(xs)
        # Without the resample test (auto_resample off) nothing renormalises the running product inside a launch --
        # the reference renormalises after every point -- so a launch is kept to a few points: the product of 8
        # particle-independent-scaled likelihoods cannot underflow for every particle at once, 128 of them can.
        cap = _lib.MULTI_MAX if self.tuning_parameters['auto_resample'] else 8
        while i < m_total:
            j = min(i + max(1, min(self._sweep_chunk, cap)), m_total)
            first, ratio = self._multi_update(xs[i:j], ys[i:j])
            if first < 0:
                self._commit_multi()
                self.just_resampled = False
                self._sweep_chunk = min(2 * self._sweep_chunk, _lib.MULTI_MAX)
                i = j
                continue
            if first != j - i - 1:                      # the weights on the device ran past the resample point
                again, ratio = self._multi_update(xs[i:i + first + 1], ys[i:i + first + 1])
                if again != first:
                    raise RuntimeError('multi-point update is not reproducible')
                self._sweep_chunk = max(4, first + 1)
            self._commit_multi()
            if ratio < 0.1:
                warnings.warn("\nParticle filter rejected > 90 % of particles. "
                              f"N_eff = {ratio * self.n_particles:.2f}. "
                              "Particle impoverishment may lead to errors.", RuntimeWarning)
            self.resample()
            self.just_resampled = True
            self.enforce_parameter_constraints()
            i += first + 1
        from .obe_base import LazyDeviceArray
        return (LazyDeviceArray(lambda: self.particles), LazyDeviceArray(lambda: self.particle_weights))

    # ---- design half
    def cost_estimate(self):
        """Pointwise costs are uniform along the sweep (obe_sweeper.py:103-105)."""
        return 1.0

    def sweep_cost_estimate(self):
        """(stop - start) + cost_of_new_sweep per pair (obe_sweeper.py:107-121)."""
        return self.start_stop_indices[:, 1] - self.start_stop_indices[:, 0] + self.cost_of_new_sweep

    def _sync_pairs(self):
        """Device copy of ``start_stop_indices`` (int32), refreshed when the attribute was replaced."""
        torch = self._torch
        pairs = np.ascontiguousarray(np.asarray(self.start_stop_indices, dtype=np.int32))
        if pairs.ndim != 2 or pairs.shape[1] != 2 or len(pairs) == 0:
            raise ValueError('start_stop_indices must have shape (n_pairs, 2)')
        n_set = len(self.setting_indices)
        if pairs.min() < 0 or pairs.max() >= n_set:
            raise ValueError('start_stop_indices out of range of the swept setting')
        if self._pairs_host is None or self._pairs_host.shape != pairs.shape or not np.array_equal(self._pairs_host, pairs):
            dev = self._buf.device
            self._pairs_host = pairs.copy()
            self._pairs_dev = torch.from_numpy(pairs).to(dev)
            self._cumsum_dev = torch.empty(n_set, dtype=torch.float64, device=dev)
            self._pair_utility_dev = torch.empty(len(pairs), dtype=torch.float64, device=dev)
            self._pair_best_dev = torch.zeros(2, dtype=torch.int64, device=dev)
            self._pair_best_host = torch.zeros(2, dtype=torch.int64).pin_memory()
            self._pair_pick_dev = torch.zeros(1, dtype=torch.int64, device=dev)
            self._pair_scratch = torch.zeros(int(self._lib.obe_select_scratch_bytes(len(pairs))), dtype=torch.uint8,
                                             device=dev)
        return len(pairs)

    def _sweep_utility_dev_run(self):
        """point utility -> cumsum -> pair utilities + argmax, all on the device."""
        n_pairs = self._sync_pairs()
        self._utility_dev_run()
        self._check(self._lib.obe_sweep_utility(
            C.c_void_p(self._utility_dev.data_ptr()), len(self.setting_indices), C.c_void_p(self._pairs_dev.data_ptr()),
            n_pairs, float(self.cost_of_new_sweep), C.c_void_p(self._cumsum_dev.data_ptr()),
            C.c_void_p(self._pair_utility_dev.data_ptr()), C.c_void_p(self._pair_best_dev.data_ptr()),
            C.c_void_p(self._select_scratch.data_ptr()), self._stream()))
        return n_pairs

    def sweep_utility(self):
        """Utility of every (start, stop) pair as a numpy array (obe_sweeper.py:123-151)."""
        self._sweep_utility_dev_run()
        return self._pair_utility_dev.cpu().numpy()

    def opt_setting(self):
        """The (start, stop) index pair with the maximum utility (obe_sweeper.py:153-169)."""
        self._sweep_utility_dev_run()
        self._pair_best_host.copy_(self._pair_best_dev, non_blocking=True)
        self._torch.cuda.current_stream().synchronize()
        index = int(self._pair_best_host[0])
        self.last_setting_index = index
        return self.start_stop_indices[index]

    def good_setting(self, pickiness=None):
        """Pair drawn with probability ~ sweep_utility**pickiness (obe_sweeper.py:171-198; the reference
        ignores its argument and uses ``self.pickiness``, which is also the default here)."""
        if pickiness is None:
            pickiness = self.pickiness
        n_pairs = self._sweep_utility_dev_run()
        u = float(rng.random())
        self._check(self._lib.obe_pick(C.c_void_p(self._pair_utility_dev.data_ptr()), n_pairs, float(pickiness), u,
                                       C.c_void_p(self._pair_pick_dev.data_ptr()),
                                       C.c_void_p(self._pair_scratch.data_ptr()), self._stream()))
        index = int(self._pair_pick_dev.item())
        self.last_setting_index = index
        return self.start_stop_indices[index]

    def random_setting(self):
        """Uniformly random (start, stop) pair (obe_sweeper.py:200-211)."""
        index = rng.choice(self.start_stop_choice_indices)
        self.last_setting_index = index
        return self.start_stop_indices[index]

    def _generate_start_stop_indices(self):
        """Valid [start, stop] index combinations, stop > start, on every ``start_stop_subsample``-th
        setting plus the last one (obe_sweeper.py:213-232)."""
        raw_length = len(self.sweep_settings)
        sub = list(range(0, raw_length, int(self.start_stop_subsample)))
        if sub[-1] != raw_length - 1:
            sub.append(raw_length - 1)
        m = len(sub)
        i, j = np.triu_indices(m, k=1)
        sub = np.asarray(sub, dtype=np.int64)
        return np.stack((sub[i], sub[j]), axis=1)
