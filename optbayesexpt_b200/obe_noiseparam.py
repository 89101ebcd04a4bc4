"""OptBayesExptNoiseParameter on the GPU (reference: optbayesexpt/obe_noiseparam.py v1.2.0).

The measurement noise sigma is one (or, per channel, several) of the particle coordinates:
the fused update kernel reads sigma_c from row ``noise_parameter_index[c]`` of the cloud, the
utility kernel takes its noise variance from the weighted mean of sigma^2 accumulated in the same
pass, and the positivity constraint is applied as a bit mask by the refresh kernel.
"""
import numpy as np

from .obe_base import OptBayesExpt
from .models import non_gaussian as _non_gaussian


class OptBayesExptNoiseParameter(OptBayesExpt):
    """OptBayesExpt with unknown measurement noise (obe_noiseparam.py:6-55)."""

    def __init__(self, measurement_model, setting_values, parameter_samples, constants,
                 noise_parameter_index=None, **kwargs):
        if _non_gaussian(measurement_model, kwargs.get('likelihood_model')):
            raise ValueError('a noise parameter is the sigma of the Gaussian likelihood: '
                             f'{type(self).__name__} takes no other likelihood_model')
        OptBayesExpt.__init__(self, measurement_model, setting_values, parameter_samples, constants, **kwargs)
        self.noise_parameter_index = np.atleast_1d(noise_parameter_index)
        if noise_parameter_index is None or len(self.noise_parameter_index) != self.n_channels:
            raise RuntimeError(f'noise_parameter_index is not compatible with'
                               f' {self.n_channels} measurement channels')
        self.noise_parameter_index = self.noise_parameter_index.astype(int)
        if np.any(self.noise_parameter_index < 0) or np.any(self.noise_parameter_index >= self.n_dims):
            raise RuntimeError('noise_parameter_index out of range')
        self._noise_index = [int(i) for i in self.noise_parameter_index]
        self._moments_valid = False   # the noise accumulators were not part of the first pass

    def set_pdf(self, samples, weights=None):
        OptBayesExpt.set_pdf(self, samples, weights)
        self._moments_valid = False

    def _constraint_masks(self):
        mask = 0
        for i in self._noise_index:
            mask |= 1 << i
        return mask, 0

    def enforce_parameter_constraints(self):
        """Zero the weight of particles whose noise parameter is <= 0 (obe_noiseparam.py:57-79)."""
        self._apply_constraint_masks(mask_le=self._constraint_masks()[0])

    def _likelihood_spec(self, measurement_record):
        """sigma comes from the particles; the record is (settings, y, ...) (obe_noiseparam.py:110-113)."""
        y_meas = np.atleast_1d(np.asarray(measurement_record[1], dtype=np.float64))
        n_lik = min(self.n_channels, len(y_meas))
        return y_meas[:n_lik], None, self._noise_index[:n_lik], n_lik

    def _noise_from_stats(self):
        return True

    def yvar_noise_model(self):
        """Weighted mean of sigma^2 per channel, (C,1) (obe_noiseparam.py:122-136)."""
        from . import _lib
        st = self._ensure_moments()
        c = self.n_channels
        return (st[_lib.ST_NOISE:_lib.ST_NOISE + c] / st[_lib.ST_SUMT]).reshape((c, 1))
