"""optbayesexpt_b200 -- B200-native particle-filter inference and setting selection.

Drop-in for the hot path of usnistgov/optbayesexpt (ParticlePDF, OptBayesExpt,
OptBayesExptNoiseParameter) with the cloud resident in HBM and hand-written sm_100a kernels
behind a C ABI (include/obe_b200.h).  Importing the package does not need a GPU; creating any
of the classes does, and fails loudly without one.
"""
from .models import DeviceModel, builtin, cuda_likelihood, cuda_source  # noqa: F401
from .particlepdf import ParticlePDF  # noqa: F401
from .obe_base import OptBayesExpt  # noqa: F401
from .obe_noiseparam import OptBayesExptNoiseParameter  # noqa: F401
from .obe_sweeper import OptBayesExptSweeper  # noqa: F401

__version__ = '0.1.0'
