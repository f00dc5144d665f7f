"""elfi_b200 -- B200-native (sm_100a) implementation of ELFI's data-parallel hot path.

The package mirrors the operator / sampler API of elfi-dev/elfi for the batched
summary -> distance -> threshold/top-n selection -> SMC weight path, the BOLFI GP
surrogate and the BSL synthetic likelihood, with the arithmetic in hand-written CUDA reached through a C ABI
(include/elfi_b200.h).  See DESIGN.md and INTEGRATION.md.
"""
__version__ = '0.1.0'

from . import _lib  # noqa: F401
from .model import (AdaptiveDistance, Constant, Discrepancy, Distance, ElfiModel,  # noqa: F401
                    NodeReference, Operation, Prior, RandomVariable, Simulator, Summary,
                    get_default_model, new_model, set_default_model)
from .samplers import (SMC, AdaptiveDistanceSMC, AdaptiveThresholdSMC,  # noqa: F401
                       DensityRatioEstimation, GMDistribution, ModelPrior, Rejection)
from .store import OutputPool  # noqa: F401
from .bo import (BOLFI, LCBSC, BayesianOptimization, BolfiPosterior, GPyRegression,  # noqa: F401
                 ExpIntVar, MaxVar, RandMaxVar, UniformAcquisition)
from . import bsl  # noqa: F401,E402
from .bsl import BSL  # noqa: F401,E402
