"""probayes_b200 -- B200-native (sm_100a) drop-in for the probayes inference hot path.

The host classes mirror the reference's public interface for the path
(``import probayes_b200 as pb``: RV, RF, SD, SP, PD, CondCov, pscales helpers);
all array work on the path runs in hand-written CUDA kernels behind the C ABI of
``include/pbx.h`` (``probayes_b200/csrc``).  There is no CPU fallback: the CUDA
library is loaded on first use and a missing library or GPU raises ``PbxError``.
"""
from .constants import (NEARLY_POSITIVE_ZERO, NEARLY_POSITIVE_INF, NEARLY_NEGATIVE_INF,
                        LOG_NEARLY_POSITIVE_INF, COMPLEX_ZERO)
from .pscales import (eval_pscale, iscomplex, log_prob, exp_logp, logp_offs, prob_coef,
                      rescale, prod_pscale, prod_rule, div_prob)
from .vtypes import uniform, isscalar, isunitset, isunitsetint, issingleton
from .rv import RV
from .rf import RF
from .sd import SD
from .sp import SP, MCMC_SAMPLERS, Walk, Sampler, AcceptRecord
from .pd import PD, product
from .cond_cov import CondCov
from .serial import (serialise, deserialise, write_serialised, read_serialised, write_dist,
                     read_dist)
from . import catalogue
from .catalogue import (NormalRegression, StudentTRegression, BallIndicator, NormalProduct,
                        BoxUniform)
from ._lib import PbxError

__version__ = "0.1.0"


def get_engine(device=None):
    """The process-wide device engine (lazy import keeps ``import probayes_b200``
    free of torch/CUDA initialisation)."""
    from .engine import get_engine as _g
    return _g(device)
