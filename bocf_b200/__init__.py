"""bocf_b200 -- B200-native EI-CF hot path behind the reference's (RaulAstudillo06/BOCF) plugin surface.

Host code is Python and mirrors the reference's classes; all arithmetic runs in hand-written sm_100a
CUDA kernels (bocf_b200/csrc) reached through a C ABI (include/bocf_b200.h).  No CPU fallback.
"""
from ._lib import load_library, launch_count, BocfError, NotPositiveDefiniteError, LIB_PATH  # noqa: F401
from . import kern  # noqa: F401
from .utility import Utility, ParameterDistribution, CudaComposite  # noqa: F401
from .model import multi_outputGP  # noqa: F401
from .acquisitions import AcquisitionBase, uEI_noiseless, uPI, maEI, maPI, EI, PI  # noqa: F401
from .optimization import (AcquisitionOptimizer, GeneralOptimizer, Design_space, Sequential,  # noqa: F401
                           initial_design)
from .cbo import CBO, MultiObjective, ExpectationUtility  # noqa: F401
from . import cbo, optimization, distributed  # noqa: F401
