"""maxent_b200 -- a B200-native Maximum-Entropy analytic-continuation engine with the Python interface of
TRIQS/maxent (``from maxent_b200 import *`` exports the names of ``from triqs_maxent import *``,
python/__init__.py:20-38, for everything on the hot path; SURVEY.md Appendix C).

The hot path -- kernel SVD, the warm-started Levenberg-Marquardt alpha sweep, probabilities and analyzers --
runs in hand-written sm_100a CUDA kernels behind the C ABI of include/maxent_b200.h
(libmaxent_b200.so, loaded with ctypes by ``_lib``).  There is no CPU fallback."""
from .alpha_meshes import *            # noqa: F401,F403
from .omega_meshes import *            # noqa: F401,F403
from .default_models import *          # noqa: F401,F403
from .logtaker import Logtaker, VerbosityFlags
from .kernels import KernelSVD, Kernel, DataKernel, TauKernel, IOmegaKernel, PreblurKernel
from .functions import (safelog, view_real, view_complex, cached, CachedFunction, GenericFunction,
                        DoublyDerivableFunction, InvertibleFunction, NullFunction, Chi2, NormalChi2, ComplexChi2,
                        Entropy, NormalEntropy, PlusMinusEntropy, ComplexPlusMinusEntropy, AbsoluteEntropy,
                        ShiftedAbsoluteEntropy, GenericH_of_v, NormalH_of_v, PlusMinusH_of_v,
                        ComplexPlusMinusH_of_v, NoExpH_of_v, IdentityH_of_v, GenericA_of_H, IdentityA_of_H,
                        PreblurA_of_H)
from .cost_functions import CostFunction, MaxEntCostFunction, BryanCostFunction
from .minimizers import (Minimizer, LevenbergMinimizer, ConvergenceMethod, AndConvergenceMethod,
                         OrConvergenceMethod, MaxDerivativeConvergenceMethod, NullConvergenceMethod,
                         FunctionChangeConvergenceMethod, RelativeFunctionChangeConvergenceMethod)
from .probabilities import Probability, NormalLogProbability
from .analyzers import (Analyzer, AnalyzerResult, LineFitAnalyzer, Chi2CurvatureAnalyzer, EntropyAnalyzer,
                        ClassicAnalyzer, BryanAnalyzer)
from .maxent_result import MaxEntResult, MaxEntResultData, recursive_map, recursive_dtype, saved
from .maxent_loop import MaxEntLoop
from .preblur import get_preblur, preblur_scan
from .tau_maxent import TauMaxEnt
from .elementwise_maxent import ElementwiseMaxEnt, DiagonalMaxEnt, PoormanMaxEnt, CallableMethodCheck
from .batched import BatchedTauMaxEnt, BatchedMaxEntResult
from .batched_matrix import BatchedElementwiseMaxEnt, BatchedPoormanMaxEnt, BatchedMatrixMaxEntResult
from .maxent_util import numder, check_der, get_G_w_from_A_w, get_G_tau_from_A_w
from .triqs_support import if_no_triqs, if_triqs_1, if_triqs_2, require_triqs, assert_text_files_equal
from .version import show_version, show_git_hash
from .sigma_continuator import SigmaContinuator, DirectSigmaContinuator, InversionSigmaContinuator

__version__ = "0.2"
