"""dgp_toolbox_b200 — B200-native doubly-stochastic DGP hot path behind the dgp-toolbox class API.

Importing the package loads libdgp_b200.so (hand-written sm_100a CUDA behind a C ABI); it raises if the library has
not been built. There is no CPU fallback.
"""
from . import _lib  # noqa: F401  (fails loudly when the CUDA library is missing)
from . import gpflow_shim as gpflow  # noqa: F401
from .gpflow_shim import RBF, Gaussian, Identity, Linear, Matern32, Matern52, Parameter, SquaredExponential, Zero  # noqa: F401
from .models.dgp import DGP, DGP_Base  # noqa: F401
from .utils.layers import Layer, SVGP_Layer  # noqa: F401
from .utils.layer_initializations import init_layers_linear  # noqa: F401
from .Infill_criteria import EI, EV, WB2, WB2S, EV_one_constraint, PoF, qEI  # noqa: F401
from .EHVI import EHVI, EHVI_with_grad, EI_and_EHVI, HV_calcul, NDC, Y_ND, optimize_EHVI, psi  # noqa: F401
from . import composite  # noqa: F401  (composite kernels with active_dims, layers on supplied kernel matrices: SURVEY §8 f2)
from .models import MF_DGP  # noqa: F401
from .models.MF_DGP import MultiFidelityDeepGP  # noqa: F401
from .models import MF_DGP_EM  # noqa: F401
from .models.MF_DGP_EM import MultiFidelityDeepGP_EM  # noqa: F401
from .models import MO_DGP  # noqa: F401
from .models.MO_DGP import MultiObjDeepGP  # noqa: F401
