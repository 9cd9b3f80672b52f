"""pspde: B200-native (sm_100a) fused path-space rollout behind the interface of
lorenzrichter/path-space-PDE-solver's training hot path.  See DESIGN.md / INTEGRATION.md."""
from .function_space import DenseNet, MySequential, SingleParam  # noqa: F401
from .problems import (LLGC, LQGC, DoubleWell, DoubleWell_multidim, HeatEquation, AllenCahn, ExponentialOnSphere,  # noqa: F401
                       ExponentialOnBallNonlinear, ExponentialOnBallNonlinearSin, Helmholtz, Committor)
from .solver import Solver  # noqa: F401
from .ensemble import SolverEnsemble  # noqa: F401
from .general_solver import GeneralSolver  # noqa: F401
from .elliptic_solver import EllipticSolver  # noqa: F401
from .utilities import do_importance_sampling_me  # noqa: F401
