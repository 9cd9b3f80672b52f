"""-m gpu: the diffusion and elliptic kernels (diffusion_kernel<32, 512, BWD>, pack_weights_kernel, reduce_dw_kernel)
across network geometries, problem data and dropped paths with many tiles per CTA, against the fp64 oracle
(oracle/manual.py) on the kernels' own Philox draws.

Each case runs at K = 2 x SMs x 32 + 17 (two tiles per CTA on all SMs and a ragged last tile) at the natural grid and
again with PSPDE_MAX_GRID=3 (about two hundred tiles per CTA).  This is where the geometry-dependent index logic meets the
compiled code: fast-math sqrt / divide in the reverse epilogue, the RED.128 flush of the weight gradient, device sinf in
Helmholtz, all SMs at once.  The same cases at emulator sizes are in tests/test_emu_diff_multitile.py."""
import numpy as np
import pytest
import torch as pt

import diff_cases as D
import multitile as M
from test_gpu_multitile import abi, grid, k_for, sms  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

N_GPU, DT = 10, 0.01
GEOMETRY = ["L1", "H5", "H300", "L4", "W40x3", "NW"]


def K_of(sms):
    return k_for(M.P_DIFF, sms)


@pytest.mark.parametrize("form", ["loss", "rand"])
@pytest.mark.parametrize("shape", GEOMETRY)
def test_diff_geometry(abi, sms, grid, shape, form):
    """Heat equation, every shape but C4X, both cotangent forms: per-path outputs, stats, the gradient as a whole and per
    layer block."""
    D.geometry_case(abi, shape, "heat", K_of(sms), N_GPU, DT, form)


@pytest.mark.parametrize("shape", ["L1", "H300", "L4", "NW"])
def test_ell_geometry(abi, sms, grid, shape):
    """The elliptic kernel (unit ball, expball_sin) on the geometries with their own TIME_NONE plan."""
    D.geometry_case(abi, shape, "expball_sin", K_of(sms), N_GPU, DT, "rand")


@pytest.mark.parametrize("elliptic", [False, True], ids=["diffusion", "elliptic"])
def test_diff_c4x(abi, sms, grid, elliptic):
    """C4X: d = 100 with [256, 256, 256], 227 696 B of shared memory, N = 2."""
    D.geometry_case(abi, "C4X", "expball_sin" if elliptic else "heat", K_of(sms), 2, DT, "rand")


@pytest.mark.parametrize("elliptic", [False, True], ids=["diffusion", "elliptic"])
def test_diff_smem_refusal(abi, elliptic):
    """The first d past C4X that does not fit is refused with -6 before any launch; d - 1 is accepted."""
    assert D.refusal_case(abi, (256, 256, 256), elliptic) == (124 if elliptic else 123)


@pytest.mark.parametrize("shape,problem", [("L4", "ou"), ("H5", "ou"), ("L4", "allencahn"), ("L4", "expsphere"),
                                           ("L4", "box2"), ((2, (16, 12)), "helmholtz"), ("L4", "drift")],
                         ids=["ou-L4", "ou-H5", "allencahn-L4", "expsphere-L4", "box2-L4", "helmholtz-d2", "drift-L4"])
def test_diff_problem_data(abi, sms, grid, shape, problem):
    """Drift and sigma through the problem pack (parabolic OU, the two-sided box and the ball with drift), Allen-Cahn,
    H_EXP_LINEAR and Helmholtz (sinf)."""
    D.geometry_case(abi, shape, problem, K_of(sms), N_GPU, DT, "loss")


@pytest.mark.parametrize("problem", ["heat", "allencahn", "expball_sin", "box2"])
def test_diff_boundary_terms(abi, sms, grid, problem):
    """The N = 0 calls of the terminal condition and the Dirichlet term at the same K: V_0 and a c0-only backward."""
    D.boundary_case(abi, "L4", problem, K_of(sms), DT)


@pytest.mark.parametrize("form", ["loss", "rand"])
@pytest.mark.parametrize("problem", ["heat", "allencahn", "expball_sin", "box2"])
def test_diff_dropped_paths(abi, sms, grid, problem, form):
    """Six 1e20 starts and one NaN start: the forward counts and excludes them, the backward with their cotangents zeroed
    is finite, bit-equal to the run from benign starts and the oracle's over the kept paths."""
    D.dropped_case(abi, "L4", problem, K_of(sms), N_GPU, DT, form)


@pytest.mark.parametrize("elliptic", [False, True], ids=["general", "elliptic"])
def test_solver_step_with_diverged_paths(elliptic):
    """One GeneralSolver / EllipticSolver gradient_descent on a batch whose X_0 has three 1e20 rows (past the boundary
    term's samples): the solver reports 3 non-finite residuals, and theta stays finite after Adam."""
    import pspde
    from pspde.general_solver import DiffusionCall
    d, K, N = 10, 1000, 10
    rng = np.random.default_rng(3)
    X0 = M._ball(rng, K, d)
    X0[[300, 601, 999]] = 1e20
    if elliptic:
        prob = pspde.ExponentialOnBallNonlinearSin(d=d, device="cuda")
        S = pspde.EllipticSolver(prob, "t", seed=1, delta_t=0.01, N=N, lr=1e-3, L=1, K=K, K_boundary=50,
                                 loss_method="diffusion", verbose=False)
        call = DiffusionCall(pt.tensor(X0).cuda(), None, None, 0)
        Xb = rng.standard_normal((50, d))
        call.Xb = pt.tensor(Xb / np.linalg.norm(Xb, axis=1, keepdims=True), dtype=pt.float32).cuda()
    else:
        prob = pspde.HeatEquation(d=d, T=1, device="cuda")
        S = pspde.GeneralSolver(prob, "t", seed=1, delta_t=0.01, N=N, lr=1e-3, L=1, K=K, K_boundary=50, verbose=False)
        t0 = rng.uniform(0.9, 1.0, K).astype(np.float32)
        call = DiffusionCall(pt.tensor(X0).cuda(), pt.tensor(t0).cuda(), None, 0)
    S._get_engine()
    before = S._theta.detach().clone()
    sums = S.gradient_descent(call).tolist()
    assert sums[3] == 3
    assert np.isfinite(sums[0]) and pt.isfinite(S._theta.grad).all()
    assert pt.isfinite(S._theta).all() and not pt.equal(S._theta, before)
