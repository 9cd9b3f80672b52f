"""-m gpu: several tiles per CTA on the sm_100a build.  The attached adjoint kernel and the diffusion / elliptic kernels
against the fp64 oracle (oracle/manual.py) on the kernels' own Philox draws, once at the natural grid with at least
two tiles per CTA on all SMs, and once with PSPDE_MAX_GRID=3 (twenty to two hundred tiles per CTA; C4 runs ~55).
This is where per-tile resets and per-CTA gradient partials are exercised in the compiled code: the register-capped
two-CTA attached build, the fast-math intrinsics, the RED.128 flush of the diffusion backward, all SMs at once.
The same cases at emulator sizes are in tests/test_emu_multitile.py."""
import numpy as np
import pytest
import torch as pt

import multitile as M
from conftest import relerr
from pspde import _lib as L

pytestmark = pytest.mark.gpu

GRIDS = [None, "3"]            # natural grid, then PSPDE_MAX_GRID=3


@pytest.fixture(scope="module")
def abi():
    return M.Abi(L.load(), "cuda")


@pytest.fixture(scope="module")
def sms():
    return pt.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(params=GRIDS, ids=["natural", "maxgrid3"])
def grid(request, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    monkeypatch.delenv("PSPDE_ATT_CTAS", raising=False)
    if request.param:
        monkeypatch.setenv("PSPDE_MAX_GRID", request.param)
    return request.param


def k_for(P, ctas, per_cta=2):
    """per_cta tiles for each of `ctas` CTAs plus a ragged tile of 17 paths."""
    return per_cta * ctas * P + 17


@pytest.mark.parametrize("ctas", [None, "1"], ids=["2cta", "1cta"])
def test_attached_re_doublewell(abi, sms, grid, ctas, monkeypatch):
    """A1 (C3 family): DoubleWell_multidim d = 50 (d_1 = 15, kappa = 5, eta = 3), MySequential(seed=123), relative entropy
    in one launch, K = 2 * 296 * 64 + 17, N = 10, dt = 0.005; two CTAs per SM (the <= 128-register build) or one."""
    if ctas:
        monkeypatch.setenv("PSPDE_ATT_CTAS", ctas)
    import pspde
    net = pspde.MySequential(51, 50, 0.0, seed=123)
    theta = np.concatenate([q.detach().reshape(-1).numpy() for q in net.parameters()]).astype(np.float32)
    K = k_for(M.P_HJB, 2 * sms)
    M.attached_case(abi, "dwm", 50, "mlp_tanh", K, 10, 0.005, "relative_entropy", theta=theta)


@pytest.mark.parametrize("loss", ["relative_entropy", "log-variance"])
def test_attached_512_thread_build(abi, sms, grid, loss):
    """A2: LQGC with DenseNet [81, 30, 30, 80] (294 weight-gradient blocks > 224: rollout_attached_kernel<64, 512, 1>),
    relative entropy and log-variance through forward -> cotangents -> adjoint."""
    assert M.n_grad_blocks("densenet", [81, 30, 30, 80]) == 294
    M.attached_case(abi, "lqgc", 80, "densenet", k_for(M.P_HJB, sms), 10, 0.01, loss)


@pytest.mark.parametrize("d", [97, 128])
@pytest.mark.parametrize("loss", ["moment", "cross_entropy"])
def test_attached_dense_ab(abi, sms, grid, d, loss):
    """A3: LLGC with dense A / B (off_diag != 0), tanh MLP, d = 97 and the validate limit d = 128 (four 32-column
    reaches of the lambda update), per-path moment and cross-entropy cotangents."""
    M.attached_case(abi, "llgc", d, "mlp_tanh", k_for(M.P_HJB, 2 * sms), 5, 0.02, loss, off_diag=0.05)


def test_attached_outer_cross_entropy(abi, sms, grid):
    """A4: LQGC d = 10, 'outer' mode (one parameter set per step), cross-entropy; checked per step and layer block (the
    kernel flushes into gp + n w_floats every step)."""
    M.attached_case(abi, "lqgc", 10, "densenet", k_for(M.P_HJB, 2 * sms), 5, 0.05, "cross_entropy", outer=True)


def test_attached_inert_rows(abi, sms, grid):
    """A5: every 7th path has exactly zero cotangents; the oracle gets the same zeros."""
    M.attached_case(abi, "lqgc", 10, "densenet", k_for(M.P_HJB, 2 * sms), 5, 0.05, "log-variance", inert=True)


@pytest.mark.parametrize("noise", ["philox", "inject"])
def test_diffusion_heat(abi, sms, grid, noise):
    """B1 (C4 family): HeatEquation d = 50, DenseNet [256, 256], N = 25, t_0 in [0.9, 1) so that every tile mixes moving
    and stopped paths; Philox and the same draws injected."""
    M.diffusion_case(abi, "heat", 50, (256, 256), k_for(M.P_DIFF, sms), 25, 0.004, noise)


def test_diffusion_allen_cahn(abi, sms, grid):
    """B2: Allen-Cahn, h = y - y^3: the backward's extra V(X_n) pass."""
    M.diffusion_case(abi, "allencahn", 20, (64, 64), k_for(M.P_DIFF, sms), 20, 0.005, "philox")


@pytest.mark.parametrize("kind", ["sphere", "box", "committor"])
def test_elliptic(abi, sms, grid, kind):
    """B3: sphere (expball_sin), one-sided box, committor annulus; V_L2 per path as well."""
    M.elliptic_case(abi, kind, 10 if kind != "committor" else 5, (30, 30), k_for(M.P_DIFF, sms), 20, 0.005)


@pytest.mark.parametrize("elliptic", [False, True], ids=["diffusion", "elliptic"])
def test_gradient_sharding(sms, elliptic):
    """B4: DiffusionEngine / EllipticEngine with K split into two k_offset shards (not at a tile boundary): the summed
    gradients equal the unsharded one.  Natural grid only: the shards regroup the paths into other tiles, so the
    difference is the rounding of the fp32 per-CTA partial sums, which grows with the tiles per CTA."""
    import pspde
    from pspde.elliptic_solver import EllipticEngine
    from pspde.general_solver import DiffusionEngine
    d, N, dt = 10, 5, 0.01
    K = k_for(M.P_DIFF, sms)
    cut = K // 2 + 5
    if elliptic:
        prob, Eng = pspde.ExponentialOnBallNonlinearSin(d=d, device="cuda"), EllipticEngine
        V = pspde.DenseNet(d_in=d, d_out=1, lr=0.0, seed=4).cuda()
    else:
        prob, Eng = pspde.HeatEquation(d=d, T=1, device="cuda"), DiffusionEngine
        V = pspde.DenseNet(d_in=d + 1, d_out=1, lr=0.0, seed=4).cuda()
    theta = pt.cat([q.detach().reshape(-1) for q in V.parameters()]).contiguous()
    w = (0.5 + pt.rand(K, device="cuda", generator=pt.Generator("cuda").manual_seed(1))) / K
    grads = []
    for lo, hi in ((0, K), (0, cut), (cut, K)):
        eng = Eng(prob, V.net_spec()[1], hi - lo, N, dt, k_offset=lo, seed=7)
        X0, t0 = eng.sample(1.0, 3)
        if not elliptic:
            t0 = 0.9 + 0.1 * t0                   # some paths stop inside the window
        gr = pt.empty(eng.n_theta, device="cuda")
        ws = w[lo:hi].contiguous()
        eng.backward(theta, X0, t0, None, 3, -ws, ws, -ws, gr)
        grads.append(gr.cpu().numpy())
    assert relerr(grads[1] + grads[2], grads[0]) < 1e-6


def test_sample_start_points_vs_restatement(abi, sms):
    """C1: diffusion_sample_kernel (Philox X_0 uniform in the ball, t_0 in [0, T)) against oracle/philox.py."""
    M.sample_case(abi, k_for(M.P_DIFF, sms), 50, 5)
    M.sample_case(abi, 1000, 3, 0, radius=1.0, T=0.3)


def test_sample_start_points_uniform(abi):
    """C2: at K = 2^16 with a fixed seed (deterministic), (|X_0| / R)^d and t_0 / T pass a KS test against U(0, 1)."""
    X0, t0 = M.sample_case(abi, 1 << 16, 50, 0, seed=2024, radius=1.0, T=1.0)
    p_r, p_t = M.sample_uniformity(X0, t0, 1.0, 1.0)
    assert p_r > 1e-3 and p_t > 1e-3, (p_r, p_t)

