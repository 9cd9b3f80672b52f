"""Several tiles per CTA on the host emulator (4 SMs): the attached adjoint kernel and the diffusion / elliptic kernels
against the fp64 oracle at about ten tiles, once at the natural grid and once with PSPDE_MAX_GRID=2 (five tiles per
CTA).  Pins the index logic of the persistent tile loops (per-tile resets, per-CTA gradient partials, checkpoint
slices) without a GPU; tests/test_gpu_multitile.py runs the same cases on the sm_100a build at B200 sizes."""
import ctypes

import numpy as np
import pytest

import emu_harness as H
import multitile as M
from conftest import relerr
from pspde import _lib as L

SMS = 4                        # the emulator's SM count (tests/emu/simt_emul.h)
GRIDS = [None, "2"]            # natural grid, then PSPDE_MAX_GRID=2
K_ATT = 9 * M.P_HJB + 17       # 10 tiles, the last one ragged
K_DIFF = 9 * M.P_DIFF + 17


@pytest.fixture(scope="module")
def abi():
    return M.Abi(H.emu_lib())


@pytest.fixture(params=GRIDS, ids=["natural", "maxgrid2"])
def grid(request, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    monkeypatch.delenv("PSPDE_ATT_CTAS", raising=False)
    if request.param:
        monkeypatch.setenv("PSPDE_MAX_GRID", request.param)
    return request.param


@pytest.mark.parametrize("ctas", [None, "1"], ids=["2cta", "1cta"])
def test_attached_re_doublewell(abi, grid, ctas, monkeypatch):
    """A1 (C3 family): DoubleWell_multidim d = 50, tanh MLP, relative entropy in one launch, two CTAs per SM or one."""
    if ctas:
        monkeypatch.setenv("PSPDE_ATT_CTAS", ctas)
    import pspde
    theta = np.concatenate([q.detach().reshape(-1).numpy() for q in pspde.MySequential(51, 50, 0.0, seed=123).parameters()])
    M.attached_case(abi, "dwm", 50, "mlp_tanh", K_ATT, 4, 0.005, "relative_entropy", theta=theta.astype(np.float32))


@pytest.mark.parametrize("loss", ["relative_entropy", "log-variance"])
def test_attached_512_thread_build(abi, grid, loss):
    """A2: DenseNet [71, 30, 30, 70] has more than 224 weight-gradient blocks, so the attached plan takes the 512-thread
    build (rollout_attached_kernel<64, 512, 1>)."""
    assert M.n_grad_blocks("densenet", [71, 30, 30, 70]) > 224
    M.attached_case(abi, "lqgc", 70, "densenet", K_ATT, 2, 0.02, loss)


@pytest.mark.parametrize("d,loss", [(97, "moment"), (128, "cross_entropy")])
def test_attached_dense_ab(abi, grid, d, loss):
    """A3: LLGC with dense A / B (off_diag != 0) up to d = 128, per-path moment and cross-entropy cotangents."""
    M.attached_case(abi, "llgc", d, "mlp_tanh", K_ATT, 2, 0.02, loss, off_diag=0.05)


def test_attached_outer_cross_entropy(abi, grid):
    """A4: 'outer' mode (one parameter set per step), cross-entropy; the kernel flushes into gp + n w_floats every step."""
    M.attached_case(abi, "lqgc", 10, "densenet", K_ATT, 3, 0.05, "cross_entropy", outer=True)


def test_attached_inert_rows(abi, grid):
    """A5: every 7th path has exactly zero cotangents (inert rows inside revisited tiles)."""
    M.attached_case(abi, "lqgc", 10, "densenet", K_ATT, 5, 0.05, "log-variance", inert=True)


@pytest.mark.parametrize("noise", ["philox", "inject"])
def test_diffusion_heat(abi, grid, noise):
    """B1 (C4 family): HeatEquation d = 50, t_0 in [0.9, 1) (the GPU test uses C4's DenseNet [256, 256])."""
    M.diffusion_case(abi, "heat", 50, (64, 64), K_DIFF, 2, 0.05, noise)


def test_diffusion_allen_cahn(abi, grid):
    """B2: Allen-Cahn, h = y - y^3: the backward's extra V(X_n) pass."""
    M.diffusion_case(abi, "allencahn", 20, (30, 30), K_DIFF, 3, 0.03, "philox")


@pytest.mark.parametrize("kind", ["sphere", "box", "committor"])
def test_elliptic(abi, grid, kind):
    """B3: sphere (expball_sin), one-sided box, committor annulus; V_L2 per path as well."""
    M.elliptic_case(abi, kind, 6 if kind != "committor" else 3, (16, 12), K_DIFF, 4, 0.04)


@pytest.mark.parametrize("elliptic", [False, True], ids=["diffusion", "elliptic"])
def test_gradient_sharding(abi, grid, elliptic):
    """B4: two k_offset shards: the summed gradients equal the unsharded one."""
    K, d, N, dt, arch = K_DIFF, 5, 6, 0.02, (12, 8)
    rng = np.random.default_rng(4)
    X0 = M._ball(rng, K, d)
    t0 = rng.uniform(0.9, 1.0, K).astype(np.float32)
    w = rng.uniform(0.5, 1.5, K) / K        # one sign: the fp32 partial sums do not cancel
    pack = H.heat_pack(d)
    ell = H.elliptic_spec("expball") if elliptic else None
    mk = H.elliptic_cfg if elliptic else H.diffusion_cfg
    dims = ([d] if elliptic else [d + 1]) + list(arch) + [1]
    theta = M._theta(dims, 3)
    grads = []
    for lo, hi in ((0, K), (0, 150), (150, K)):
        cfg = mk(hi - lo, d, N, dt, arch, noise=L.NOISE_PHILOX, k_offset=lo, seed=13, offset=2)
        tt = None if elliptic else t0[lo:hi]
        grads.append(abi.diff_bwd(cfg, 1.0, theta, pack, X0[lo:hi], tt, None, -w[lo:hi], w[lo:hi], -w[lo:hi], ell=ell))
    assert relerr(grads[1] + grads[2], grads[0]) < 1e-6


def test_sample_start_points(abi, grid):
    """C1 / C2: diffusion_sample_kernel against its restatement, and the uniformity of |X_0|^d and t_0 (KS)."""
    M.sample_case(abi, 37, 7, 5)
    X0, t0 = M.sample_case(abi, 2048, 10, 0, radius=1.0)
    p_r, p_t = M.sample_uniformity(X0, t0, 1.0, 1.0)
    assert p_r > 1e-3 and p_t > 1e-3, (p_r, p_t)


def test_max_grid_workspace_follows_the_grid(abi, monkeypatch):
    """PSPDE_MAX_GRID shrinks the per-CTA workspace of the attached and diffusion plans (they apply it last); a workspace
    sized with the hook set is then too small without it, which the launch reports (-7) instead of overrunning."""
    d = 10
    cfg = L.make_cfg(K_ATT, d, 4, 0.05, L.PROBLEM_OU, L.NET_DENSENET, [d + 1, 30, 30, d], L.TIME_FIRST)
    dcfg = H.diffusion_cfg(K_DIFF, 6, 4, 0.02, (16,), noise=L.NOISE_PHILOX)
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    monkeypatch.delenv("PSPDE_ATT_CTAS", raising=False)
    full = abi.lib.pspde_workspace_bytes(ctypes.byref(cfg)), abi.lib.pspde_diffusion_workspace_bytes(ctypes.byref(dcfg), ctypes.c_float(1.0))
    monkeypatch.setenv("PSPDE_MAX_GRID", "2")
    small = abi.lib.pspde_workspace_bytes(ctypes.byref(cfg)), abi.lib.pspde_diffusion_workspace_bytes(ctypes.byref(dcfg), ctypes.c_float(1.0))
    assert small[0] < full[0] and small[1] < full[1]
    monkeypatch.delenv("PSPDE_MAX_GRID")
    ws = np.zeros(small[1] // 8 + 1, np.float64)
    theta = M._theta([7, 16, 1], 0)
    X0, t0 = np.zeros((K_DIFF, 6), np.float32), np.full(K_DIFF, 0.5, np.float32)
    w = np.ones(K_DIFF, np.float32)
    grad = np.zeros(theta.size, np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = abi.lib.pspde_diffusion_bwd(ctypes.byref(dcfg), ctypes.c_float(1.0), p(theta), p(H.heat_pack(6)), p(X0), p(t0),
                                     None, p(w), p(w), p(w), p(grad), p(ws), ws.nbytes, None)
    assert rc == -7 and b"workspace" in abi.lib.pspde_last_error()


def test_attached_densenet_too_wide_fails_loudly(abi):
    """The attached DenseNet plan is refused for shared memory from d ~ 92 on (d = 95 needs 233 680 B): an error that
    names shared memory, not a launch that faults."""
    d = 95
    pid, flags, pack = H.problem_pack("lqgc", d, {})
    cfg = L.make_cfg(100, d, 2, 0.01, pid, L.NET_DENSENET, [d + 1, 30, 30, d], L.TIME_FIRST, problem_flags=flags)
    theta = np.zeros(abi.lib.pspde_theta_size(ctypes.byref(cfg)), np.float32)
    with pytest.raises(RuntimeError, match="shared memory"):
        abi.attached(cfg, theta, pack, np.zeros(d, np.float32), 0.01)
