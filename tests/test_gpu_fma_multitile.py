"""-m gpu: the FP32-FMA detached rollout kernels -- rollout_kernel<64, 512, false, 1> (forward, importance sampling) and
rollout_kernel<64, 256 | 512, true, 1> (recompute backward) with reduce_grad_image_kernel -- across network geometries
with many tiles per CTA, against the fp64 oracle (oracle/manual.py) on the kernels' own Philox draws.

These kernels run every configuration outside the tensor-core shape class: 'outer' mode, dense A / B, d > 102, and any
control network but two hidden layers of width <= 32.  Each shape of fma_cases.FMA_SHAPES runs at K = 2 x SMs x 64 + 17
(two tiles per CTA on all SMs and a ragged last tile) at the natural grid and again with PSPDE_MAX_GRID=3 (~200 tiles
per CTA).  Tensor-core-eligible shapes are forced onto the FMA kernels (PSPDE_FWD_PATH / PSPDE_BWD_PATH=simt), the
others take their natural route, and the launch counts are checked either way: a silent reroute to the tensor-core
kernels fails.  The same cases at emulator sizes are in tests/test_emu_fma_multitile.py; the tensor-core rows here
(per-path start points under sharding, importance sampling's look-ahead of t_index) are device only."""
import numpy as np
import pytest

import fma_cases as F
import multitile as M
from test_gpu_multitile import abi, grid, k_for, sms  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

N_GPU = 10
ENV = ("PSPDE_FWD_PATH", "PSPDE_BWD_PATH", "PSPDE_GRAD_PATH", "PSPDE_GRAD_FLUSH_STAGES", "PSPDE_WAVE_TILES_PER_SM",
       "PSPDE_CKPT_ZETA", "PSPDE_FWD_CKPT_MAX_GB")


@pytest.fixture(autouse=True)
def natural_paths(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


def K_of(sms):
    return k_for(M.P_HJB, sms)


@pytest.mark.parametrize("shape", sorted(F.FMA_SHAPES))
def test_fma_geometry(abi, sms, grid, shape, monkeypatch):
    """The forward and recompute backward of every shape of fma_cases.FMA_SHAPES: per-path outputs, stats, the gradient
    as a whole and per (set, layer) block, a second backward bit-equal to the first."""
    F.use_fma_paths(shape, monkeypatch)
    F.geometry_case(abi, shape, K_of(sms), N_GPU)


def test_fma_nonadaptive_z_cotangent(abi, sms, grid, monkeypatch):
    """NA: C1's network, uncontrolled process with a cotangent on Z_sum (zeta involves Z)."""
    F.use_fma_paths("C1i", monkeypatch)
    F.geometry_case(abi, "C1i", K_of(sms), N_GPU, adaptive=False, wz=True)


def test_fma_refuses_past_its_limits(abi):
    """DenseNet [30, 30] at d = 107 (backward refused for shared memory, forward vs the oracle) and d = 121 (backward
    refused for its 528 gradient blocks, forward for shared memory): host-side refusals, no launch."""
    F.refusal_case(abi, 300)


# ----------------------------------------------------------------------------------- shards, per-path start points
def test_fma_shards_per_path_start(abi, sms, grid):
    """Dense A / B with per-path X_0 and y_0, two k_offset shards cut inside a 64-path tile (64 x SMs + 45)."""
    c = F.FmaCase(abi, "AB", K_of(sms), N_GPU, x0_per_path=True, y0=0.25)
    F.shard_case(abi, c, M.P_HJB * sms + 45)


def test_tc_shards_per_path_start(abi, sms, grid, monkeypatch):
    """The same on the tensor-core forward and checkpointed backward at the C2 shape."""
    monkeypatch.setenv("PSPDE_FWD_PATH", "tc")
    monkeypatch.setenv("PSPDE_BWD_PATH", "ckpt")
    c = M.TcCase(abi, "c2", K_of(sms), x0_per_path=True, y0=0.25)
    whole, _, _ = abi.fwd_ckpt(c.cfg(), c.theta, c.pack, c.x0, y0=c.y0)
    cut = M.P_HJB * sms + 45
    outs, grad = [], 0.0
    for lo, hi in ((0, cut), (cut, c.K)):
        cfg = c.cfg(K_local=hi - lo, k_offset=lo)
        outs.append(abi.fwd_ckpt(cfg, c.theta, c.pack, c.x0[lo:hi], y0=c.y0)[0])
        grad = grad + abi.bwd_detached(cfg, c.theta, c.pack, c.x0[lo:hi], c.wY[lo:hi])[0].astype(np.float64)
    for k in ("X", "Y", "gX", "Zsum"):
        assert np.array_equal(np.concatenate([o[k] for o in outs]), whole[k]), k
    m = c.oracle()
    M.check_tc_forward(whole, m)
    M.check_grad(grad, m["grad"], c.blocks(), "tc shards")


# ------------------------------------------------------------------------------------------- importance sampling
@pytest.mark.parametrize("shape", ["L2", "AB", "OUT"])
def test_fma_importance_sampling_time_index(abi, sms, grid, shape):
    """pspde_importance_sampling with dt_net = 2.5 dt: L2 and AB ('inner'), OUT ('outer' with 3 parameter sets, so the
    set index runs past the last one and is clamped)."""
    n_sets = 3 if shape == "OUT" else None
    c = F.FmaCase(abi, shape, K_of(sms), N_GPU, n_sets=n_sets)
    t_index = F.importance_sampling_case(abi, c)
    assert n_sets is None or t_index[-1] > n_sets - 1


def test_tc_importance_sampling_time_index(abi, sms, grid, monkeypatch):
    """The tensor-core forward at the C2 shape (forced: an ineligible configuration is an error), which reads t_index[n + 1]
    ahead of step n: the last step's network time matters."""
    monkeypatch.setenv("PSPDE_FWD_PATH", "tc")
    c = F.FmaCase(abi, "C2s", K_of(sms), N_GPU)
    F.importance_sampling_case(abi, c, launches=None)
