"""The FP32-FMA detached rollout kernels on the host emulator (4 SMs) across network geometries, against the fp64 oracle at
ten tiles (K = 9 x 64 + 17), once at the natural grid and once with PSPDE_MAX_GRID=2 (five tiles per CTA).  Pins the
geometry-dependent index logic (thread build, row-split and leftover weight-gradient blocks and their flush, layer
count, per-tile resets, network time remap, per-path start points) without a GPU; tests/test_gpu_fma_multitile.py runs
the same cases on the sm_100a build at B200 sizes.  The tensor-core rows of that file are device only."""
import pytest

import emu_harness as H
import fma_cases as F
import multitile as M

SMS = 4                        # the emulator's SM count (tests/emu/simt_emul.h)
K_EMU = 9 * M.P_HJB + 17       # 10 tiles, the last one ragged
N_EMU = 3


@pytest.fixture(scope="module")
def abi():
    return M.Abi(H.emu_lib())


@pytest.fixture(params=[None, "2"], ids=["natural", "maxgrid2"])
def grid(request, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    if request.param:
        monkeypatch.setenv("PSPDE_MAX_GRID", request.param)
    return request.param


@pytest.mark.parametrize("shape", sorted(F.FMA_SHAPES))
def test_fma_geometry(abi, grid, shape):
    """The forward and recompute backward of every shape of fma_cases.FMA_SHAPES (N = 2 for the widest ones)."""
    F.geometry_case(abi, shape, K_EMU, 2 if shape in ("C2s", "D106", "M4") else N_EMU)


def test_fma_nonadaptive_z_cotangent(abi, grid):
    """NA: C1's network, uncontrolled process with a cotangent on Z_sum (zeta involves Z)."""
    F.geometry_case(abi, "C1i", K_EMU, N_EMU, adaptive=False, wz=True)


def test_fma_regimes_covered():
    """Every regime the sweep claims to reach is in FMA_PLAN: row-split with cpb 2, 4 and 32, leftovers in both builds,
    nb = 224 and 225, L = 1 .. 4."""
    regs = {(T, r[0]) for _, T, r in F.FMA_PLAN.values()}
    assert {(256, "row-split"), (512, "row-split"), (256, "leftovers"), (512, "leftovers"), (256, "exact")} <= regs
    assert {r[1] for _, _, r in F.FMA_PLAN.values() if r[0] == "row-split"} >= {2, 4, 32}
    assert {224, 225} <= {nb for nb, _, _ in F.FMA_PLAN.values()}
    assert {len(F.shape_dims(s)) - 1 for s in F.FMA_SHAPES} == {1, 2, 3, 4}


def test_fma_shards_per_path_start(abi, grid):
    """Dense A / B with per-path X_0 and y_0, two k_offset shards cut inside a tile."""
    c = F.FmaCase(abi, "AB", K_EMU, N_EMU, x0_per_path=True, y0=0.25)
    F.shard_case(abi, c, M.P_HJB * SMS + 45)


@pytest.mark.parametrize("shape", ["L2", "AB", "OUT"])
def test_fma_importance_sampling_time_index(abi, grid, shape):
    """pspde_importance_sampling with dt_net = 2.5 dt: L2 and AB ('inner'), OUT ('outer' with 3 parameter sets, so the
    set index runs past the last one and is clamped)."""
    n_sets = 3 if shape == "OUT" else None
    c = F.FmaCase(abi, shape, K_EMU, 8, n_sets=n_sets)
    t_index = F.importance_sampling_case(abi, c)
    assert t_index[-1] >= 2 and (n_sets is None or t_index[-1] > n_sets - 1)


def test_fma_refuses_past_its_limits(abi):
    """DenseNet [30, 30] at d = 107 (backward refused for shared memory, forward vs the oracle) and d = 121 (backward
    refused for its 528 gradient blocks, forward for shared memory): host-side refusals, no launch."""
    F.refusal_case(abi, 200)
