"""-m gpu: the attached adjoint kernel rollout_attached_kernel (detach_forward=False) across network geometries, launch
options and dropped trajectories with many tiles per CTA, against the fp64 discrete adjoint (oracle/manual.py) on the
kernels' own Philox draws.

Each case runs at K = 2 x (CTAs per SM x SMs) x 64 + 17 (two tiles per CTA on all SMs and a ragged last tile) at the
natural grid and again with PSPDE_MAX_GRID=3.  The shapes of att_cases.ATT_SHAPES reach the input cotangent dx of L = 1 .. 4
DenseNets and tanh MLPs, both sides of the two-CTA threshold of the attached plan (the register-capped
rollout_attached_kernel<64, 256, 1, 2> with leftover lanes included), both thread builds and d > 128.  Injected noise,
per-path X_0 and y_0, k_offset shards, the u_L2 diagnostic and the blow-up bound run on a few of them.  The same cases at
emulator sizes are in tests/test_emu_att_multitile.py."""
import pytest

import att_cases as A
import multitile as M
from test_gpu_multitile import abi, grid, k_for, sms  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

N_GPU = 10


def K_of(shape, sms):
    return k_for(M.P_HJB, A.ctas_per_sm(shape) * sms)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", sorted(A.ATT_SHAPES))
def test_att_geometry(abi, sms, grid, shape, form, monkeypatch):
    """Every shape in both forms: per-path outputs, stats, the gradient as a whole and per (set, layer) block, the launch
    count, a second launch bit-equal to the first; two-CTA shapes also with PSPDE_ATT_CTAS=1 (per-path outputs
    bit-equal to the two-CTA run)."""
    A.geometry_case(abi, shape, K_of(shape, sms), N_GPU, form, monkeypatch)


@pytest.mark.parametrize("shape", ["L4", "W64"])
def test_att_injected_noise(abi, sms, grid, shape):
    """The Philox draws injected in the reference layout (K, d, N + 1): against the oracle and bit-equal to the Philox
    run."""
    A.inject_case(abi, shape, K_of(shape, sms), N_GPU)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["AB40", "B225"])
def test_att_per_path_start(abi, sms, grid, shape, form):
    """Per-path X_0 and y_0 = 0.25 against the oracle."""
    A.start_case(abi, shape, K_of(shape, sms), N_GPU, form)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["L4", "AB40"])
def test_att_shards(abi, sms, grid, shape, form):
    """Two k_offset shards cut inside a tile (64 x SMs + 45), as C3re is sharded over GPUs."""
    A.shard_case(abi, shape, K_of(shape, sms), N_GPU, form, M.P_HJB * sms + 45)


@pytest.mark.parametrize("shape", ["DW4", "W160"])
def test_att_u_l2_diagnostic(abi, sms, grid, shape):
    """u_L2 through pspde_rollout_attached_diag (mode-1 table), relative-entropy form, as RolloutEngine.attached calls it."""
    A.ul2_case(abi, shape, K_of(shape, sms), N_GPU)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["L4", "W64", "C3"])
def test_att_dropped_trajectories(abi, sms, grid, shape, form):
    """The blow-up bound d_abs_max and 1e20 starts: dropped paths' cotangents are zeroed inside the same launch."""
    A.dropped_case(abi, shape, K_of(shape, sms), N_GPU, form)
