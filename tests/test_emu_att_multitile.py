"""The attached adjoint kernel on the host emulator (4 SMs) across network geometries, launch options and dropped
trajectories, against the fp64 discrete adjoint at ten tiles (K = 9 x 64 + 17, the last one ragged) with
PSPDE_MAX_GRID=3 (three or four tiles per CTA).  Pins the geometry- and option-dependent code of rollout_attached_kernel
(input cotangent dx, lambda tile, d > 128 reload, injected draws in the backward sweep, u_L2, in-launch dropping)
without a GPU; tests/test_gpu_att_multitile.py runs the same cases on the sm_100a build at B200 sizes.  Every shape runs
at the same sizes as there but for N; W160 and M4 run at N = 2."""
import ctypes
import re

import numpy as np
import pytest

import att_cases as A
import emu_harness as H
import multitile as M
from pspde import _lib as L

SMS = 4                        # the emulator's SM count (tests/emu/simt_emul.h)
K_ATT = 9 * M.P_HJB + 17       # 10 tiles, the last one ragged
N_EMU = 3


@pytest.fixture(scope="module")
def abi():
    return M.Abi(H.emu_lib())


@pytest.fixture(autouse=True)
def max_grid(monkeypatch):
    monkeypatch.delenv("PSPDE_ATT_CTAS", raising=False)
    monkeypatch.setenv("PSPDE_MAX_GRID", "3")


def n_of(shape):
    return 2 if shape in ("W160", "M4") else N_EMU


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", sorted(A.ATT_SHAPES))
def test_att_geometry(abi, shape, form, monkeypatch):
    """Every shape of att_cases.ATT_SHAPES in both forms (two-CTA shapes also with PSPDE_ATT_CTAS=1)."""
    A.geometry_case(abi, shape, K_ATT, n_of(shape), form, monkeypatch)


@pytest.mark.parametrize("shape", sorted(A.ATT_SHAPES))
def test_att_plan_is_the_library_plan(abi, shape, monkeypatch):
    """The CTAs per SM each case claims are what make_plan chooses: with no grid cap the attached workspace (gradient
    partials and checkpoints per CTA) is that of min(tiles, CTAs per SM x SMs) CTAs -- larger than with
    PSPDE_ATT_CTAS=1 exactly for the two-CTA shapes."""
    c = A.AttCase(abi, shape, K_ATT, 2)
    c.check_plan()
    ws = lambda: abi.lib.pspde_workspace_bytes(ctypes.byref(c.cfg()))
    monkeypatch.delenv("PSPDE_MAX_GRID")
    free = ws()
    monkeypatch.setenv("PSPDE_MAX_GRID", str(A.ctas_per_sm(shape) * SMS))
    assert ws() == free > 0
    monkeypatch.delenv("PSPDE_MAX_GRID")
    monkeypatch.setenv("PSPDE_ATT_CTAS", "1")
    assert (free > ws()) == (A.ctas_per_sm(shape) == 2)


def test_att_regimes_covered(abi):
    """The sweep reaches L = 1 .. 4 with both networks and both time modes, both thread builds, every bw_slot_rows regime,
    nb = 224 and 225, d > 128, and shapes on either side of the two-CTA threshold (smem <= 115 712 B).  The shared
    memory restatement reproduces the library's refusal of DenseNet [96, 30, 30, 95] (233 680 B)."""
    plans = A.ATT_PLAN.values()
    assert {(T, r[0]) for _, T, r, _, _ in plans} >= {(256, "row-split"), (512, "row-split"), (256, "leftovers"),
                                                      (256, "exact")}
    assert {224, 225} <= {nb for nb, _, _, _, _ in plans}
    assert {len(A.shape_dims(s)) - 1 for s in A.ATT_SHAPES} == {1, 2, 3, 4}
    assert {len(A.shape_dims(s)) - 1 for s in A.ATT_SHAPES if A.ATT_SHAPES[s][2] == "mlp_tanh"} >= {3, 4}
    assert max(A.ATT_SHAPES[s][1] for s in A.ATT_SHAPES) > 128
    assert A.ATT_PLAN["AB40"][3:] == (2, 114736) and A.ATT_PLAN["L4X"][3:] == (1, 116592)
    assert 2 * (114736 + 1024) <= A.MAX_SMEM + 1024 < 2 * (116592 + 1024)
    d = 95
    dims = [d + 1, 30, 30, d]
    pid, flags, pack = H.problem_pack("lqgc", d, {})
    cfg = L.make_cfg(100, d, 2, 0.01, pid, L.NET_DENSENET, dims, L.TIME_FIRST, problem_flags=flags)
    theta = np.zeros(abi.lib.pspde_theta_size(ctypes.byref(cfg)), np.float32)
    with pytest.raises(RuntimeError, match="shared memory") as e:
        abi.attached(cfg, theta, pack, np.zeros(d, np.float32), 0.01)
    assert int(re.search(r"need (\d+) B", str(e.value)).group(1)) == A.att_smem("densenet", dims, d) == 233680
    assert A.att_plan("densenet", dims, d)[3] == 0


@pytest.mark.parametrize("shape", ["L4", "W64"])
def test_att_injected_noise(abi, shape):
    """The Philox draws injected in the reference layout: against the oracle and bit-equal to the Philox run."""
    A.inject_case(abi, shape, K_ATT, N_EMU)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["AB40", "B225"])
def test_att_per_path_start(abi, shape, form):
    """Per-path X_0 and y_0 = 0.25."""
    A.start_case(abi, shape, K_ATT, N_EMU, form)


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["L4", "AB40"])
def test_att_shards(abi, shape, form):
    """Two k_offset shards cut inside a tile (64 x SMs + 45)."""
    A.shard_case(abi, shape, K_ATT, N_EMU, form, M.P_HJB * SMS + 45)


@pytest.mark.parametrize("shape", ["DW4", "W160"])
def test_att_u_l2_diagnostic(abi, shape):
    """u_L2 through pspde_rollout_attached_diag (mode-1 table), relative-entropy form."""
    A.ul2_case(abi, shape, K_ATT, n_of(shape))


@pytest.mark.parametrize("form", ["pp", "re"])
@pytest.mark.parametrize("shape", ["L4", "W64", "C3"])
def test_att_dropped_trajectories(abi, shape, form):
    """The blow-up bound d_abs_max and 1e20 starts: dropped paths' cotangents are zeroed inside the launch."""
    A.dropped_case(abi, shape, K_ATT, N_EMU, form)
