"""The diffusion and elliptic kernels on the host emulator (4 SMs) across network geometries, problem data and dropped
paths, against the fp64 oracle at ten tiles (K = 9 x 32 + 17, the last one ragged), at the natural grid (two or three
tiles per CTA) and with PSPDE_MAX_GRID=2 (five).  Pins the geometry-dependent index logic of diffusion_kernel,
pack_weights_kernel and reduce_dw_kernel, the drift / sigma / h paths and the inert backward of dropped paths without a
GPU; tests/test_gpu_diff_multitile.py runs the same cases on the sm_100a build at B200 sizes."""
import ctypes

import pytest

import diff_cases as D
import emu_harness as H
import multitile as M
from pspde import _lib as L

SMS = 4                        # the emulator's SM count (tests/emu/simt_emul.h)
K_DIFF = 9 * M.P_DIFF + 17     # 10 tiles, the last one ragged
N_EMU, DT_PAR, DT_ELL = 3, 0.03, 0.04
GEOMETRY = ["L1", "H5", "H300", "L4", "W40x3", "NW"]


@pytest.fixture(scope="module")
def abi():
    return M.Abi(H.emu_lib())


@pytest.fixture(params=[None, "2"], ids=["natural", "maxgrid2"])
def grid(request, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    if request.param:
        monkeypatch.setenv("PSPDE_MAX_GRID", request.param)
    return request.param


def test_diff_regimes_covered(abi, monkeypatch):
    """Every shape's plan (DIFF_PLAN, both time modes) and regime; together they reach L = 1 .. 4, d = 1 and 7, ragged
    and 8-aligned widths, more column patches than warps in both GEMMs, a three-term gemm_pairs_nt sum and a tile within
    5 KB of 227 KB.  The library's workspace (per-CTA gradient partials of the block count, the packed weights) equals
    its restatement for every shape, so the block counts are the library's."""
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    for s in D.DIFF_SHAPES:
        D.check_plan(s)
        d = D.DIFF_SHAPES[s][0]
        for elliptic in (False, True):
            dims = D.shape_dims(s, elliptic)
            tm = L.TIME_NONE if elliptic else L.TIME_LAST
            cfg = L.make_cfg(K_DIFF, d, 2, 0.01, L.PROBLEM_HEAT, L.NET_DENSENET, dims, tm, adaptive=False,
                             n_sets=1 if elliptic else 0)
            ws = abi.lib.pspde_elliptic_workspace_bytes(ctypes.byref(cfg), ctypes.byref(H.elliptic_spec("expball"))) \
                if elliptic else abi.lib.pspde_diffusion_workspace_bytes(ctypes.byref(cfg), ctypes.c_float(1.0))
            assert ws == D.workspace_bytes(D.diff_plan(dims, d, tm), SMS), (s, elliptic)
    plans = {s: D.diff_plan(D.shape_dims(s, False), D.DIFF_SHAPES[s][0], L.TIME_LAST) for s in D.DIFF_SHAPES}
    assert {p["L"] for p in plans.values()} == {1, 2, 3, 4}
    assert {p["d"] for p in plans.values()} >= {1, 7}
    assert any(p["nn"] and p["nn"][0] > D.NWARPS for p in plans.values())
    assert max(p["smem"] for p in plans.values()) > D.MAX_SMEM - 5 * 1024


@pytest.mark.parametrize("elliptic", [False, True], ids=["diffusion", "elliptic"])
def test_diff_smem_refusal(abi, elliptic):
    """With C4X's widths the first d that does not fit (d = 123 parabolic, 124 elliptic) is refused with -6 before any
    launch, with the byte count of the restatement; d - 1 is accepted."""
    assert D.refusal_case(abi, (256, 256, 256), elliptic) == (124 if elliptic else 123)


@pytest.mark.parametrize("form", ["loss", "rand"])
@pytest.mark.parametrize("shape", GEOMETRY)
def test_diff_geometry(abi, grid, shape, form):
    """Heat equation, every shape but C4X, both cotangent forms."""
    D.geometry_case(abi, shape, "heat", K_DIFF, N_EMU, DT_PAR, form)


@pytest.mark.parametrize("shape", ["L1", "H300", "L4", "NW"])
def test_ell_geometry(abi, grid, shape):
    """The elliptic kernel (unit ball, expball_sin) on the geometries with their own TIME_NONE plan."""
    D.geometry_case(abi, shape, "expball_sin", K_DIFF, N_EMU, DT_ELL, "rand")


def test_diff_c4x(abi):
    """C4X (d = 100, [256, 256, 256], 227 696 B) at N = 1, PSPDE_MAX_GRID unset."""
    D.geometry_case(abi, "C4X", "heat", K_DIFF, 1, DT_PAR, "rand")


@pytest.mark.parametrize("shape,problem", [("L4", "ou"), ("H5", "ou"), ("L4", "allencahn"), ("L4", "expsphere"),
                                           ("L4", "box2"), ((2, (16, 12)), "helmholtz"), ("L4", "drift")],
                         ids=["ou-L4", "ou-H5", "allencahn-L4", "expsphere-L4", "box2-L4", "helmholtz-d2", "drift-L4"])
def test_diff_problem_data(abi, grid, shape, problem):
    """Drift and sigma through the problem pack (parabolic OU, the two-sided box and the ball with drift), Allen-Cahn,
    H_EXP_LINEAR and Helmholtz (sinf) on many tiles."""
    D.geometry_case(abi, shape, problem, K_DIFF, N_EMU, DT_ELL if problem in D.ELLIPTIC else DT_PAR, "loss")


@pytest.mark.parametrize("problem", ["heat", "allencahn", "expball_sin", "box2"])
def test_diff_boundary_terms(abi, grid, problem):
    """The N = 0 calls of the terminal condition and the Dirichlet term at the same K: V_0 and a c0-only backward."""
    D.boundary_case(abi, "L4", problem, K_DIFF, DT_PAR)


@pytest.mark.parametrize("form", ["loss", "rand"])
@pytest.mark.parametrize("problem", ["heat", "allencahn", "expball_sin", "box2"])
def test_diff_dropped_paths(abi, grid, problem, form):
    """Six 1e20 starts and one NaN start: the forward counts and excludes them, the backward with their cotangents zeroed
    is finite and bit-equal to the run from benign starts."""
    D.dropped_case(abi, "L4", problem, K_DIFF, N_EMU, DT_ELL if problem in D.ELLIPTIC else DT_PAR, form)
