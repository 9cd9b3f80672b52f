"""The ensemble entry points (pspde_ensemble_*) on the host emulator (4 SMs): three members with different Philox keys,
parameters, cotangents and y0 on C1's network ('inner', per-path start points), 'outer' mode and C3's tanh network.
Each member's per-path outputs equal the single-model forward's bit for bit; statistics, loss, cotangents and gradient
too whenever the members get the standalone grid (one tile each, or PSPDE_MAX_GRID=1 for both), else within the fp32
tolerances of the multitile tests; every member matches the fp64 oracle.  The same at B200 sizes and through
SolverEnsemble is in tests/test_gpu_ensemble.py."""
import pytest

import emu_harness as H
import ensemble_cases as E
import multitile as M

SMS = 4                        # the emulator's SM count (tests/emu/simt_emul.h)
N_EMU = 3
SHAPES = ["C1i", "OUT", "C3s"]


@pytest.fixture(scope="module")
def abi():
    return M.Abi(H.emu_lib())


# (K, PSPDE_MAX_GRID): one tile per member (3 x 1 <= 4 SMs: the standalone grid), three tiles per member (9 > 4 SMs: one
# CTA each instead of three), and three tiles per member with both grids capped to one CTA
GRIDS = [(50, None), (2 * M.P_HJB + 17, None), (2 * M.P_HJB + 17, "1")]


@pytest.mark.parametrize("K,max_grid", GRIDS, ids=["one-tile", "shared-sms", "maxgrid1"])
@pytest.mark.parametrize("shape", SHAPES)
def test_ensemble_members_equal_single_calls(abi, shape, K, max_grid, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    if max_grid:
        monkeypatch.setenv("PSPDE_MAX_GRID", max_grid)
    e = E.EnsembleCase(abi, shape, K, N_EMU, 3, x0_per_path=shape == "C1i")
    n_tiles = (K + M.P_HJB - 1) // M.P_HJB
    bitwise = E.ens_grid_x(3, n_tiles, SMS, max_grid) == E.single_grid(n_tiles, SMS, max_grid)
    assert bitwise == (K == 50 or max_grid is not None)
    E.check_ensemble(e, bitwise)


def test_ensemble_adam(abi):
    E.check_adam(abi)


def test_ensemble_workspace_exact(abi, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    E.check_workspace(E.EnsembleCase(abi, "C1i", 2 * M.P_HJB + 17, 2, 3))
