"""-m gpu: ensembles of independent models -- the pspde_ensemble_* entry points (one launch per phase for all members on
the FP32-FMA kernels) and pspde.SolverEnsemble on top of them.

Kernels: six shapes of fma_cases.FMA_SHAPES ('inner' C1 / C3 / C2 networks forced off the tensor-core path for the
single-model reference, 'outer' mode, dense A / B with per-path start points per member, the 512-thread backward) with
M = 1, 5, 37 and 64 members at K = 200 and K = 2 x 64 + 17, at the natural grid and with PSPDE_MAX_GRID=3.  Per-path
outputs equal the single-model calls bit for bit; statistics, loss, cotangents and gradient too while M * n_tiles <= #SMs
(64 members of 4 tiles share the SMs: within the multitile tolerances); every member matches the fp64 oracle.

SolverEnsemble: members of the C1 configuration (LQGC d = 10, 'outer', K = 200) against the same Solvers trained alone
on the FP32-FMA kernels: every log, the final parameters and the Adam state bit for bit."""
import numpy as np
import pytest
import torch as pt

import ensemble_cases as E
import fma_cases as F
import multitile as M
from test_gpu_multitile import abi, grid, sms  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

N_GPU = 6
SHAPES = ["C1i", "OUT", "C3s", "C2s", "AB", "B225"]
ENV = ("PSPDE_FWD_PATH", "PSPDE_BWD_PATH", "PSPDE_GRAD_PATH", "PSPDE_CKPT_ZETA", "PSPDE_FWD_CKPT_MAX_GB")


@pytest.fixture(autouse=True)
def natural_paths(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


@pytest.mark.parametrize("K", [200, 2 * M.P_HJB + 17])
@pytest.mark.parametrize("n_models", [1, 5, 37, 64])
@pytest.mark.parametrize("shape", SHAPES)
def test_ensemble_members_equal_single_calls(abi, sms, grid, shape, n_models, K, monkeypatch):
    F.use_fma_paths(shape, monkeypatch)            # the single-model reference on the FMA kernels
    e = E.EnsembleCase(abi, shape, K, N_GPU, n_models, x0_per_path=shape == "AB")
    n_tiles = (K + M.P_HJB - 1) // M.P_HJB
    bitwise = E.ens_grid_x(n_models, n_tiles, sms, grid) == E.single_grid(n_tiles, sms, grid)
    assert bitwise or n_models * n_tiles > sms
    E.check_ensemble(e, bitwise)


def test_ensemble_ignores_path_knobs(abi, monkeypatch):
    """PSPDE_FWD_PATH=tc / PSPDE_BWD_PATH=ckpt do not reroute the ensemble (two launches each way: the FMA kernels)."""
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    e = E.EnsembleCase(abi, "C1i", 200, N_GPU, 5)
    monkeypatch.setenv("PSPDE_FWD_PATH", "tc")
    monkeypatch.setenv("PSPDE_BWD_PATH", "ckpt")
    for call in (e.forward, e.backward):
        _, rc, n = call()
        assert (rc, n) == (0, 2), (call.__name__, rc, n)


def test_ensemble_adam(abi):
    E.check_adam(abi, n_models=9, n=60000)


def test_ensemble_workspace_exact(abi, monkeypatch):
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    E.check_workspace(E.EnsembleCase(abi, "B225", 200, 2, 5))


# ------------------------------------------------------------------------------------------------ SolverEnsemble
def c1_solver(seed, lr=1e-3, L=5, loss="log-variance", **kw):
    import pspde
    prob = pspde.LQGC(d=10, device="cuda")
    return pspde.Solver("c1", prob, lr=lr, L=L, K=200, delta_t=0.05, loss_method=loss, time_approx="outer",
                        detach_forward=True, early_stopping_time=None, verbose=False, seed=seed, **kw)


def state(s):
    fa = s._flat_adam
    y = [s.y_0.Y_0.detach().cpu().numpy().copy()] if s.learn_Y_0 else []
    return [s._theta.detach().cpu().numpy().copy(), fa["exp_avg"].cpu().numpy().copy(),
            fa["exp_avg_sq"].cpu().numpy().copy(), fa["step"].numpy().copy()] + y


LOGS = ("loss_log", "nonfinite_log", "u_L2_loss", "Y_0_log")


def alone(make, monkeypatch):
    monkeypatch.setenv("PSPDE_FWD_PATH", "simt")
    monkeypatch.setenv("PSPDE_BWD_PATH", "simt")
    s = make()
    s.train()
    monkeypatch.delenv("PSPDE_FWD_PATH")
    monkeypatch.delenv("PSPDE_BWD_PATH")
    return s


@pytest.mark.parametrize("loss,learn_y0,cfgs", [
    ("log-variance", False, [(1, 1e-3, 5), (2, 3e-3, 5), (3, 1e-2, 3), (4, 5e-4, 5)]),      # member 2 stops at L = 3
    ("moment", True, [(5, 1e-3, 5), (6, 2e-3, 5), (7, 4e-3, 5)]),
    ("cross_entropy", False, [(8, 1e-3, 5), (9, 2e-3, 4), (10, 5e-3, 5)]),
], ids=["log-variance", "moment-y0", "cross-entropy"])
def test_solver_ensemble_equals_solvers_alone(loss, learn_y0, cfgs, monkeypatch):
    import pspde
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    make = [lambda c=c: c1_solver(c[0], lr=c[1], L=c[2], loss=loss, learn_Y_0=learn_y0) for c in cfgs]
    ref = [alone(mk, monkeypatch) for mk in make]
    ens = pspde.SolverEnsemble([mk() for mk in make], verbose=False)
    ens.train()
    for c, s, r in zip(cfgs, ens.members, ref):
        assert len(s.loss_log) == c[2]
        for k in LOGS:
            assert getattr(s, k) == getattr(r, k) or (k == "u_L2_loss" and np.array_equal(
                np.array(s.u_L2_loss), np.array(r.u_L2_loss), equal_nan=True)), (c, k, getattr(s, k), getattr(r, k))
        for a, b in zip(state(s), state(r)):
            assert np.array_equal(a, b), c
        assert np.isfinite(s.loss_log).all()


def test_solver_ensemble_members_work_alone(monkeypatch):
    """After training, a member evaluates its control and runs importance sampling like a standalone Solver with its
    parameters; update_Phis() between iterations re-homes it without changing the results."""
    import pspde
    from pspde import do_importance_sampling_me
    monkeypatch.delenv("PSPDE_MAX_GRID", raising=False)
    ens = pspde.SolverEnsemble([c1_solver(s, L=4) for s in (21, 22, 23)], verbose=False)
    ens.train_step(0)
    ens.members[1].update_Phis()
    for l in range(1, 4):
        ens.train_step(l)
    m = ens.members[1]
    ref = alone(lambda: c1_solver(22, L=4), monkeypatch)
    assert m.loss_log == ref.loss_log
    assert m._theta.data_ptr() == ens.theta[1].data_ptr()
    s = c1_solver(22, L=4)
    s._theta.data.copy_(m._theta.detach())
    x = pt.randn(7, 10, device="cuda")
    assert pt.equal(m.Z_n(x, 0.3), s.Z_n(x, 0.3))
    assert do_importance_sampling_me(m.problem, m, 1000) == do_importance_sampling_me(s.problem, s, 1000)


@pytest.mark.parametrize("kw", [dict(noise="inject"), dict(process_group=object()), dict(detach_forward=False),
                                dict(IS_variance_K=100)], ids=["inject", "process-group", "attached", "IS-variance"])
def test_solver_ensemble_refuses(kw):
    import pspde
    base = dict(detach_forward=True)
    base.update(kw)
    import pspde as P
    prob = P.LQGC(d=10, device="cuda")
    bad = P.Solver("c1", prob, K=200, delta_t=0.05, time_approx="outer", early_stopping_time=None, verbose=False, seed=1,
                   **base)
    with pytest.raises(NotImplementedError):
        pspde.SolverEnsemble([c1_solver(2), bad], verbose=False)
