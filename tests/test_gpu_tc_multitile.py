"""-m gpu: the tensor-core (tcgen05) rollout and gradient kernels with many tiles, stages and flushes per CTA, against the
fp64 oracle (oracle/manual.py) on the kernels' own Philox draws.

Every log-variance workload (C2, C3, C5) runs on these kernels, and all of them are persistent: rollout_tc_fwd_kernel
loops `tile += gridDim.x` over 128-path tiles, and the gradient kernels loop over 32-sample stages, flushing their
tensor-memory accumulators into the CTA's partial every few stages (grad_tc2_kernel at a per-CTA offset, deferring the
D1 flush by one stage).  At C5 a CTA runs ~55 forward tiles and ~1 600 gradient stages per launch.  Each case runs at
K = 2 x SMs x 128 + 17 (two tiles per CTA on all SMs and a ragged last tile) at the natural grid and again with
PSPDE_MAX_GRID=3 (~100 tiles per CTA; the wave size stays per_sm x SMs tiles, so each gradient CTA runs ~2 000 stages
per launch).  The paths are forced (PSPDE_FWD_PATH=tc, PSPDE_BWD_PATH=ckpt, PSPDE_GRAD_PATH=tc / tc1) and the launch
counts checked: a fall-back to the FP32-FMA kernels fails.

The largest column-group instantiation of the forward (NG = kTcMaxG = 12) is reached by no valid shape: tc_geom needs
2 s0 + 2 x 32 + 64 + np3 <= 512 tensor-memory columns (np3 = s0 rounded up to 16), so s0 <= 104 (d <= 102) and at
most ceil(104 / 16) = 7 groups per thread.  d = 102 (all 512 columns, NG = 7) is the largest case, and d = 103 must be
refused."""
import ctypes

import numpy as np
import pytest
import torch as pt

import multitile as M
from conftest import relerr
from pspde import _lib as L
from test_gpu_multitile import abi, grid, k_for, sms  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

ENV = ("PSPDE_FWD_PATH", "PSPDE_BWD_PATH", "PSPDE_GRAD_PATH", "PSPDE_GRAD_FLUSH_STAGES", "PSPDE_WAVE_TILES_PER_SM",
       "PSPDE_CKPT_ZETA", "PSPDE_FWD_CKPT_MAX_GB")


@pytest.fixture(autouse=True)
def tc_paths(monkeypatch):
    """The tensor-core forward, the checkpointed backward and a tensor-core gradient kernel, or an error."""
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("PSPDE_FWD_PATH", "tc")
    monkeypatch.setenv("PSPDE_BWD_PATH", "ckpt")
    monkeypatch.setenv("PSPDE_GRAD_PATH", "tc")


def K_of(sms):
    return k_for(M.P_TC, sms)


def n_tiles(K):
    return (K + M.P_TC - 1) // M.P_TC


# ---------------------------------------------------------------------------------------------------------- forward
@pytest.mark.parametrize("shape", ["c2", "c3", "lqgc7", "d102"])
def test_tc_forward(abi, sms, grid, shape):
    """F1-F4: rollout_tc_fwd_kernel (plain build): X_N, Y_N, g(X_N), Z_sum per path and the stats.  c2: LLGC d = 100 with
    DenseNet [30, 30] (NG = 7); c3: DoubleWell d = 50, MySequential, dt = 0.005 (NG = 4); lqgc7: d % 4 != 0 (NG = 2);
    d102: DenseNet [32, 32], every tensor-memory column in use."""
    c = M.TcCase(abi, shape, K_of(sms))
    o, _, n = abi.fwd_ckpt(c.cfg(), c.theta, c.pack, c.x0)
    assert n == 3                  # weight pack + tensor-core rollout + stats reduction
    M.check_tc_forward(o, c.oracle())


def test_tc_forward_refuses_d103(abi):
    """No tensor-core instantiation beyond d = 102: the forced path is an error, not a fall-back."""
    c = M.TcCase(abi, ("llgc", 103, "densenet", (32, 32), 2, 0.01), 300)
    with pytest.raises(RuntimeError, match="shape class"):
        abi.fwd_ckpt(c.cfg(), c.theta, c.pack, c.x0)


def test_tc_forward_u_l2(abi, sms, grid):
    """F5: the DIAG build at the C2 shape: u_L2 per path (mode 1, linear table) against a numpy restatement of the
    kernel's sum on the oracle's per-step Z and states."""
    c = M.TcCase(abi, "c2", K_of(sms))
    o, _, n = abi.fwd_ckpt(c.cfg(), c.theta, c.pack, c.x0, table=c.table)
    assert n == 3
    m = c.oracle()
    M.check_tc_forward(o, m)
    assert o["uL2"].min() > 0
    assert relerr(o["uL2"], m["uL2"]) < M.TOL_PATH, relerr(o["uL2"], m["uL2"])


def test_tc_forward_keeping_rows(abi, sms, grid):
    """F6: pspde_rollout_fwd_ckpt keeping the rows of every tile computes what the plain forward computes, bit for bit
    (the stats up to the order of their fp64 atomic adds)."""
    c = M.TcCase(abi, "c2", K_of(sms))
    cfg = c.cfg()
    o0, _, _ = abi.fwd_ckpt(cfg, c.theta, c.pack, c.x0)
    o1, ck, n = abi.fwd_ckpt(cfg, c.theta, c.pack, c.x0, ckpt_bytes=abi.lib.pspde_fwd_ckpt_bytes(ctypes.byref(cfg)))
    assert n == 3
    for k in ("X", "Y", "gX", "Zsum"):
        assert np.array_equal(o0[k], o1[k]), k
    np.testing.assert_allclose(o1["stats"], o0["stats"], rtol=1e-12, atol=0)


# --------------------------------------------------------------------------------------------------------- gradient
@pytest.mark.parametrize("shape", ["c2", "c3"])
def test_tc2_wave_backward(abi, sms, grid, shape, monkeypatch):
    """G1: the wave-checkpointed backward through grad_tc2_kernel (zeta regenerated from Philox) at the C2 and C3 shapes,
    one tile per SM per wave: three waves, the last of one tile."""
    monkeypatch.setenv("PSPDE_WAVE_TILES_PER_SM", "1")
    c = M.TcCase(abi, shape, K_of(sms))
    g, n = abi.bwd_detached(c.cfg(), c.theta, c.pack, c.x0, c.wY)
    assert n_tiles(c.K) == 2 * sms + 1 and n == 3 * 3 + 1      # per wave: pack + rollout + gradient; one reduction
    M.check_grad(g, c.oracle()["grad"], c.blocks(), "tc2 " + shape)


@pytest.mark.parametrize("shape", ["c2", "c3"])
@pytest.mark.parametrize("how", ["inject", "tc1"])
def test_tc1_wave_backward(abi, sms, grid, shape, how, monkeypatch):
    """G2: the same through grad_tc_kernel: injected increments (zeta read from the checkpoint) or PSPDE_GRAD_PATH=tc1
    on Philox."""
    monkeypatch.setenv("PSPDE_WAVE_TILES_PER_SM", "1")
    c = M.TcCase(abi, shape, K_of(sms))
    if how == "tc1":
        monkeypatch.setenv("PSPDE_GRAD_PATH", "tc1")
        g, n = abi.bwd_detached(c.cfg(), c.theta, c.pack, c.x0, c.wY)
    else:
        g, n = abi.bwd_detached(c.cfg(inject=True), c.theta, c.pack, c.x0, c.wY, xi=c.xi_ref())
    assert n == 3 * 3 + 1
    M.check_grad(g, c.oracle()["grad"], c.blocks(), "tc1 %s %s" % (shape, how))


def test_tc1_nonadaptive_z_cotangent(abi, sms, grid, monkeypatch):
    """G2: grad_tc_kernel for a non-adaptive process with a cotangent on Z_sum (zeta involves Z: read from the
    checkpoint), C2 shape."""
    monkeypatch.setenv("PSPDE_WAVE_TILES_PER_SM", "1")
    c = M.TcCase(abi, "c2", K_of(sms), adaptive=False, wz=True)
    g, n = abi.bwd_detached(c.cfg(), c.theta, c.pack, c.x0, c.wY, c.wZ)
    assert n == 3 * 3 + 1
    M.check_grad(g, c.oracle()["grad"], c.blocks(), "tc1 non-adaptive wZ")


@pytest.mark.parametrize("flush", ["1", "7"])
@pytest.mark.parametrize("kern", ["tc2", "tc1"])
def test_flush_period(abi, sms, kern, flush, monkeypatch):
    """G3: PSPDE_GRAD_FLUSH_STAGES = 1 (tc2 defers its D1 flush on every stage) and 7 (divides no CTA's stage count:
    1 976 / 1 972 per full wave, 16 / 12 in the last) with three CTAs (tc2 flush offsets 0, 1, 2; tc1 has none)."""
    monkeypatch.setenv("PSPDE_MAX_GRID", "3")
    monkeypatch.setenv("PSPDE_WAVE_TILES_PER_SM", "1")
    monkeypatch.setenv("PSPDE_GRAD_FLUSH_STAGES", flush)
    if kern == "tc1":
        monkeypatch.setenv("PSPDE_GRAD_PATH", "tc1")
    c = M.TcCase(abi, "c2", K_of(sms))
    g, n = abi.bwd_detached(c.cfg(), c.theta, c.pack, c.x0, c.wY)
    assert n == 3 * 3 + 1
    M.check_grad(g, c.oracle()["grad"], c.blocks(), "%s flush %s" % (kern, flush))


@pytest.mark.parametrize("part", ["all", "third"])
def test_single_rollout_step(abi, sms, grid, part, monkeypatch):
    """G4: pspde_rollout_fwd_ckpt keeps the rows of every tile (or of the first third; the rest then goes through waves
    of one tile per SM starting at tile0 = n_keep and n_keep + SMs), then pspde_grad_from_fwd_ckpt applies dL/dY_N."""
    c = M.TcCase(abi, "c2", K_of(sms))
    cfg = c.cfg()
    need, nt = abi.lib.pspde_fwd_ckpt_bytes(ctypes.byref(cfg)), n_tiles(c.K)
    assert need > 0 and need % nt == 0
    keep = nt if part == "all" else nt // 3
    if part == "third":
        monkeypatch.setenv("PSPDE_WAVE_TILES_PER_SM", "1")
    o, ck, _ = abi.fwd_ckpt(cfg, c.theta, c.pack, c.x0, ckpt_bytes=keep * (need // nt))
    m = c.oracle()
    M.check_tc_forward(o, m)
    g, n = abi.grad_from_fwd_ckpt(cfg, c.theta, c.pack, c.x0, ck, c.wY)
    n_waves = -(-(nt - keep) // sms)
    assert n == 1 + 3 * n_waves + 1 and n_waves == (0 if part == "all" else 2)
    M.check_grad(g, m["grad"], c.blocks(), "single rollout " + part)


def test_gradient_shards(abi, sms, grid):
    """G5: two k_offset shards split inside a tile (128 x SMs + 45): the summed gradient matches the oracle of the whole
    batch and the per-path outputs equal the unsharded run's."""
    c = M.TcCase(abi, "c2", K_of(sms))
    whole, _, _ = abi.fwd_ckpt(c.cfg(), c.theta, c.pack, c.x0)
    cut = 128 * sms + 45
    outs, grad = [], 0.0
    for lo, hi in ((0, cut), (cut, c.K)):
        cfg = c.cfg(K_local=hi - lo, k_offset=lo)
        outs.append(abi.fwd_ckpt(cfg, c.theta, c.pack, c.x0)[0])
        grad = grad + abi.bwd_detached(cfg, c.theta, c.pack, c.x0, c.wY[lo:hi])[0].astype(np.float64)
    for k in ("X", "Y", "gX", "Zsum"):
        assert np.array_equal(np.concatenate([o[k] for o in outs]), whole[k]), k
    M.check_grad(grad, c.oracle()["grad"], c.blocks(), "shards")


# -------------------------------------------------------------------------------------------------------- workspace
def test_forward_workspace_bounds(abi, sms, monkeypatch):
    """W1: with PSPDE_MAX_GRID=3 the tensor-core forward launches 3 CTAs, so its stats rows fit a workspace of exactly
    pspde_workspace_bytes_fwd: pspde_rollout_fwd and pspde_importance_sampling leave the sentinel behind it alone.  A
    workspace sized with the hook is refused (-7) by the checkpointed backward once the hook is unset."""
    monkeypatch.setenv("PSPDE_MAX_GRID", "3")
    lib = abi.lib
    c = M.TcCase(abi, "lqgc7", K_of(sms))
    cfg = c.cfg()
    K, d = c.K, c.d
    nb = lib.pspde_workspace_bytes_fwd(ctypes.byref(cfg))
    assert 0 < nb < sms * 4 * 8 and nb % 8 == 0
    sentinel = 0x3A5A5A5AA5A5A5A5
    buf = pt.full(((nb + (64 << 10)) // 8,), sentinel, dtype=pt.int64, device="cuda")
    ins = [abi.dev(a) for a in (c.theta, c.pack, c.x0)]
    o = abi._out(dict(X=(K, d), Y=K, gX=K, Zsum=K, stats=4, Fint=K))
    n0 = lib.pspde_launch_count()
    L.check(lib, lib.pspde_rollout_fwd(ctypes.byref(cfg), *[abi.p(a) for a in ins], None, None, abi.p(o["X"]),
                                       abi.p(o["Y"]), abi.p(o["gX"]), abi.p(o["Zsum"]), abi.p(o["stats"]), abi.p(buf), nb,
                                       None))
    assert lib.pspde_launch_count() - n0 == 3
    f = abi._host_all(o)
    tail = buf[nb // 8:]
    assert bool((tail == sentinel).all()), "forward wrote %d B past its workspace" % (8 * int((tail != sentinel).nonzero().max() + 1))
    M.check_stats(f)
    M.check_tc_forward(f, c.oracle())
    o2 = abi._out(dict(X=(K, d), Y=K, gX=K, Fint=K))
    L.check(lib, lib.pspde_importance_sampling(ctypes.byref(cfg), *[abi.p(a) for a in ins], None, None, ctypes.c_float(0.0),
                                               abi.p(o2["X"]), abi.p(o2["Y"]), abi.p(o2["gX"]), abi.p(o2["Fint"]),
                                               abi.p(buf), nb, None))
    is_ = abi._host_all(o2)
    assert bool((tail == sentinel).all()), "importance sampling wrote past its workspace"
    for k in ("X", "Y", "gX"):
        assert np.array_equal(is_[k], f[k]), k
    ws_hook = lib.pspde_workspace_bytes(ctypes.byref(cfg))
    monkeypatch.delenv("PSPDE_MAX_GRID")
    assert 0 < ws_hook < lib.pspde_workspace_bytes(ctypes.byref(cfg))
    ws = abi.ws(ws_hook)
    grad = abi.zeros(lib.pspde_theta_size(ctypes.byref(cfg)))
    wY = abi.dev(c.wY)
    rc = lib.pspde_rollout_bwd_detached(ctypes.byref(cfg), *[abi.p(a) for a in ins], None, abi.p(wY), None, abi.p(grad),
                                        abi.p(ws), ws_hook, None)
    assert rc == -7, (rc, lib.pspde_last_error())
