"""Cases shared by test_emu_fma_multitile.py (host emulator) and test_gpu_fma_multitile.py (sm_100a build): the FP32-FMA
detached rollout kernels -- rollout_kernel<64, 512, false, 1> (forward, importance sampling) and rollout_kernel<64, 256 |
512, true, 1> (recompute backward) reduced by reduce_grad_image_kernel -- across network geometries with several tiles
per CTA, against the fp64 oracle (oracle/manual.py).

The library sends every configuration outside the tensor-core shape class to these kernels: 'outer' mode, dense A / B,
d > 102, any control network but two hidden layers of width <= 32.  Most of their index logic depends on the geometry:
the thread build, the block -> lane assignment of the weight gradient (bw_slot_rows), the forward row tile and the
layer count.  FMA_SHAPES spans those regimes and every case asserts the regime it claims (fma_plan), so that a later
change of a shape or a threshold cannot silently drop coverage."""
import ctypes

import numpy as np

import multitile as M
from conftest import relerr
from oracle import manual as man
from pspde import _lib as L

# id: (problem, d, network, hidden widths, dt, dense A/B off-diagonal scale, tensor-core eligible), and the expected
# (weight-gradient blocks, backward threads, bw_slot_rows regime).  Tensor-core-eligible shapes (two hidden layers of
# width <= 32, d <= 102, diagonal A / B) are forced onto the FMA kernels with PSPDE_FWD_PATH / PSPDE_BWD_PATH=simt.
FMA_SHAPES = {
    "L1":   ("lqgc", 10, "densenet", (), 0.05, 0.0, False),             # L = 1: linear control, no hidden cotangents
    "L2":   ("lqgc", 10, "densenet", (100,), 0.05, 0.0, False),         # L = 2, one wide hidden layer
    "C1i":  ("lqgc", 10, "densenet", (30, 30), 0.05, 0.0, True),        # C1's network in 'inner' mode
    "C3s":  ("dwm", 50, "mlp_tanh", (30, 30), 0.005, 0.0, True),        # tanh, a bias column in every segment
    "W64":  ("lqgc", 20, "densenet", (64, 64), 0.02, 0.0, False),       # 256 threads, full warps + leftovers
    "B224": ("llgc", 64, "densenet", (32, 32), 0.01, 0.0, True),        # top of the 256-thread build
    "B225": ("lqgc", 20, "densenet", (48, 48, 48), 0.02, 0.0, False),   # L = 4, bottom of the 512-thread build
    "M4":   ("lqgc", 32, "mlp_tanh", (64, 64, 64), 0.02, 0.0, False),   # tanh with three hidden layers
    "C2s":  ("llgc", 100, "densenet", (30, 30), 0.01, 0.0, True),       # C2 / C5 shape on the FMA kernels
    "D106": ("llgc", 106, "densenet", (30, 30), 0.01, 0.0, False),      # largest d of DenseNet [30, 30] whose backward fits
    "AB":   ("llgc", 40, "densenet", (30, 30), 0.02, 0.05, False),      # dense A / B
    "OUT":  ("lqgc", 10, "densenet", (30, 30), 0.05, 0.0, False),       # 'outer': one parameter set per step
}
FMA_PLAN = {
    "L1": (4, 256, ("row-split", 32)),
    "L2": (54, 256, ("row-split", 4)),
    "C1i": (52, 256, ("row-split", 4)),
    "C3s": (72, 256, ("row-split", 2)),
    "W64": (169, 256, ("leftovers", 5, 9, 8)),
    "B224": (224, 256, ("exact", 7)),
    "B225": (225, 512, ("row-split", 2)),
    "M4": (220, 256, ("leftovers", 6, 28, 2)),
    "C2s": (393, 512, ("leftovers", 12, 9, 8)),
    "D106": (436, 512, ("leftovers", 13, 20, 4)),
    "AB": (134, 256, ("leftovers", 4, 6, 16)),
    "OUT": (52, 256, ("row-split", 4)),
}
FWD_LAUNCHES = 2                # FMA forward: rollout_kernel + reduce_stats_kernel (tensor-core forward: 3)
BWD_LAUNCHES = 2                # FMA backward: rollout_kernel<BWD> + reduce_grad_image_kernel (checkpointed: >= 4)
IS_LAUNCHES = 1                 # FMA importance sampling: rollout_kernel alone


def fma_plan(kind, dims, P=M.P_HJB):
    """(threads of the backward build, bw_slot_rows regime) for a network: restates make_plan (csrc/api_common.h:136-141:
    256 threads for <= 224 blocks, 512 for <= 512, refused above) and bw_slot_rows (csrc/rollout_kernels.cuh:297-318):
      ('row-split', cpb)                when 2 nb <= threads: every block's rows over cpb interleaved lanes;
      ('leftovers', warps, rem, cpb)    whole warps own one block per lane, the rem = nb mod 32 leftover blocks are
                                        row-split over cpb lanes of the idle warps;
      ('exact', warps)                  nb is a multiple of 32: no leftovers."""
    nb = M.n_grad_blocks(kind, dims)
    T = 256 if nb <= 224 else 512 if nb <= 512 else None
    if T is None:
        return None, None
    if 2 * nb <= T:
        cpb = 2
        while cpb * 2 <= 32 and cpb * 2 <= P and cpb * 2 * nb <= T:
            cpb *= 2
        return T, ("row-split", cpb)
    full = nb & ~31
    rem = nb - full
    if rem == 0:
        return T, ("exact", full // 32)
    cpb = 1
    while cpb * 2 <= 32 and cpb * 2 <= P and cpb * 2 * rem <= T - full:
        cpb *= 2
    return T, ("leftovers", full // 32, rem, cpb)


def shape_dims(shape):
    kind, d, net, arch = FMA_SHAPES[shape][:4]
    return [d if shape == "OUT" else d + 1] + list(arch) + [d]


def use_fma_paths(shape, monkeypatch):
    """Force the FMA kernels for a tensor-core-eligible shape; the others take their natural route."""
    if FMA_SHAPES[shape][6]:
        monkeypatch.setenv("PSPDE_FWD_PATH", "simt")
        monkeypatch.setenv("PSPDE_BWD_PATH", "simt")


def fan_in_theta(net, dims, n_sets, rng, gain=0.6):
    """Parameters of n_sets networks, each (W_l, b_l) block drawn with standard deviation gain / sqrt(fan_in + 1)."""
    blocks = M.grad_blocks(net, dims, n_sets)
    theta = np.zeros(blocks[-1].stop)
    for i, s in enumerate(blocks):
        l = i % (len(dims) - 1)
        fan_in = sum(dims[:l + 1]) if net == "densenet" else dims[l]
        theta[s] = gain / np.sqrt(fan_in + 1) * rng.standard_normal(s.stop - s.start)
    return theta.astype(np.float32)


class FmaCase:
    """Inputs of one FMA case: K paths from k_offset 0, the network (theta scaled by fan-in), random-sign cotangents with
    every 7th path exactly zero, the kernels' Philox increments; `oracle()` is the fp64 rollout + gradient
    (man.grad_mode_a) on them, chunked over paths and cached.
      time:      'inner' (t is the first input) or 'outer' (n_sets parameter sets, default N; step n uses set n)
      adaptive:  the controlled process (c = -Z) or the uncontrolled one; wz: a cotangent on Z_sum too
      x0_per_path, y0: one start point per path (around the problem's X_0), a start value of Y"""

    def __init__(self, abi, shape, K, N, adaptive=True, wz=False, x0_per_path=False, y0=None, n_sets=None, seed=5,
                 offset=3):
        kind, d, net, arch, dt, off_diag, _ = FMA_SHAPES[shape]
        self.shape, self.kind, self.d, self.net, self.K, self.N = shape, kind, d, net, K, N
        self.dt, self.adaptive, self.seed, self.offset, self.y0 = np.float32(dt), adaptive, seed, offset, y0
        self.outer = shape == "OUT"
        self.n_sets = (n_sets or N) if self.outer else 1
        self.dims = shape_dims(shape)
        self.mp, (self.pid, self.flags, self.pack), self.x0 = M.hjb_problem(kind, d, off_diag, seed)
        rng = np.random.default_rng(seed)
        self.theta = fan_in_theta(net, self.dims, self.n_sets, rng)
        assert self.theta.size == abi.lib.pspde_theta_size(ctypes.byref(self.cfg())), abi.lib.pspde_last_error()
        self.wY = (rng.choice([-1.0, 1.0], K) * (0.5 + rng.uniform(0, 1, K)) / K).astype(np.float32)
        self.wZ = (rng.standard_normal(K) / K).astype(np.float32) if wz else None
        for w in (self.wY, self.wZ):
            if w is not None:
                w[::7] = 0.0
        if x0_per_path:
            self.x0 = (self.x0 + 0.5 * rng.standard_normal((K, d))).astype(np.float32)
        self.xi_dump = abi.philox_dump(self.cfg())                   # (N, K, d)

    def cfg(self, K_local=None, k_offset=0):
        return L.make_cfg(self.K if K_local is None else K_local, self.d, self.N, self.dt, self.pid,
                          L.NET_DENSENET if self.net == "densenet" else L.NET_MLP_TANH, self.dims,
                          L.TIME_NONE if self.outer else L.TIME_FIRST, adaptive=self.adaptive, k_offset=k_offset,
                          problem_flags=self.flags, noise_mode=L.NOISE_PHILOX, seed=self.seed, offset=self.offset,
                          x0_per_path=self.x0.ndim == 2, n_sets=self.n_sets if self.outer else 0)

    def nets(self):
        nth = self.theta.size // self.n_sets
        th = self.theta.astype(np.float64)
        nets = [man.Net(self.net, self.dims, th[s * nth:(s + 1) * nth]) for s in range(self.n_sets)]
        return nets if self.outer else nets[0]

    def blocks(self):
        return M.grad_blocks(self.net, self.dims, self.n_sets)

    def oracle(self, t_index=None, dt_net=None, chunk=4096):
        """fp64: X_N, Y_N, g(X_N), Z_sum, Fint per path and the gradient of sum_k wY_k Y_N,k + wZ_k Z_sum,k; with t_index
        the network of step n is evaluated at t_index[n] dt_net (importance sampling on the network's grid)."""
        key = ("fma", self.shape, self.K, self.N, self.adaptive, self.wZ is not None, self.x0.ndim, self.y0,
               self.n_sets, self.seed, self.offset, None if t_index is None else tuple(t_index), dt_net)
        if key in M._ORACLE:
            return M._ORACLE[key]
        nets, dt = self.nets(), float(self.dt)
        wZ = np.zeros(self.K) if self.wZ is None else self.wZ.astype(np.float64)
        x0 = self.x0.astype(np.float64)
        y0 = float(np.float32(self.y0 or 0.0))
        parts = []
        for lo in range(0, self.K, chunk):
            hi = min(self.K, lo + chunk)
            xi = np.zeros((hi - lo, self.d, self.N + 1))
            xi[:, :, 1:] = self.xi_dump[:, lo:hi].transpose(1, 2, 0)
            g, ro = man.grad_mode_a(self.mp, nets, xi, dt, self.N, x0[lo:hi] if x0.ndim == 2 else x0,
                                    self.wY[lo:hi].astype(np.float64), wZ[lo:hi], self.adaptive,
                                    "none" if self.outer else "first", y0, t_index,
                                    None if dt_net is None else float(np.float32(dt_net)))
            parts.append(dict(grad=g, **{k: ro[k] for k in ("X", "Y", "gX", "Zsum", "Fint")}))
        out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "grad"}
        out["grad"] = sum(p["grad"] for p in parts)
        M._ORACLE[key] = out
        return out

    def check_plan(self):
        """The thread build and bw_slot_rows regime this case claims (FMA_PLAN)."""
        nb, T, regime = FMA_PLAN[self.shape]
        assert M.n_grad_blocks(self.net, self.dims) == nb
        assert fma_plan(self.net, self.dims) == (T, regime), fma_plan(self.net, self.dims)

    def forward(self, abi, K_local=None, k_offset=0):
        lo, hi = k_offset, k_offset + (self.K if K_local is None else K_local)
        x0 = self.x0[lo:hi] if self.x0.ndim == 2 else self.x0
        o, _, n = abi.fwd_ckpt(self.cfg(hi - lo, lo), self.theta, self.pack, x0, y0=self.y0)
        assert n == FWD_LAUNCHES, n
        return o

    def backward(self, abi, K_local=None, k_offset=0):
        lo, hi = k_offset, k_offset + (self.K if K_local is None else K_local)
        x0 = self.x0[lo:hi] if self.x0.ndim == 2 else self.x0
        wZ = None if self.wZ is None else self.wZ[lo:hi]
        g, n = abi.bwd_detached(self.cfg(hi - lo, lo), self.theta, self.pack, x0, self.wY[lo:hi], wZ)
        assert n == BWD_LAUNCHES, n
        return g


def refusal(abi, c, bwd):
    """(return code, error message, launches) of the forward or the backward of case c with a 64 KB workspace: for a
    network the plan refuses, make_plan returns before any launch."""
    ws = abi.zeros(8192, np.float64)
    out = abi.zeros(c.K * c.d)
    ins = [abi.dev(a) for a in (c.theta, c.pack, c.x0, c.wY)]
    p = [abi.p(a) for a in ins]
    n0 = abi.lib.pspde_launch_count()
    if bwd:
        rc = abi.lib.pspde_rollout_bwd_detached(ctypes.byref(c.cfg()), p[0], p[1], p[2], None, p[3], None, abi.p(out),
                                                abi.p(ws), abi.nbytes(ws), None)
    else:
        rc = abi.lib.pspde_rollout_fwd(ctypes.byref(c.cfg()), p[0], p[1], p[2], None, None, abi.p(out), abi.p(out),
                                       abi.p(out), abi.p(out), None, abi.p(ws), abi.nbytes(ws), None)
    return rc, abi.lib.pspde_last_error().decode(), abi.lib.pspde_launch_count() - n0


def refusal_case(abi, K):
    """LLGC with DenseNet [30, 30] past the FMA kernels' limits.  d = 107: the backward's tile needs more than 227 KB of
    shared memory and is refused, while the forward still fits and matches the oracle.  d = 121: the backward has
    528 > 512 weight-gradient blocks and is refused for that, and the forward for shared memory."""
    for d in (107, 121):
        FMA_SHAPES["_D%d" % d] = ("llgc", d, "densenet", (30, 30), 0.01, 0.0, False)
        try:
            c = FmaCase(abi, "_D%d" % d, K, 2)
            assert fma_plan(c.net, c.dims)[0] == (512 if d == 107 else None)
            if d == 107:
                check_forward(c.forward(abi), c.oracle())
            else:
                rc, msg, n = refusal(abi, c, False)
                assert (rc, n) == (-6, 0) and "shared memory" in msg, (rc, msg, n)
            rc, msg, n = refusal(abi, c, True)
            assert (rc, n) == (-6, 0), (rc, msg, n)
            assert ("shared memory" if d == 107 else "network too large") in msg, msg
        finally:
            del FMA_SHAPES["_D%d" % d]


def check_forward(o, m):
    """Per-path outputs of a forward against the oracle, and its stats (no path dropped)."""
    assert relerr(o["X"], m["X"]) < M.TOL_END, ("X_N", relerr(o["X"], m["X"]))
    for k in ("Y", "gX", "Zsum"):
        assert relerr(o[k], m[k]) < M.TOL_PATH, (k, relerr(o[k], m[k]))
    assert o["stats"][3] == 0
    M.check_stats(o)


def geometry_case(abi, shape, K, N, **kw):
    """§ geometry sweep: the forward and the recompute backward of one shape (launch counts prove the FMA kernels ran)
    against the oracle: per-path outputs, stats, the gradient as a whole and per (set, layer) block, and a second
    backward bit-equal to the first."""
    c = FmaCase(abi, shape, K, N, **kw)
    c.check_plan()
    m = c.oracle()
    check_forward(c.forward(abi), m)
    g = c.backward(abi)
    M.check_grad(g, m["grad"], c.blocks(), "%s %s" % (shape, kw))
    assert np.array_equal(c.backward(abi), g), "second backward differs"


def shard_case(abi, c, cut):
    """Two k_offset shards cut inside a tile, per-path start points and a start value of Y: the per-path outputs equal the
    unsharded run's bit for bit and the summed gradient matches the whole-batch oracle per block."""
    whole = c.forward(abi)
    outs, grad = [], 0.0
    for lo, hi in ((0, cut), (cut, c.K)):
        outs.append(c.forward(abi, hi - lo, lo))
        grad = grad + c.backward(abi, hi - lo, lo).astype(np.float64)
    for k in ("X", "Y", "gX", "Zsum"):
        assert np.array_equal(np.concatenate([o[k] for o in outs]), whole[k]), k
    m = c.oracle()
    check_forward(whole, m)
    M.check_grad(grad, m["grad"], c.blocks(), "shards")


def time_index(N, dt, dt_net):
    """t_index[n] = ceil(n dt / dt_net) as Solver.Z_n forms it (solver.py:360-362): the float n * dt divided in fp32 by the
    network's fp32 step.  Asserted equal to pspde.utilities._time_index."""
    import torch as pt
    from types import SimpleNamespace
    from pspde.utilities import _time_index
    ref = np.array([np.ceil(np.float32(n * float(dt)) / np.float32(dt_net)) for n in range(N)], np.int32)
    lib = _time_index(SimpleNamespace(delta_t=pt.tensor(dt_net, dtype=pt.float32)), N, float(dt)).numpy()
    assert np.array_equal(ref, lib), (ref, lib)
    return ref


def importance_sampling_case(abi, c, launches=IS_LAUNCHES, ratio=2.5):
    """pspde_importance_sampling on a network grid ratio x coarser than the step grid: X_N, Y_N, g(X_N) and Fint against
    the oracle evaluating step n's network at t_index[n] dt_net (in 'outer' mode: set min(t_index[n], n_sets - 1))."""
    dt_net = np.float32(ratio * float(c.dt))
    t_index = time_index(c.N, c.dt, dt_net)
    o, n = abi.importance_sampling(c.cfg(), c.theta, c.pack, c.x0, t_index, float(dt_net))
    if launches is not None:
        assert n == launches, n
    m = c.oracle(t_index, dt_net)
    assert relerr(o["X"], m["X"]) < M.TOL_END, ("X_N", relerr(o["X"], m["X"]))
    for k in ("Y", "gX", "Fint"):
        assert relerr(o[k], m[k]) < M.TOL_PATH, (k, relerr(o[k], m[k]))
    return t_index
