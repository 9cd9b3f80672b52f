"""Cases shared by test_emu_att_multitile.py (host emulator) and test_gpu_att_multitile.py (sm_100a build): the attached
adjoint kernel rollout_attached_kernel (detach_forward=False) across network geometries, launch options and dropped
trajectories with several tiles per CTA, against the fp64 discrete adjoint (oracle/manual.py::grad_attached).

The kernel is the only implementation of the attached process, and it has geometry- and option-dependent code that the
detached kernels do not share: the input cotangent dx (every layer of a DenseNet, layer 0 of a tanh MLP), its own
shared-memory layout with the lambda tile (which decides between one CTA per SM and the register-capped two-CTA build),
the row-by-row checkpoint reload for d > 128, the injected draws restaged by the backward sweep, the u_L2 diagnostic
of the forward sweep and the in-launch zeroing of a dropped path's cotangents.  ATT_SHAPES spans those regimes and every
case asserts the plan it claims (att_plan), so that a later change of a shape or a threshold cannot silently drop
coverage.

Two forms run every case: 'pp' (per-path cotangents wY, wZ, wG: the general loss, one adjoint launch) and 're'
(relative entropy in one launch: wY = 0, wZ = wG = w = 1 / K_global)."""
import ctypes

import numpy as np

import fma_cases as F
import multitile as M
from conftest import relerr
from oracle import manual as man
from pspde import _lib as L

# id: (problem, d, network, hidden widths, dt, dense A/B off-diagonal scale, 'outer' mode)
ATT_SHAPES = {
    "L1":   ("lqgc", 10, "densenet", (), 0.05, 0.0, False),             # linear control: dx from zeta alone
    "L2":   ("lqgc", 10, "densenet", (100,), 0.05, 0.0, False),         # one wide hidden layer
    "L4":   ("lqgc", 16, "densenet", (16, 16, 16), 0.05, 0.0, False),   # dx sums three hidden deltas + zeta
    "DW4":  ("dwm", 20, "densenet", (24, 24, 24), 0.005, 0.0, False),   # double-well Jacobian / terminal gradient, L = 4
    "AB40": ("llgc", 40, "densenet", (30, 30), 0.02, 0.05, False),      # two-CTA build with leftovers, dense lambda update
    "L4X":  ("lqgc", 24, "densenet", (32, 32, 32), 0.02, 0.0, False),   # just over the two-CTA threshold
    "W64":  ("lqgc", 20, "densenet", (64, 64), 0.02, 0.0, False),
    "M4":   ("lqgc", 32, "mlp_tanh", (64, 64, 64), 0.02, 0.0, False),   # tanh, L = 4: dx from layer 0 only
    "B224": ("llgc", 64, "densenet", (32, 32), 0.01, 0.0, False),       # top of the 256-thread build
    "B225": ("lqgc", 20, "densenet", (48, 48, 48), 0.02, 0.0, False),   # bottom of the 512-thread build, L = 4
    "W160": ("lqgc", 160, "mlp_tanh", (16, 16), 0.02, 0.0, False),      # d > 128: row-by-row reload, 5 lambda reaches
    "OUT1": ("lqgc", 10, "densenet", (), 0.05, 0.0, True),              # 'outer': per-step flush, L = 1
    "OUT4": ("lqgc", 10, "densenet", (16, 16, 16), 0.05, 0.0, True),    # 'outer', L = 4
    "C3":   ("dwm", 50, "mlp_tanh", (30, 30), 0.005, 0.0, False),       # C3's shape (DoubleWell d = 50)
}
# id: (weight-gradient blocks, threads, bw_slot_rows regime, CTAs per SM, shared memory bytes)
ATT_PLAN = {
    "L1":   (4, 256, ("row-split", 32), 2, 16352),
    "L2":   (54, 256, ("row-split", 4), 2, 77152),
    "L4":   (48, 256, ("row-split", 4), 2, 59920),
    "DW4":  (90, 256, ("row-split", 2), 2, 84608),
    "AB40": (134, 256, ("leftovers", 4, 6, 16), 2, 114736),
    "L4X":  (144, 256, ("leftovers", 4, 16, 8), 1, 116592),
    "W64":  (169, 256, ("leftovers", 5, 9, 8), 1, 132608),
    "M4":   (220, 256, ("leftovers", 6, 28, 2), 1, 198096),
    "B224": (224, 256, ("exact", 7), 1, 162640),
    "B225": (225, 512, ("row-split", 2), 1, 154880),
    "W160": (108, 256, ("row-split", 2), 1, 220624),
    "OUT1": (4, 256, ("row-split", 32), 2, 16352),
    "OUT4": (40, 256, ("row-split", 4), 2, 48608),
    "C3":   (72, 256, ("row-split", 2), 2, 108032),
}
ATT_LAUNCHES = 3                # rollout_attached_kernel + reduce_stats_kernel + reduce_grad_image_kernel
MAX_SMEM = 227 * 1024           # opt-in dynamic shared memory per CTA (api_common.h kMaxSmem)


def att_smem(kind, dims, d, P=M.P_HJB):
    """Bytes of smem_layout(g, P, bwd=true, attached=true) (csrc/rollout_kernels.cuh): weights, act, z, xi, delta, lambda,
    scalars (8 P), problem (7 ceil4(d)), red (16) and zero (4) regions, with the strides of build_geom
    (csrc/pspde_geom.h: segments padded to 4, leading dimensions the next s % 8 == 4)."""
    c4 = lambda x: (x + 3) & ~3
    cf = lambda x: c4(x) if c4(x) % 8 == 4 else c4(x) + 4
    nl = len(dims) - 1
    seg = [c4(dims[s] + (1 if (kind == "mlp_tanh" or s == 0) else 0)) for s in range(nl)]
    col = sum(seg)
    lda, ldz, ldd = cf(col), cf(dims[nl]), cf(col - seg[0] if nl > 1 else 4)
    w = sum((sum(seg[:l + 1]) if kind == "densenet" else seg[l]) * c4(dims[l + 1]) for l in range(nl))
    return 4 * (w + P * lda + 3 * P * ldz + P * ldd + 8 * P + 7 * c4(d) + 16 + 4)


def att_plan(kind, dims, d):
    """(blocks, threads, regime, CTAs per SM, shared memory bytes) of the attached plan, restating make_plan
    (csrc/api_common.h: 256 threads for <= 224 blocks, 512 for <= 512; two CTAs per SM with 256 threads when
    2 (smem + 1024) <= 227 KB + 1024, i.e. smem <= 115 712 B; refused above 227 KB: CTAs = 0) and, for the regime,
    bw_slot_rows (fma_cases.fma_plan)."""
    T, regime = F.fma_plan(kind, dims)
    smem = att_smem(kind, dims, d)
    ctas = 0 if smem > MAX_SMEM else 2 if (T == 256 and 2 * (smem + 1024) <= MAX_SMEM + 1024) else 1
    return M.n_grad_blocks(kind, dims), T, regime, ctas, smem


def shape_dims(shape):
    d, arch, outer = ATT_SHAPES[shape][1], ATT_SHAPES[shape][3], ATT_SHAPES[shape][6]
    return [d if outer else d + 1] + list(arch) + [d]


def ctas_per_sm(shape):
    return ATT_PLAN[shape][3]


def _cot(rng, K):
    return rng.choice([-1.0, 1.0], K) * (0.5 + rng.uniform(0, 1, K)) / K


class AttCase:
    """Inputs of one attached case: K paths from k_offset 0, the network (theta scaled by fan-in), independent random-sign
    per-path cotangents wY, wZ, wG with every 7th path all zero (none of the three cotangent paths can hide behind
    cancellation or behind another's term), the kernels' Philox increments and a u_L2 table; `oracle()` is the fp64
    rollout + discrete adjoint (man.grad_attached) on them, chunked over paths and cached.
      x0_per_path, y0: one start point per path (around the problem's X_0), a start value of Y."""

    def __init__(self, abi, shape, K, N, x0_per_path=False, y0=None, seed=5, offset=3):
        kind, d, net, arch, dt, off_diag, outer = ATT_SHAPES[shape]
        self.shape, self.kind, self.d, self.net, self.K, self.N = shape, kind, d, net, K, N
        self.dt, self.seed, self.offset, self.y0, self.outer = np.float32(dt), seed, offset, y0, outer
        self.n_sets = N if outer else 1
        self.dims = shape_dims(shape)
        self.mp, (self.pid, self.flags, self.pack), self.x0 = M.hjb_problem(kind, d, off_diag, seed)
        rng = np.random.default_rng(seed)
        self.theta = F.fan_in_theta(net, self.dims, self.n_sets, rng)
        assert self.theta.size == abi.lib.pspde_theta_size(ctypes.byref(self.cfg())), abi.lib.pspde_last_error()
        self.wY, self.wZ, self.wG = (_cot(rng, K).astype(np.float32) for _ in range(3))
        for w in (self.wY, self.wZ, self.wG):
            w[::7] = 0.0
        if x0_per_path:
            self.x0 = (self.x0 + 0.5 * rng.standard_normal((K, d))).astype(np.float32)
        self.table = (0.3 * rng.standard_normal((2 * N, d))).astype(np.float32)
        self.xi_dump = abi.philox_dump(self.cfg())                   # (N, K, d)

    def cfg(self, K_local=None, k_offset=0, inject=False, d_abs_max=0.0, x0_per_path=None):
        strides = (self.d * (self.N + 1), self.N + 1, 1) if inject else (0, 0, 0)
        return L.make_cfg(self.K if K_local is None else K_local, self.d, self.N, self.dt, self.pid,
                          L.NET_DENSENET if self.net == "densenet" else L.NET_MLP_TANH, self.dims,
                          L.TIME_NONE if self.outer else L.TIME_FIRST, adaptive=True, k_offset=k_offset,
                          problem_flags=self.flags, noise_mode=L.NOISE_INJECT if inject else L.NOISE_PHILOX,
                          seed=self.seed, offset=self.offset, xi_strides=strides,
                          x0_per_path=self.x0.ndim == 2 if x0_per_path is None else x0_per_path,
                          n_sets=self.n_sets if self.outer else 0, d_abs_max=d_abs_max)

    def plan(self):
        return att_plan(self.net, self.dims, self.d)

    def check_plan(self):
        """The block count, thread build, regime, CTAs per SM and shared memory this case claims (ATT_PLAN); it fits."""
        assert self.plan() == ATT_PLAN[self.shape], (self.plan(), ATT_PLAN[self.shape])
        assert ATT_PLAN[self.shape][3] > 0

    def nets(self):
        nth = self.theta.size // self.n_sets
        th = self.theta.astype(np.float64)
        nets = [man.Net(self.net, self.dims, th[s * nth:(s + 1) * nth]) for s in range(self.n_sets)]
        return nets if self.outer else nets[0]

    def blocks(self):
        return M.grad_blocks(self.net, self.dims, self.n_sets)

    def xi_ref(self, lo=0, hi=None):
        """The Philox increments of paths [lo, hi) in the reference layout (K, d, N + 1), float32."""
        xi = np.zeros((self.K if hi is None else hi - lo, self.d, self.N + 1), np.float32)
        xi[:, :, 1:] = self.xi_dump[:, lo:hi].transpose(1, 2, 0)
        return xi

    def cotangents(self, form, drop=None):
        """(wY, wZ, wG) of the form in fp64 ('re': 0, w, w with the kernel's float32 w = 1 / K); zero on `drop`."""
        if form == "re":
            w = float(np.float32(1.0 / self.K))
            ws = [np.zeros(self.K), np.full(self.K, w), np.full(self.K, w)]
        else:
            ws = [a.astype(np.float64) for a in (self.wY, self.wZ, self.wG)]
        if drop is not None:
            for a in ws:
                a[drop] = 0.0
        return ws

    def run(self, abi, form, K_local=None, k_offset=0, inject=False, table=False, d_abs_max=0.0, x0=None):
        """One attached launch of paths [k_offset, k_offset + K_local) in `form`; asserts the launch count."""
        lo, hi = k_offset, k_offset + (self.K if K_local is None else K_local)
        x0 = self.x0 if x0 is None else x0
        cfg = self.cfg(hi - lo, lo, inject, d_abs_max, x0.ndim == 2)
        kw = dict(y0=self.y0, xi=self.xi_ref(lo, hi) if inject else None, table=self.table if table else None)
        xl = x0[lo:hi] if x0.ndim == 2 else x0
        if form == "re":
            o, n = abi.attached(cfg, self.theta, self.pack, xl, 1.0 / self.K, **kw)
        else:
            o, n = abi.attached(cfg, self.theta, self.pack, xl, 0.0, self.wY[lo:hi], self.wZ[lo:hi], self.wG[lo:hi], **kw)
        assert n == ATT_LAUNCHES, n
        return o

    def oracle(self, form, drop=None, x0=None, chunk=4096):
        """fp64: X_N, Y_N, g(X_N), Z_sum, u_L2 per path and the gradient of the loss given by the form's cotangents (zero
        on `drop`), from the start points x0 (default the case's)."""
        x0 = (self.x0 if x0 is None else x0).astype(np.float64)
        key = ("att", self.shape, self.K, self.N, form, self.seed, self.offset, self.y0, x0.shape, hash(x0.tobytes()),
               None if drop is None else hash(np.asarray(drop).tobytes()))
        if key in M._ORACLE:
            return M._ORACLE[key]
        wY, wZ, wG = self.cotangents(form, drop)
        nets, dt = self.nets(), float(self.dt)
        y0 = float(np.float32(self.y0 or 0.0))
        parts = []
        for lo in range(0, self.K, chunk):
            hi = min(self.K, lo + chunk)
            g, ro = man.grad_attached(self.mp, nets, self.xi_ref(lo, hi).astype(np.float64), dt, self.N,
                                      x0[lo:hi] if x0.ndim == 2 else x0, wY[lo:hi], wZ[lo:hi], wG[lo:hi],
                                      "none" if self.outer else "first", y0)
            parts.append(dict(grad=g, uL2=M.u_l2(self.table, ro, dt), **{k: ro[k] for k in ("X", "Y", "gX", "Zsum")}))
        out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "grad"}
        out["grad"] = sum(p["grad"] for p in parts)
        M._ORACLE[key] = out
        return out


PER_PATH = ("X", "Y", "gX", "Zsum")


def check_outputs(o, m, kept=None):
    """Per-path outputs of an attached launch against the oracle (on the kept paths), and its stats: stats[2] is the sum
    of Z_sum + g(X_N) over the kept paths, stats[3] counts the dropped ones."""
    kept = np.ones(len(o["Y"]), bool) if kept is None else kept
    assert relerr(o["X"][kept], m["X"][kept]) < M.TOL_END, ("X_N", relerr(o["X"][kept], m["X"][kept]))
    for k in ("Y", "gX", "Zsum"):
        assert relerr(o[k][kept], m[k][kept]) < M.TOL_PATH, (k, relerr(o[k][kept], m[k][kept]))
    v = o["Zsum"][kept].astype(np.float64) + o["gX"][kept]
    assert o["stats"][3] == (~kept).sum(), (o["stats"][3], (~kept).sum())
    assert abs(o["stats"][2] - v.sum()) <= 1e-9 * np.abs(v).sum(), (o["stats"][2], v.sum())


def check_launch(o, m, blocks, what, kept=None):
    check_outputs(o, m, kept)
    M.check_grad(o["grad"], m["grad"], blocks, what)


def same(a, b, keys=PER_PATH + ("stats", "grad")):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def geometry_case(abi, shape, K, N, form, monkeypatch=None):
    """§ geometry sweep: one attached launch of a shape against the oracle (per-path outputs, stats, the gradient as a
    whole and per (set, layer) block, the launch count) and a second launch bit-equal to the first.  For a two-CTA shape
    also with PSPDE_ATT_CTAS=1: against the oracle, and per-path outputs bit-equal to the two-CTA run."""
    c = AttCase(abi, shape, K, N)
    c.check_plan()
    m = c.oracle(form)
    o = c.run(abi, form)
    check_launch(o, m, c.blocks(), "%s %s" % (shape, form))
    same(c.run(abi, form), o)
    if ctas_per_sm(shape) == 2:
        monkeypatch.setenv("PSPDE_ATT_CTAS", "1")
        o1 = c.run(abi, form)
        check_launch(o1, m, c.blocks(), "%s %s one CTA per SM" % (shape, form))
        same(o1, o, PER_PATH)


def inject_case(abi, shape, K, N):
    """The Philox draws fed back as injected noise (reference layout (K, d, N + 1)), per-path form: against the oracle, and
    bit-equal to the Philox run (the kernel consumes the same floats in both sweeps)."""
    c = AttCase(abi, shape, K, N)
    o = c.run(abi, "pp", inject=True)
    check_launch(o, c.oracle("pp"), c.blocks(), "%s injected" % shape)
    same(o, c.run(abi, "pp"))


def start_case(abi, shape, K, N, form):
    """Per-path X_0 and a start value y_0 against the oracle."""
    c = AttCase(abi, shape, K, N, x0_per_path=True, y0=0.25)
    check_launch(c.run(abi, form), c.oracle(form), c.blocks(), "%s %s x0/y0" % (shape, form))


def shard_case(abi, shape, K, N, form, cut):
    """Two k_offset shards cut inside a tile (w = 1 / K_global in the 're' form): per-path outputs equal the unsharded
    run's bit for bit, the summed gradient matches the whole-batch oracle per block."""
    assert cut % M.P_HJB != 0
    c = AttCase(abi, shape, K, N)
    whole = c.run(abi, form)
    outs, grad = [], 0.0
    for lo, hi in ((0, cut), (cut, K)):
        o = c.run(abi, form, hi - lo, lo)
        outs.append(o)
        grad = grad + o["grad"].astype(np.float64)
    for k in PER_PATH:
        assert np.array_equal(np.concatenate([o[k] for o in outs]), whole[k]), k
    m = c.oracle(form)
    check_outputs(whole, m)
    M.check_grad(grad, m["grad"], c.blocks(), "%s %s shards" % (shape, form))


def ul2_case(abi, shape, K, N):
    """pspde_rollout_attached_diag with a mode-1 table, relative-entropy form: u_L2 per path against its restatement
    (multitile.u_l2); outputs and gradient bit-equal to the launch without the diagnostic."""
    c = AttCase(abi, shape, K, N)
    o = c.run(abi, "re", table=True)
    m = c.oracle("re")
    assert o["uL2"].min() > 0
    assert relerr(o["uL2"], m["uL2"]) < M.TOL_PATH, relerr(o["uL2"], m["uL2"])
    same(o, c.run(abi, "re"))
    check_launch(o, m, c.blocks(), "%s u_L2" % shape)


def dropped_case(abi, shape, K, N, form, n_blowup=6):
    """The blow-up bound d_abs_max and non-finite trajectories, dropped inside the launch.  n_blowup paths spread over
    revisited tiles start at 1e20 (non-finite at X_N); the bound is the midpoint of two neighbouring sorted |D| values
    near the 80th percentile (D = Y_N - g(X_N) in fp64 as the kernel forms it), so the split is exact and falls in every
    tile.  Against the run without a bound: stats[3] counts the dropped paths, Y_N is NaN exactly there, every other
    per-path output is bit-equal and stats[2] sums the kept paths; the gradient matches the oracle with zero cotangents
    on the dropped paths (whose 1e20 starts are 0 there, so that 0 * inf cannot poison it)."""
    c = AttCase(abi, shape, K, N)
    x0 = np.tile(c.x0, (K, 1)).astype(np.float32)
    big = np.linspace(K // 2, K - 3, n_blowup).astype(int)        # tiles past the first wave of CTAs
    x0[big] = 1e20
    free = c.run(abi, form, x0=x0)
    D = free["Y"].astype(np.float64) - free["gX"]
    fin = np.isfinite(D) & np.isfinite(free["Zsum"])
    assert np.array_equal(~fin, np.isin(np.arange(K), big)), "only the 1e20 starts blow up"
    a = np.sort(np.abs(D[fin]))
    i = int(0.8 * a.size)
    while not (a[i] < np.float32(0.5 * (a[i] + a[i + 1])) < a[i + 1]):
        i += 1
    bound = np.float32(0.5 * (a[i] + a[i + 1]))
    drop = ~fin | (np.abs(D) >= bound)
    n_tiles = (K + M.P_HJB - 1) // M.P_HJB
    assert all(drop[t * M.P_HJB:(t + 1) * M.P_HJB].any() for t in range(n_tiles)), "a tile without a dropped path"
    assert int(free["stats"][3]) == n_blowup
    o = c.run(abi, form, d_abs_max=float(bound), x0=x0)
    assert o["stats"][3] == drop.sum(), (o["stats"][3], drop.sum())
    assert np.array_equal(np.isnan(o["Y"]), drop)
    for k in PER_PATH:
        assert np.array_equal(o[k][~drop], free[k][~drop]), k
    for k in ("X", "gX", "Zsum"):
        assert np.array_equal(o[k], free[k], equal_nan=True), k
    v = o["Zsum"][~drop].astype(np.float64) + o["gX"][~drop]
    assert abs(o["stats"][2] - v.sum()) <= 1e-9 * np.abs(v).sum(), (o["stats"][2], v.sum())
    x0m = x0.copy()
    x0m[big] = 0.0
    m = c.oracle(form, drop=drop, x0=x0m)
    check_launch(o, m, c.blocks(), "%s %s dropped" % (shape, form), kept=~drop)
