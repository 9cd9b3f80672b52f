"""Cases shared by test_emu_diff_multitile.py (host emulator) and test_gpu_diff_multitile.py (sm_100a build): the diffusion
kernels diffusion_kernel<32, 512, BWD>, pack_weights_kernel and reduce_dw_kernel (GeneralSolver, C4, and every
EllipticSolver workload) across network geometries, problem data and dropped paths with several tiles per CTA, against
the fp64 oracle (oracle/manual.py::diffusion, ::elliptic).

The kernels' index logic depends on the value network: gemm_pairs_nn deals ceil(Np / 16) column patches to 16 warps
(C4's width 256 is exactly 16, so the wrap-around never ran), gemm_pairs_nt sums the cotangent of hidden segment l + 1
over every later layer and deals 2 ceil(ceil(seg / 4) / 4) warp tiles, dw_accum_flush handles the half-blocks of ragged
widths, the output layer is a warp-strided dot product over Kp, and the host refuses a tile over 227 KB of shared
memory.  DIFF_SHAPES spans those regimes; every case asserts the regime it claims (diff_plan restates build_geom and
diff_smem_layout), so that a later change of a shape cannot silently drop coverage.

Two cotangent forms run: 'loss' (c0, cE, cD) = (-w, w, -w) with w = 2 r / K from the kernel's forward, as the solvers
form them, and 'rand' (independent random-sign c0, cE, cD, every 7th path all zero).  The oracle gets the same float32
cotangents."""
import ctypes
import re

import numpy as np

import emu_harness as H
import multitile as M
from conftest import relerr
from oracle import manual as man
from pspde import _lib as L

P = M.P_DIFF
NWARPS = 16                     # diffusion_kernel<32, 512>
MAX_SMEM = 227 * 1024           # opt-in dynamic shared memory per CTA (api_common.h kMaxSmem)

# id: (d, hidden widths); a DenseNet with scalar output, input [X, t] (parabolic) or X (elliptic)
DIFF_SHAPES = {
    "L1":    (7, ()),                   # linear V: no hidden layer, no reverse GEMM
    "H5":    (1, (5,)),                 # one ragged hidden layer, d = 1
    "H300":  (7, (300,)),               # more column patches than warps in both GEMMs
    "L4":    (7, (13, 7, 3)),           # three ragged hidden layers: gemm_pairs_nt sums three layers for segment 1
    "W40x3": (7, (40, 40, 40)),
    "NW":    (1, (3, 70)),              # a narrow layer feeding a wide one
    "C4X":   (100, (256, 256, 256)),    # C4's layers and one more at d = 100: 227 696 B, 4.6 KB under the limit
}
# id: (lda, weight-gradient blocks, shared memory bytes) of the parabolic (TIME_LAST) and elliptic (TIME_NONE) plans
DIFF_PLAN = {
    "L1":    ((12, 2, 5776), (12, 1, 5776)),
    "H5":    ((12, 3, 5744), (12, 3, 5744)),
    "H300":  ((316, 115, 83600), (308, 77, 81552)),
    "L4":    ((44, 18, 13968), (36, 14, 11920)),
    "W40x3": ((132, 122, 36496), (132, 106, 36496)),
    "NW":    ((84, 20, 24176), (84, 20, 24176)),
    "C4X":   ((876, 4429, 227696), (876, 4429, 227696)),
}
# the regime each shape is there for, on diff_plan's fields
DIFF_REGIME = {
    "L1":    lambda p: p["L"] == 1,
    "H5":    lambda p: p["L"] == 2 and p["d"] % 4 and p["ragged"],
    "H300":  lambda p: p["nn"][0] > NWARPS and p["nt"][0] > NWARPS,
    "L4":    lambda p: p["L"] == 4 and p["ragged"],
    "W40x3": lambda p: p["L"] == 4 and not p["ragged"],
    "NW":    lambda p: p["d"] % 4 and p["nn"] == [1, 5],
    "C4X":   lambda p: 227000 < p["smem"] <= MAX_SMEM and p["nn"] == [NWARPS] * 3,
}


def diff_plan(dims, d, time_mode):
    """The plan of a DenseNet value network, restating build_geom (csrc/pspde_geom.h: segment 0 = [X | t | 1] padded to 4,
    hidden segments padded to 4, lda the next s % 8 == 4) and diff_smem_layout(g, 32) (2 P rows of lda, 2 P x 4 output
    rows, 12 P scalars, 2 ceil4(d) problem floats, 16 + 4): lda, weight-gradient blocks, shared-memory bytes, and per
    hidden layer l the column patches of gemm_pairs_nn (ceil(Np / 16)) and the warp tiles of gemm_pairs_nt for segment
    l + 1 (2 ceil(ceil(seg / 4) / 4)); ragged: some hidden width is not a multiple of 8 (a half-block of dw_accum_flush
    or a column patch is partly padding)."""
    c4 = lambda x: (x + 3) & ~3
    cf = lambda x: c4(x) if c4(x) % 8 == 4 else c4(x) + 4
    nl = len(dims) - 1
    assert dims[0] == d + (1 if time_mode == L.TIME_LAST else 0) and dims[-1] == 1
    seg = [c4(dims[s] + (1 if s == 0 else 0)) for s in range(nl)]
    lda = cf(sum(seg))
    smem = 4 * (2 * P * lda + 2 * P * 4 + 12 * P + 2 * c4(d) + 16 + 4)
    w_floats = sum(sum(seg[:l + 1]) * c4(dims[l + 1]) for l in range(nl))
    return dict(L=nl, d=d, lda=lda, blocks=M.n_grad_blocks("densenet", dims), smem=smem, w_floats=w_floats,
                nn=[(c4(dims[l + 1]) // 4 + 3) // 4 for l in range(nl - 1)],
                nt=[2 * (((seg[l + 1] + 3) // 4 + 3) // 4) for l in range(nl - 1)],
                ragged=any(w % 8 for w in dims[1:-1]))


def shape_dims(shape, elliptic):
    d, arch = DIFF_SHAPES[shape] if isinstance(shape, str) else shape
    return [d if elliptic else d + 1] + list(arch) + [1]


def check_plan(shape):
    """The plan each shape claims (DIFF_PLAN, both time modes) and the regime it is there for; it fits."""
    d = DIFF_SHAPES[shape][0]
    for elliptic, want in zip((False, True), DIFF_PLAN[shape]):
        p = diff_plan(shape_dims(shape, elliptic), d, L.TIME_NONE if elliptic else L.TIME_LAST)
        assert (p["lda"], p["blocks"], p["smem"]) == want, (shape, elliptic, p)
        assert p["smem"] <= MAX_SMEM and DIFF_REGIME[shape](p), (shape, elliptic, p)


def workspace_bytes(p, grid):
    """pspde_diffusion_workspace_bytes restated (api_diffusion.cu): stats, packed weights, per-CTA gradient partials
    (blocks rounded up to 32, 64 floats each), each 256-aligned, + 256."""
    a = lambda x: (x + 255) // 256 * 256
    return a(grid * 32) + a(4 * p["w_floats"]) + a(grid * 4 * 64 * 32 * ((p["blocks"] + 31) // 32)) + 256


def first_refused_d(arch, time_mode):
    """The smallest d whose plan with hidden widths `arch` no longer fits 227 KB of shared memory."""
    d = 1
    while diff_plan([d + (time_mode == L.TIME_LAST)] + list(arch) + [1], d, time_mode)["smem"] <= MAX_SMEM:
        d += 1
    return d


# ------------------------------------------------------------------------------------------------ problem data
ELLIPTIC = ("expsphere", "expball_sin", "box2", "helmholtz", "drift")


def _drift(rng, d):
    """Mixed-sign a_diag and non-uniform b_diag (float32, as the pack holds them)."""
    a = (rng.uniform(0.5, 2.0, d) * np.where(np.arange(d) % 2, -1.0, 1.0)).astype(np.float32)
    b = rng.uniform(0.5, 2.0, d).astype(np.float32)
    return a, b


def _pack(d, a=None, b=None):
    pack = H.heat_pack(d)
    if a is not None:
        pack[:d], pack[d:2 * d] = a, b
    return pack


class DiffCase:
    """Inputs of one case: K paths from k_offset 0 of a shape (a DIFF_SHAPES id or (d, widths)) and a problem, the value
    network (theta scaled by the widest layer), start points, the kernels' Philox increments and the random-sign
    cotangents; `oracle()` is the fp64 rollout and gradient on them, chunked over paths and cached.
      parabolic (t_0 in [0.9, 1), T = 1, so that every tile mixes moving and stopped paths):
        heat       b = 0, sigma = sqrt(2) I
        ou         PSPDE_PROBLEM_OU with mixed-sign a_diag and non-uniform b_diag
        allencahn  h = y - y^3 (the backward's extra V(X_n) pass)
      elliptic:
        expsphere    unit ball, H_EXP_LINEAR
        expball_sin  unit ball, H_EXP_NONLINEAR_SIN
        box2         two-sided box [-1, 1]^d, H_EXP_NONLINEAR (alpha = 1/2), mixed-sign drift, non-uniform sigma: the
                     proposal X + (a X dt + v) decides the exit
        helmholtz    two-sided box [-1, 1]^2, H_HELMHOLTZ (device sinf)
        drift        unit ball, H_EXP_NONLINEAR_SIN, mixed-sign drift, non-uniform sigma"""

    def __init__(self, abi, shape, problem, K, N, dt, seed=7):
        self.shape, self.problem, self.K, self.N, self.dt, self.seed = shape, problem, K, N, np.float32(dt), seed
        self.elliptic = problem in ELLIPTIC
        self.d = d = DIFF_SHAPES[shape][0] if isinstance(shape, str) else shape[0]
        self.dims = shape_dims(shape, self.elliptic)
        rng = np.random.default_rng(seed)
        self.theta = M._theta(self.dims, seed)
        a = b = None
        if problem in ("ou", "box2", "drift"):
            a, b = _drift(rng, d)
        self.pack = _pack(d, a, b)
        pid = L.PROBLEM_OU if a is not None else L.PROBLEM_ALLEN_CAHN if problem == "allencahn" else L.PROBLEM_HEAT
        self.t0, self.pde, self.ell = None, None, None
        if self.elliptic:
            box = problem in ("box2", "helmholtz")
            if problem == "helmholtz":
                self.ell, self.mp = H.elliptic_spec("helmholtz"), man.EllipticProblem("helmholtz", d)
            elif problem == "box2":
                self.ell = L.make_elliptic(L.DOMAIN_BOX, x_l=-1.0, x_r=1.0, one_boundary=False, h_id=L.H_EXP_NONLINEAR,
                                           h_param=(0.5, 0, 0))
                self.mp = man.EllipticProblem("expball", d, alpha=0.5, a=a, b=b)
                self.mp.boundary, self.mp.one_boundary, self.mp.X_l, self.mp.X_r = "square", False, -1.0, 1.0
            else:
                kind = "expsphere" if problem == "expsphere" else "expball_sin"
                self.ell, self.mp = H.elliptic_spec(kind), man.EllipticProblem(kind, d, a=a, b=b)
            self.X0 = rng.uniform(-1, 1, (K, d)).astype(np.float32) if box else M._ball(rng, K, d)
        else:
            self.mp = man.Problem("heat", d) if a is None else \
                man.Problem("llgc", d, A=np.diag(a.astype(np.float64)), B=np.diag(b.astype(np.float64)))
            self.pde = man.ALLEN_CAHN if problem == "allencahn" else None
            self.X0 = M._ball(rng, K, d)
            self.t0 = rng.uniform(0.9, 1.0, K).astype(np.float32)
        self.pid = pid
        self.rand = [(rng.choice([-1.0, 1.0], K) * (0.5 + rng.uniform(0, 1, K)) / K).astype(np.float32) for _ in range(3)]
        for c in self.rand:
            c[::7] = 0.0
        self.xs = abi.philox_dump(self.cfg()) if N else np.zeros((0, K, d), np.float32)     # (N, K, d)

    def cfg(self, N=None):
        return L.make_cfg(self.K, self.d, self.N if N is None else N, self.dt, self.pid, L.NET_DENSENET, self.dims,
                          L.TIME_NONE if self.elliptic else L.TIME_LAST, adaptive=False, noise_mode=L.NOISE_PHILOX,
                          seed=self.seed, offset=2, n_sets=1 if self.elliptic else 0)

    def plan(self):
        return diff_plan(self.dims, self.d, L.TIME_NONE if self.elliptic else L.TIME_LAST)

    def blocks(self):
        return M.grad_blocks("densenet", self.dims)

    def fwd(self, abi, X0=None, N=None, t0=None):
        X0 = self.X0 if X0 is None else X0
        t0 = self.t0 if t0 is None else t0
        return abi.diff_fwd(self.cfg(N), 1.0, self.theta, self.pack, X0, t0, None, ell=self.ell)

    def bwd(self, abi, cot, X0=None, N=None, t0=None):
        X0 = self.X0 if X0 is None else X0
        t0 = self.t0 if t0 is None else t0
        return abi.diff_bwd(self.cfg(N), 1.0, self.theta, self.pack, X0, t0, None, *cot, ell=self.ell)

    def cotangents(self, form, f, kept=None):
        """float32 (c0, cE, cD): 'loss' from the forward outputs f (w = 2 r / K, zero where r is not finite, as
        GeneralSolver / EllipticSolver form it), 'rand' the case's; zero off `kept`."""
        if form == "loss":
            r = f["VE"].astype(np.float64) - f["Y"]
            w = np.where(np.isfinite(r), 2 * r / self.K, 0.0).astype(np.float32)
            cot = [-w, w.copy(), -w]
        else:
            cot = [c.copy() for c in self.rand]
        if kept is not None:
            for c in cot:
                c[~kept] = 0.0
        return cot

    def oracle(self, cot, kept=None, chunk=2048):
        """fp64 per-path outputs (X, t, Y, VE, V0, V_L2) of the paths in `kept` (default all) and the gradient of
        sum_k c0 V(X_0) + cE V(X_end) + cD (every active directional derivative - h dt) over them."""
        idx = np.arange(self.K) if kept is None else np.flatnonzero(kept)
        cot = [np.asarray(c, np.float64)[idx] for c in cot]
        key = ("diffcase", self.shape, self.problem, self.K, self.N, float(self.dt), self.seed, hash(idx.tobytes()),
               hash(b"".join(c.tobytes() for c in cot)))
        if key in M._ORACLE:
            return M._ORACLE[key]
        net = man.Net("densenet", self.dims, self.theta.astype(np.float64))
        X64, x64, dt = self.X0.astype(np.float64)[idx], self.xs.astype(np.float64)[:, idx], float(self.dt)

        def part(lo, hi, _):
            c = tuple(v[lo:hi] for v in cot)
            if self.elliptic:
                m = man.elliptic(self.mp, net, X64[lo:lo + 1], X64[lo:hi], x64[:, lo:hi], dt, self.N, (1.0, 0.0), cot=c)
                m["VE"] = m["r"] + m["Y"]
                m["V0"] = net.forward(X64[lo:hi])[0][:, 0]
                return m
            t64 = self.t0.astype(np.float64)[idx]
            m = man.diffusion(self.mp, net, X64[lo:hi], t64[lo:hi], x64[:, lo:hi], dt, self.N, 1, alpha=(1.0, 0.0, 0.0),
                              T=1.0, pde=self.pde, cot=c)
            m["VE"] = net.forward(np.concatenate([m["X"], m["t"][:, None]], 1))[0][:, 0]
            m["V0"] = net.forward(np.concatenate([X64[lo:hi], t64[lo:hi, None]], 1))[0][:, 0]
            return m
        M._ORACLE[key] = M._chunked(part, idx.size, chunk)
        return M._ORACLE[key]


PER_PATH = ("V0", "VE", "Y", "X", "t", "VL2")


def check_forward(c, f, m, kept=None):
    """Per-path outputs of a forward against the oracle (on the kept paths) and its stats: stats[1] the active steps,
    stats[0] and stats[2] the sums of r^2 and r over the finite r = VE - Y, stats[3] the others."""
    kept = np.ones(c.K, bool) if kept is None else kept
    assert 0 < m["K_count"] < kept.sum() * c.N, "every case mixes moving and stopped paths"
    assert relerr(f["X"][kept], m["X"]) < M.TOL_END, ("X", relerr(f["X"][kept], m["X"]))
    keys = ("Y", "VE", "V0") + (("V_L2",) if c.elliptic else ())
    if not c.elliptic:
        assert relerr(f["t"][kept], m["t"]) < M.TOL_END
    for k in keys:
        o = f["VL2" if k == "V_L2" else k][kept]
        assert relerr(o, m[k]) < M.TOL_PATH, (k, relerr(o, m[k]))
    r = f["VE"].astype(np.float64) - f["Y"]
    ok = np.isfinite(r)
    assert f["stats"][3] == (~ok).sum()
    np.testing.assert_allclose(f["stats"][[0, 2]], [(r[ok] * r[ok]).sum(), r[ok].sum()], rtol=1e-9)


def geometry_case(abi, shape, problem, K, N, dt, form):
    """One forward and backward of a shape / problem against the oracle: per-path outputs, stats (the active steps
    equal the oracle's), the gradient as a whole and per layer block."""
    c = DiffCase(abi, shape, problem, K, N, dt)
    if isinstance(shape, str):
        check_plan(shape)
    f = c.fwd(abi)
    cot = c.cotangents(form, f)
    m = c.oracle(cot)
    assert int(f["stats"][1]) == m["K_count"]
    check_forward(c, f, m)
    M.check_grad(c.bwd(abi, cot), m["grad"], c.blocks(), "%s %s %s" % (shape, problem, form))


def boundary_case(abi, shape, problem, K, dt):
    """The N = 0 call of the terminal condition (parabolic, t_0 = T) and of the Dirichlet term (elliptic) at the same K:
    V_0 per path, and the gradient of sum_k c0 V(X_0) from a c0-only backward."""
    c = DiffCase(abi, shape, problem, K, 0, dt)
    tT = None if c.elliptic else np.ones(K, np.float32)
    f = c.fwd(abi, t0=tT)
    net = man.Net("densenet", c.dims, c.theta.astype(np.float64))
    a0 = c.X0.astype(np.float64) if c.elliptic else np.concatenate([c.X0.astype(np.float64), np.ones((K, 1))], 1)
    v0, tape = net.forward(a0)
    assert relerr(f["V0"], v0[:, 0]) < M.TOL_PATH and np.array_equal(f["V0"], f["VE"])
    assert f["stats"][1] == 0
    c0 = c.rand[0]
    grad = c.bwd(abi, (c0, None, None), t0=tT)
    M.check_grad(grad, net.vjp(tape, c0.astype(np.float64)[:, None]), c.blocks(), "%s %s N = 0" % (shape, problem))


def dropped_case(abi, shape, problem, K, N, dt, form):
    """Paths the solvers drop: six X_0 rows at 1e20 and one NaN row over different tiles and CTAs.  Forward: r is not
    finite exactly there, stats[3] counts them, stats[0] / stats[2] sum the finite r, every other path's outputs are
    bit-equal to a run where those rows hold benign starts.  Backward with zero cotangents on the dropped rows: finite,
    bit-equal to the benign-start run, and the oracle's gradient over the kept paths.  (V_L2 of a dropped elliptic path
    need not be finite.)"""
    c = DiffCase(abi, shape, problem, K, N, dt)
    bad = np.linspace(K // 3, K - 3, 7).astype(int)
    assert len({i // P for i in bad}) == 7
    X0 = c.X0.copy()
    X0[bad[:-1]] = 1e20
    X0[bad[-1]] = np.nan
    kept = ~np.isin(np.arange(K), bad)
    f, ref = c.fwd(abi, X0), c.fwd(abi)
    r = f["VE"].astype(np.float64) - f["Y"]
    assert np.array_equal(np.isfinite(r), kept), "exactly the bad starts give a non-finite r"
    assert f["stats"][3] == 7
    for k in PER_PATH:
        assert np.array_equal(f[k][kept], ref[k][kept]), k
    cot = c.cotangents(form, f, kept)
    m = c.oracle(cot, kept)
    check_forward(c, f, m, kept)
    grad = c.bwd(abi, cot, X0)
    assert np.isfinite(grad).all(), "a dropped path's zero cotangents turned into NaN"
    assert np.array_equal(grad, c.bwd(abi, cot))
    M.check_grad(grad, m["grad"], c.blocks(), "%s %s %s dropped" % (shape, problem, form))


def refusal_case(abi, arch, elliptic):
    """The first d whose tile no longer fits 227 KB of shared memory (diff_plan) is refused with -6 by the forward and the
    backward before any launch, with the byte count of the restatement; d - 1 is accepted."""
    tm = L.TIME_NONE if elliptic else L.TIME_LAST
    d = first_refused_d(arch, tm)
    ell = H.elliptic_spec("expball_sin") if elliptic else None
    out = {}
    for dd in (d - 1, d):
        dims = [dd + (0 if elliptic else 1)] + list(arch) + [1]
        cfg = L.make_cfg(100, dd, 2, np.float32(0.01), L.PROBLEM_HEAT, L.NET_DENSENET, dims, tm, adaptive=False,
                         n_sets=1 if elliptic else 0)
        ws = abi.lib.pspde_elliptic_workspace_bytes(ctypes.byref(cfg), ctypes.byref(ell)) if elliptic else \
            abi.lib.pspde_diffusion_workspace_bytes(ctypes.byref(cfg), ctypes.c_float(1.0))
        out[dd] = (ws, abi.lib.pspde_last_error(), cfg, dims)
    assert out[d - 1][0] > 0 and out[d][0] == 0
    ws, msg, cfg, dims = out[d]
    assert int(re.search(rb"need (\d+) B of shared memory", msg).group(1)) == diff_plan(dims, d, tm)["smem"] > MAX_SMEM
    assert diff_plan([d - 1 + (not elliptic)] + list(arch) + [1], d - 1, tm)["smem"] <= MAX_SMEM
    theta = abi.dev(np.zeros(abi.lib.pspde_theta_size(ctypes.byref(cfg)), np.float32))
    keep = [abi.dev(a) for a in (H.heat_pack(d), np.zeros((100, d)), np.full(100, 0.5), np.zeros(100))]
    outs = [abi.zeros(100) for _ in range(5)]
    buf = abi.zeros(1 << 20, np.float64)
    p = abi.p
    n0 = abi.lib.pspde_launch_count()
    if elliptic:
        rf = abi.lib.pspde_elliptic_fwd(ctypes.byref(cfg), ctypes.byref(ell), p(theta), p(keep[0]), p(keep[1]), None,
                                        *[p(o) for o in outs], None, p(buf), abi.nbytes(buf), None)
        rb = abi.lib.pspde_elliptic_bwd(ctypes.byref(cfg), ctypes.byref(ell), p(theta), p(keep[0]), p(keep[1]), None,
                                        p(keep[3]), None, None, p(theta), p(buf), abi.nbytes(buf), None)
    else:
        rf = abi.lib.pspde_diffusion_fwd(ctypes.byref(cfg), ctypes.c_float(1.0), p(theta), p(keep[0]), p(keep[1]),
                                         p(keep[2]), None, *[p(o) for o in outs], None, p(buf), abi.nbytes(buf), None)
        rb = abi.lib.pspde_diffusion_bwd(ctypes.byref(cfg), ctypes.c_float(1.0), p(theta), p(keep[0]), p(keep[1]),
                                         p(keep[2]), None, p(keep[3]), None, None, p(theta), p(buf), abi.nbytes(buf), None)
    assert (rf, rb) == (-6, -6) and abi.lib.pspde_launch_count() == n0
    return d
