"""Cases shared by test_emu_ensemble.py (host emulator) and test_gpu_ensemble.py (sm_100a build): the ensemble entry points
(pspde_ensemble_*: M independent models of one configuration, one launch per phase) against the single-model calls and
the fp64 oracle.

Member m is fma_cases.FmaCase number m % n_distinct: its own Philox key, parameters, cotangents, y0 and (x0_per_path) start
points.  The members sit in the ensemble buffers with a gap of NaN between them (theta) or a sentinel (grad_theta): a
kernel that reads past its member's parameters turns the outputs NaN, one that writes past its member's gradient is seen
in the gap."""
import ctypes

import numpy as np

import fma_cases as F
import multitile as M
from pspde import _lib as L

GAP = 3                          # floats between two members' parameter sets
SENTINEL = 7.25


def ens_grid_x(n_models, n_tiles, sms, max_grid=None):
    """CTAs per member: the grid policy of make_ens_plan (csrc/api_core.cu) restated."""
    gx = min(n_tiles, sms)
    if n_models * n_tiles > sms:
        gx = max(1, sms // n_models)
    if max_grid:
        gx = min(gx, int(max_grid))
    return gx


def single_grid(n_tiles, sms, max_grid=None):
    g = min(n_tiles, sms)
    return min(g, int(max_grid)) if max_grid else g


class EnsembleCase:
    def __init__(self, abi, shape, K, N, n_models, x0_per_path=False, n_distinct=5, seed0=5):
        nd = min(n_distinct, n_models)
        self.abi, self.shape, self.K, self.N, self.M = abi, shape, K, N, n_models
        self.cases = [F.FmaCase(abi, shape, K, N, x0_per_path=x0_per_path, y0=0.2 * i - 0.3, seed=seed0 + 3 * i)
                      for i in range(nd)]
        c0 = self.cases[0]
        for c in self.cases[1:]:               # one problem for all (dense A / B are drawn from the case's seed)
            c.mp, c.pid, c.flags, c.pack = c0.mp, c0.pid, c0.flags, c0.pack
        self.member = [self.cases[m % nd] for m in range(n_models)]
        self.d, self.n_theta = c0.d, c0.theta.size
        self.stride = self.n_theta + GAP
        self.theta = np.full((n_models, self.stride), np.nan, np.float32)
        for m, c in enumerate(self.member):
            self.theta[m, :self.n_theta] = c.theta
        self.seeds = np.array([c.seed for c in self.member], np.uint64)
        self.y0 = np.array([c.y0 for c in self.member], np.float32)
        self.wY = np.stack([c.wY for c in self.member])
        self.x0_per_path = x0_per_path
        self.x0 = np.stack([c.x0 for c in self.member]) if x0_per_path else c0.x0
        self.x0_stride = K * self.d if x0_per_path else 0
        self.table = (0.3 * np.random.default_rng(seed0).standard_normal((2 * N, self.d))).astype(np.float32)
        self._single = {}

    def cfg(self):
        return self.cases[0].cfg()

    def ens(self, keep):
        seeds = self.abi.dev(self.seeds.view(np.int64), np.int64)
        keep.append(seeds)
        return L.pspde_ensemble(n_models=self.M, seeds=self.abi.addr(seeds), theta_stride=self.stride,
                                x0_stride=self.x0_stride)

    def diag(self, table, uL2):
        return L.pspde_udiag(mode=1, nx1=0, d1=0, xb=0.0, dx=0.0, table=self.abi.addr(table), uL2=self.abi.addr(uL2),
                             quirk_path=-1)

    def workspace_bytes(self):
        keep = []
        n = self.abi.lib.pspde_ensemble_workspace_bytes(ctypes.byref(self.cfg()), ctypes.byref(self.ens(keep)))
        assert n > 0, self.abi.lib.pspde_last_error()
        return n

    # -- the ensemble entry points
    def forward(self, ws=None, ws_bytes=None):
        """pspde_ensemble_fwd: (outputs [M][...], return code, launches)."""
        a, M_, K, d = self.abi, self.M, self.K, self.d
        keep = []
        ens = self.ens(keep)
        o = a._out(dict(X=(M_, K, d), Y=(M_, K), gX=(M_, K), Zsum=(M_, K), stats=(M_, 4), uL2=(M_, K)))
        ins = [a.dev(x) for x in (self.theta, self.cases[0].pack, self.x0, self.y0, self.table)]
        if ws is None:
            ws = a.ws(self.workspace_bytes())
            ws_bytes = a.nbytes(ws)
        diag = self.diag(ins[4], o["uL2"])
        n0 = a.lib.pspde_launch_count()
        rc = a.lib.pspde_ensemble_fwd(ctypes.byref(self.cfg()), ctypes.byref(ens), *[a.p(x) for x in ins[:4]], a.p(o["X"]),
                                      a.p(o["Y"]), a.p(o["gX"]), a.p(o["Zsum"]), a.p(o["stats"]), ctypes.byref(diag),
                                      a.p(ws), ws_bytes, None)
        return a._host_all(o), rc, a.lib.pspde_launch_count() - n0

    def backward(self, ws=None, ws_bytes=None):
        """pspde_ensemble_bwd_detached: (grad [M][stride] with SENTINEL wherever it did not write, return code, launches)."""
        a = self.abi
        keep = []
        ens = self.ens(keep)
        grad = a.dev(np.full((self.M, self.stride), SENTINEL, np.float32))
        ins = [a.dev(x) for x in (self.theta, self.cases[0].pack, self.x0, self.wY)]
        if ws is None:
            ws = a.ws(self.workspace_bytes())
            ws_bytes = a.nbytes(ws)
        n0 = a.lib.pspde_launch_count()
        rc = a.lib.pspde_ensemble_bwd_detached(ctypes.byref(self.cfg()), ctypes.byref(ens), *[a.p(x) for x in ins], None,
                                               a.p(grad), a.p(ws), ws_bytes, None)
        return a.host(grad), rc, a.lib.pspde_launch_count() - n0

    def lv_cotangents(self, stats, moment):
        a = self.abi
        ins = [a.dev(x) for x in (stats["Y"], stats["gX"])] + [a.dev(stats["stats"], np.float64)]
        wY, out = a.zeros((self.M, self.K)), a.zeros((self.M, 3), np.float64)
        n0 = a.lib.pspde_launch_count()
        L.check(a.lib, a.lib.pspde_ensemble_lv_cotangents(self.M, self.K, float(self.K), moment, *[a.p(x) for x in ins],
                                                          a.p(wY), a.p(out), None))
        assert a.lib.pspde_launch_count() - n0 == 1
        return a.host(wY), a.host(out)

    # -- the single-model calls of member m's inputs
    def single(self, c):
        """pspde_rollout_fwd_diag, pspde_lv_cotangents (log-variance and moment) and pspde_rollout_bwd_detached of case c."""
        key = id(c)
        if key not in self._single:
            a, K, d = self.abi, self.K, self.d
            o = a._out(dict(X=(K, d), Y=K, gX=K, Zsum=K, stats=4, uL2=K))
            ins = [a.dev(x) for x in (c.theta, c.pack, c.x0, [c.y0], self.table)]
            ws = a.ws(a.lib.pspde_workspace_bytes(ctypes.byref(c.cfg())))
            diag = self.diag(ins[4], o["uL2"])
            n0 = a.lib.pspde_launch_count()
            L.check(a.lib, a.lib.pspde_rollout_fwd_diag(ctypes.byref(c.cfg()), *[a.p(x) for x in ins[:4]], None, a.p(o["X"]),
                                                        a.p(o["Y"]), a.p(o["gX"]), a.p(o["Zsum"]), a.p(o["stats"]),
                                                        ctypes.byref(diag), a.p(ws), a.nbytes(ws), None))
            assert a.lib.pspde_launch_count() - n0 == F.FWD_LAUNCHES
            r = a._host_all(o)
            for moment in (0, 1):
                w, out = a.zeros(K), a.zeros(3, np.float64)
                L.check(a.lib, a.lib.pspde_lv_cotangents(K, float(K), moment, a.p(o["Y"]), a.p(o["gX"]), a.p(o["stats"]),
                                                         a.p(w), a.p(out), None))
                r["lv%d" % moment] = (a.host(w), a.host(out))
            r["grad"] = c.backward(a)
            self._single[key] = r
        return self._single[key]


def check_ensemble(e, bitwise):
    """Every member of the ensemble against the single-model calls on its inputs (per-path outputs bit-equal; statistics,
    loss, cotangents and gradient bit-equal if `bitwise`, else within the multitile tolerances) and against the fp64 oracle."""
    o, rc, n = e.forward()
    L.check(e.abi.lib, rc)
    assert n == F.FWD_LAUNCHES, n
    g, rc, n = e.backward()
    L.check(e.abi.lib, rc)
    assert n == F.BWD_LAUNCHES, n
    assert np.all(g[:, e.n_theta:] == SENTINEL), "a member's gradient spilled into the gap"
    lv = {moment: e.lv_cotangents(o, moment) for moment in (0, 1)}
    for m, c in enumerate(e.member):
        s = e.single(c)
        om = {k: o[k][m] for k in o}
        for k in ("X", "Y", "gX", "Zsum", "uL2"):
            assert np.array_equal(om[k], s[k]), ("member", m, k)
        gm = g[m, :e.n_theta]
        if bitwise:
            assert np.array_equal(om["stats"], s["stats"]), ("member", m, om["stats"], s["stats"])
            assert np.array_equal(gm, s["grad"]), ("member", m, "gradient")
            for moment in (0, 1):
                assert np.array_equal(lv[moment][0][m], s["lv%d" % moment][0]), ("member", m, "cotangents", moment)
                assert np.array_equal(lv[moment][1][m], s["lv%d" % moment][1]), ("member", m, "loss", moment)
        else:
            np.testing.assert_allclose(om["stats"], s["stats"], rtol=1e-12, atol=1e-12 * np.abs(s["stats"]).max())
            M.check_grad(gm, s["grad"], c.blocks(), "member %d vs single call" % m)
            for moment in (0, 1):
                np.testing.assert_allclose(lv[moment][0][m], s["lv%d" % moment][0], rtol=1e-6, atol=1e-12)
                np.testing.assert_allclose(lv[moment][1][m], s["lv%d" % moment][1], rtol=1e-10)
        ref = c.oracle()
        F.check_forward(om, ref)
        M.check_grad(gm, ref["grad"], c.blocks(), "member %d vs oracle" % m)


def check_adam(abi, n_models=6, n=1000, seed=3):
    """pspde_ensemble_adam against one pspde_adam_flat per member (bit for bit), member 2 marked finished (step 0)."""
    rng = np.random.default_rng(seed)
    stride = n + 5
    bufs = {k: rng.standard_normal((n_models, stride)).astype(np.float32) for k in ("theta", "grad", "m")}
    bufs["v"] = rng.uniform(0, 1, (n_models, stride)).astype(np.float32)
    hyper = [(1e-3 * (1 + m), 0.9 - 0.01 * m, 0.999 - 0.001 * m, 1e-8 * (1 + m), 0 if m == 2 else 1 + 2 * m)
             for m in range(n_models)]
    table = (L.pspde_adam_member * n_models)()
    for m, h in enumerate(hyper):
        L.check(abi.lib, abi.lib.pspde_adam_member_make(*h, ctypes.byref(table[m])))
    tab = abi.dev(np.frombuffer(bytes(table), np.uint8).copy(), np.uint8)
    ens = {k: abi.dev(v) for k, v in bufs.items()}
    n0 = abi.lib.pspde_launch_count()
    L.check(abi.lib, abi.lib.pspde_ensemble_adam(n_models, n, stride, abi.p(ens["theta"]), abi.p(ens["grad"]), abi.p(ens["m"]),
                                                 abi.p(ens["v"]), abi.p(tab), None))
    assert abi.lib.pspde_launch_count() - n0 == 1
    ens = {k: abi.host(v) for k, v in ens.items()}
    for m, (lr, b1, b2, eps, step) in enumerate(hyper):
        one = {k: abi.dev(np.ascontiguousarray(v[m, :n])) for k, v in bufs.items()}
        if step:
            L.check(abi.lib, abi.lib.pspde_adam_flat(n, abi.p(one["theta"]), abi.p(one["grad"]), abi.p(one["m"]),
                                                     abi.p(one["v"]), lr, b1, b2, eps, step, None))
        for k in ("theta", "m", "v"):
            assert np.array_equal(ens[k][m, :n], abi.host(one[k])), (m, k)
            assert np.array_equal(ens[k][m, n:], bufs[k][m, n:]), (m, k, "gap")
        if not step:
            assert all(np.array_equal(ens[k][m], bufs[k][m]) for k in ("theta", "m", "v"))


def check_workspace(e):
    """A workspace of exactly pspde_ensemble_workspace_bytes with a sentinel behind it: both calls leave the sentinel
    intact; one byte less is refused with -7 before any launch."""
    a = e.abi
    nbytes = e.workspace_bytes()
    buf = a.dev(np.full(nbytes + 256, 0xAB, np.uint8), np.uint8)
    for call in (e.forward, e.backward):
        r = call(buf, nbytes)
        L.check(a.lib, r[1])
        assert np.all(a.host(buf)[nbytes:] == 0xAB), call.__name__
    _, rc, n = e.backward(buf, nbytes - 1)
    assert (rc, n) == (-7, 0), (rc, n)
