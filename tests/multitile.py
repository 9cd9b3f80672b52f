"""Cases shared by test_emu_multitile.py (host emulator) and test_gpu_multitile.py (sm_100a build): the attached adjoint
kernel and the diffusion / elliptic kernels with several tiles per CTA, against the fp64 oracle (oracle/manual.py).
TcCase and check_tc_forward serve test_gpu_tc_multitile.py (tensor-core kernels, device only).

A persistent CTA loops `for (tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)`: per-tile state must be reset and
the per-CTA gradient partials must collect every tile exactly once.  Each case is run by the test files at a K that
gives at least two tiles per CTA at the natural grid, and again with PSPDE_MAX_GRID for many tiles per CTA.  The
last tile is always ragged.  The increments are the kernels' own Philox draws, read back with pspde_philox_dump.

`Abi` drives the C ABI with numpy buffers (emulator) or CUDA tensors (device), so both files run the same code."""
import ctypes

import numpy as np

import emu_harness as H
from conftest import relerr
from oracle import manual as man
from pspde import _lib as L

TOL_PATH, TOL_END, TOL_GRAD, TOL_BLOCK = 1e-5, 1e-6, 2e-5, 5e-5
P_HJB, P_DIFF = 64, 32          # paths per tile of the rollout / attached kernels and of the diffusion kernel


class Abi:
    """The library's entry points on host (device=None: numpy, emulator build) or device (torch CUDA tensors) buffers;
    inputs and outputs are numpy arrays either way."""

    def __init__(self, lib, device=None):
        self.lib, self.device = lib, device
        if device is not None:
            import torch
            self.pt = torch

    def dev(self, a, dtype=np.float32):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype)
        return a if self.device is None else self.pt.from_numpy(a).to(self.device)

    def zeros(self, shape, dtype=np.float32):
        a = np.zeros(shape, dtype)
        return a if self.device is None else self.pt.from_numpy(a).to(self.device)

    def host(self, a):
        return a if self.device is None else a.cpu().numpy()

    def p(self, a):
        """Raw pointer; a device tensor passed here must stay referenced until the call returns (the caching allocator
        reuses a freed block for the next upload before the kernel runs)."""
        if a is None:
            return None
        return a.ctypes.data_as(ctypes.c_void_p) if self.device is None else ctypes.c_void_p(a.data_ptr())

    def ws(self, nbytes):
        assert nbytes > 0, self.lib.pspde_last_error()
        return self.zeros(nbytes // 8 + 1, np.float64)

    def nbytes(self, a):
        return a.nbytes if self.device is None else a.numel() * a.element_size()

    def _out(self, names):
        return {k: self.zeros(s, np.float64 if k == "stats" else np.float32) for k, s in names.items()}

    def _host_all(self, o):
        return {k: self.host(v) for k, v in o.items()}

    # -- HJB rollout
    def philox_dump(self, cfg):
        """(N, K, d) float32: the increments the kernels draw for cfg."""
        out = self.zeros((cfg.N, cfg.K_local, cfg.d))
        L.check(self.lib, self.lib.pspde_philox_dump(ctypes.byref(cfg), self.p(out), None))
        return self.host(out)

    def fwd(self, cfg, theta, pack, x0):
        K, d = cfg.K_local, cfg.d
        ws = self.ws(self.lib.pspde_workspace_bytes(ctypes.byref(cfg)))
        o = self._out(dict(X=(K, d), Y=K, gX=K, Zsum=K, stats=4))
        ins = [self.dev(a) for a in (theta, pack, x0)]
        rc = self.lib.pspde_rollout_fwd(ctypes.byref(cfg), *[self.p(a) for a in ins], None, None, self.p(o["X"]),
                                        self.p(o["Y"]), self.p(o["gX"]), self.p(o["Zsum"]), self.p(o["stats"]), self.p(ws),
                                        self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self._host_all(o)

    def addr(self, a):
        return a.ctypes.data if self.device is None else a.data_ptr()

    def attached(self, cfg, theta, pack, x0, w, wY=None, wZ=None, wG=None, y0=None, xi=None, table=None):
        """pspde_rollout_attached: relative entropy in one launch (w, no per-path cotangents) or per-path cotangents;
        y0 (a float) is Y's start value, xi the injected increments in the reference layout (K, d, N + 1).  With a
        `table` it calls pspde_rollout_attached_diag with the u_L2 diagnostic (mode 1, linear table).  Returns
        (outputs, launches it took)."""
        K, d = cfg.K_local, cfg.d
        ws = self.ws(self.lib.pspde_workspace_bytes(ctypes.byref(cfg)))
        o = self._out(dict(X=(K, d), Y=K, gX=K, Zsum=K, stats=4, grad=self.lib.pspde_theta_size(ctypes.byref(cfg)),
                           uL2=K))
        keep = [self.dev(a) for a in (theta, pack, x0, None if y0 is None else [y0], xi, wY, wZ, wG, table)]
        args = [ctypes.byref(cfg), *[self.p(a) for a in keep[:4]], self.xi_ptr(keep[4]), ctypes.c_float(w),
                *[self.p(a) for a in keep[5:8]], self.p(o["X"]), self.p(o["Y"]), self.p(o["gX"]), self.p(o["Zsum"]),
                self.p(o["stats"])]
        tail = [self.p(o["grad"]), self.p(ws), self.nbytes(ws), None]
        n0 = self.lib.pspde_launch_count()
        if table is None:
            rc = self.lib.pspde_rollout_attached(*args, *tail)
        else:
            diag = L.pspde_udiag(mode=1, nx1=0, d1=0, xb=0.0, dx=0.0, table=self.addr(keep[8]), uL2=self.addr(o["uL2"]),
                                 quirk_path=-1)
            rc = self.lib.pspde_rollout_attached_diag(*args, ctypes.byref(diag), *tail)
        L.check(self.lib, rc)
        return self._host_all(o), self.lib.pspde_launch_count() - n0

    # -- diffusion / elliptic
    def diff_fwd(self, cfg, T, theta, pack, X0, t0, xis, ell=None):
        K, d = cfg.K_local, cfg.d
        o = self._out(dict(V0=K, VE=K, Y=K, X=(K, d), t=K, VL2=K, stats=4))
        ins = [self.dev(a) for a in (theta, pack, X0, t0, xis)]
        if ell is None:
            ws = self.ws(self.lib.pspde_diffusion_workspace_bytes(ctypes.byref(cfg), ctypes.c_float(T)))
            rc = self.lib.pspde_diffusion_fwd(ctypes.byref(cfg), ctypes.c_float(T), *[self.p(a) for a in ins],
                                              self.p(o["V0"]), self.p(o["VE"]), self.p(o["Y"]), self.p(o["X"]),
                                              self.p(o["t"]), self.p(o["stats"]), self.p(ws), self.nbytes(ws), None)
        else:
            ws = self.ws(self.lib.pspde_elliptic_workspace_bytes(ctypes.byref(cfg), ctypes.byref(ell)))
            rc = self.lib.pspde_elliptic_fwd(ctypes.byref(cfg), ctypes.byref(ell), self.p(ins[0]), self.p(ins[1]),
                                             self.p(ins[2]), self.p(ins[4]), self.p(o["V0"]), self.p(o["VE"]),
                                             self.p(o["Y"]), self.p(o["X"]), self.p(o["VL2"]), self.p(o["stats"]),
                                             self.p(ws), self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self._host_all(o)

    def diff_bwd(self, cfg, T, theta, pack, X0, t0, xis, c0, cE, cD, ell=None):
        grad = self.zeros(self.lib.pspde_theta_size(ctypes.byref(cfg)))
        ins = [self.dev(a) for a in (theta, pack, X0, t0, xis, c0, cE, cD)]
        if ell is None:
            ws = self.ws(self.lib.pspde_diffusion_workspace_bytes(ctypes.byref(cfg), ctypes.c_float(T)))
            rc = self.lib.pspde_diffusion_bwd(ctypes.byref(cfg), ctypes.c_float(T), *[self.p(a) for a in ins],
                                              self.p(grad), self.p(ws), self.nbytes(ws), None)
        else:
            ws = self.ws(self.lib.pspde_elliptic_workspace_bytes(ctypes.byref(cfg), ctypes.byref(ell)))
            ins = ins[:3] + ins[4:]
            rc = self.lib.pspde_elliptic_bwd(ctypes.byref(cfg), ctypes.byref(ell), *[self.p(a) for a in ins],
                                             self.p(grad), self.p(ws), self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self.host(grad)

    def sample(self, cfg, radius, T):
        X0, t0 = self.zeros((cfg.K_local, cfg.d)), self.zeros(cfg.K_local)
        L.check(self.lib, self.lib.pspde_diffusion_sample(ctypes.byref(cfg), ctypes.c_float(radius), ctypes.c_float(T),
                                                          self.p(X0), self.p(t0), None))
        return self.host(X0), self.host(t0)

    # -- tensor-core rollout and gradient kernels (device only: tcgen05 has no host emulation)
    def fwd_ckpt(self, cfg, theta, pack, x0, xi=None, table=None, ckpt_bytes=0, y0=None):
        """pspde_rollout_fwd_ckpt: the forward, with the u_L2 diagnostic (mode 1, linear table) if `table` is given and
        keeping the operand rows of its first tiles in a buffer of ckpt_bytes if that is > 0; y0 (a float) is Y's
        start value.  Returns (outputs, device checkpoint buffer or None, launches it took)."""
        K, d = cfg.K_local, cfg.d
        ws = self.ws(self.lib.pspde_workspace_bytes(ctypes.byref(cfg)))
        o = self._out(dict(X=(K, d), Y=K, gX=K, Zsum=K, stats=4, uL2=K))
        ins = [self.dev(a) for a in (theta, pack, x0, xi, table, None if y0 is None else [y0])]
        diag = None
        if table is not None:
            diag = L.pspde_udiag(mode=1, nx1=0, d1=0, xb=0.0, dx=0.0, table=ins[4].data_ptr(), uL2=o["uL2"].data_ptr(),
                                 quirk_path=-1)
        ck = self.zeros(ckpt_bytes // 4) if ckpt_bytes else None
        n0 = self.lib.pspde_launch_count()
        rc = self.lib.pspde_rollout_fwd_ckpt(ctypes.byref(cfg), *[self.p(a) for a in ins[:3]], self.p(ins[5]), self.xi_ptr(ins[3]),
                                             self.p(o["X"]), self.p(o["Y"]), self.p(o["gX"]), self.p(o["Zsum"]),
                                             self.p(o["stats"]), None if diag is None else ctypes.byref(diag), self.p(ck),
                                             ckpt_bytes, self.p(ws), self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self._host_all(o), ck, self.lib.pspde_launch_count() - n0

    def xi_ptr(self, xi):
        """Injected increments in the reference layout (K, d, N + 1): slice n + 1 drives step n."""
        if xi is None:
            return None
        return ctypes.c_void_p(xi.ctypes.data + xi.strides[2] if self.device is None else xi.data_ptr() + 4 * xi.stride(2))

    def bwd_detached(self, cfg, theta, pack, x0, wY, wZ=None, xi=None):
        """pspde_rollout_bwd_detached: (gradient, launches it took)."""
        grad = self.zeros(self.lib.pspde_theta_size(ctypes.byref(cfg)))
        ws = self.ws(self.lib.pspde_workspace_bytes(ctypes.byref(cfg)))
        ins = [self.dev(a) for a in (theta, pack, x0, xi, wY, wZ)]
        n0 = self.lib.pspde_launch_count()
        rc = self.lib.pspde_rollout_bwd_detached(ctypes.byref(cfg), *[self.p(a) for a in ins[:3]], self.xi_ptr(ins[3]),
                                                 self.p(ins[4]), self.p(ins[5]), self.p(grad), self.p(ws), self.nbytes(ws),
                                                 None)
        L.check(self.lib, rc)
        return self.host(grad), self.lib.pspde_launch_count() - n0

    def importance_sampling(self, cfg, theta, pack, x0, t_index=None, dt_net=0.0):
        """pspde_importance_sampling (network time index t_index[n] on a grid of spacing dt_net, if given): (outputs
        X, Y, gX, Fint, launches it took)."""
        K, d = cfg.K_local, cfg.d
        ws = self.ws(self.lib.pspde_workspace_bytes_fwd(ctypes.byref(cfg)))
        o = self._out(dict(X=(K, d), Y=K, gX=K, Fint=K))
        ins = [self.dev(a) for a in (theta, pack, x0)] + [self.dev(t_index, np.int32)]
        n0 = self.lib.pspde_launch_count()
        rc = self.lib.pspde_importance_sampling(ctypes.byref(cfg), *[self.p(a) for a in ins[:3]], None, self.p(ins[3]),
                                                ctypes.c_float(dt_net), self.p(o["X"]), self.p(o["Y"]), self.p(o["gX"]),
                                                self.p(o["Fint"]), self.p(ws), self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self._host_all(o), self.lib.pspde_launch_count() - n0

    def grad_from_fwd_ckpt(self, cfg, theta, pack, x0, ck, wY, xi=None):
        """pspde_grad_from_fwd_ckpt on the rows a fwd_ckpt call kept: (gradient, launches it took)."""
        grad = self.zeros(self.lib.pspde_theta_size(ctypes.byref(cfg)))
        ws = self.ws(self.lib.pspde_workspace_bytes(ctypes.byref(cfg)))
        ins = [self.dev(a) for a in (theta, pack, x0, xi, wY)]
        n0 = self.lib.pspde_launch_count()
        rc = self.lib.pspde_grad_from_fwd_ckpt(ctypes.byref(cfg), *[self.p(a) for a in ins[:3]], self.xi_ptr(ins[3]),
                                               self.p(ck), self.nbytes(ck), self.p(ins[4]), self.p(grad), self.p(ws),
                                               self.nbytes(ws), None)
        L.check(self.lib, rc)
        return self.host(grad), self.lib.pspde_launch_count() - n0


# ------------------------------------------------------------------------------------------------------------ helpers
def grad_blocks(kind, dims, n_sets=1):
    """Slices of theta, one per (parameter set, layer): W_l and b_l of that layer."""
    out, off = [], 0
    for _ in range(n_sets):
        for i in range(len(dims) - 1):
            fan_in = sum(dims[:i + 1]) if kind == "densenet" else dims[i]
            n = (fan_in + 1) * dims[i + 1]
            out.append(slice(off, off + n))
            off += n
    return out


def n_grad_blocks(kind, dims):
    """The attached / backward kernels' count of 8x8 weight-gradient blocks (build_geom, csrc/pspde_geom.h): more than
    224 selects the 512-thread build."""
    c4 = lambda x: (x + 3) & ~3
    L_ = len(dims) - 1
    seg = [c4(dims[s] + (1 if (kind == "mlp_tanh" or s == 0) else 0)) for s in range(L_)]
    blk = 0
    for l in range(L_):
        Kp = sum(seg[:l + 1]) if kind == "densenet" else seg[l]
        nkg, nng = Kp // 4, c4(dims[l + 1]) // 4
        blk += ((nkg + 1) // 2) * ((nng + 1) // 2)
    return blk


def check_grad(grad, ref, blocks, what=""):
    assert np.isfinite(grad).all(), what
    e = relerr(grad, ref)
    assert e < TOL_GRAD, (what, e)
    for i, s in enumerate(blocks):        # a flush into the wrong slice shows up as one bad block
        assert relerr(grad[s], ref[s]) < TOL_BLOCK, (what, "block", i, relerr(grad[s], ref[s]))


def tiles_per_cta(K, P, grid):
    n_tiles = (K + P - 1) // P
    return n_tiles / min(n_tiles, grid)


# ------------------------------------------------------------------------------------------------ attached kernel
def hjb_problem(kind, d, off_diag=0.0, seed=0):
    """(man.Problem, (problem_id, flags, pack), x0) for 'lqgc', 'llgc' (optionally with dense A / B) and 'dwm' (C3's
    DoubleWell_multidim: d_1 = 15, kappa = 5, eta = 3)."""
    if kind == "dwm":
        pkw = dict(d_1=15, d_2=d - 15, eta=3.0, kappa=5.0)
        eta = np.array([3.0] * 15 + [1.0] * (d - 15))
        kap = np.array([5.0] * 15 + [1.0] * (d - 15))
        return man.Problem("dwm", d, eta_=eta, kappa_=kap), H.problem_pack("dwm", d, pkw), -np.ones(d, np.float32)
    A = B = None
    if off_diag:
        rng = np.random.default_rng(seed)
        A = (-np.eye(d) + off_diag * rng.standard_normal((d, d))).astype(np.float32)
        B = (np.eye(d) + off_diag * rng.standard_normal((d, d))).astype(np.float32)
    pk = H.problem_pack(kind, d, {}, A, B)
    mp = man.Problem(kind, d, A=None if A is None else A.astype(np.float64), B=None if B is None else B.astype(np.float64))
    return mp, pk, np.zeros(d, np.float32)


def attached_case(abi, kind, d, net, K, N, dt, loss, off_diag=0.0, outer=False, inert=False, seed=5, theta=None):
    """The attached kernel against the fp64 discrete adjoint: relative entropy in one launch (man.grad_mode_b) or a
    general loss through the forward launch -> per-path cotangents -> adjoint launch (man.grad_attached).  inert: every
    7th path gets exactly zero cotangents (the oracle gets the same zeros)."""
    mp, (pid, flags, pack), x0 = hjb_problem(kind, d, off_diag, seed)
    dims = [d if outer else d + 1, 30, 30, d]
    n_sets = N if outer else 1
    tm = L.TIME_NONE if outer else L.TIME_FIRST
    net_id = L.NET_DENSENET if net == "densenet" else L.NET_MLP_TANH
    cfg = L.make_cfg(K, d, N, np.float32(dt), pid, net_id, dims, tm, adaptive=True, problem_flags=flags,
                     noise_mode=L.NOISE_PHILOX, seed=seed, offset=3, n_sets=N if outer else 0)
    n_theta = abi.lib.pspde_theta_size(ctypes.byref(cfg))
    assert n_theta > 0, abi.lib.pspde_last_error()
    if theta is None:
        theta = (0.1 * np.random.default_rng(seed).standard_normal(n_theta)).astype(np.float32)
    nth = n_theta // n_sets
    th64 = theta.astype(np.float64)
    nets = [man.Net(net, dims, th64[s * nth:(s + 1) * nth]) for s in range(n_sets)]
    xi = np.zeros((K, d, N + 1))
    xi[:, :, 1:] = abi.philox_dump(cfg).transpose(1, 2, 0)
    mode = "none" if outer else "first"
    if loss == "relative_entropy":
        o, _ = abi.attached(cfg, theta, pack, x0, 1.0 / K)
        gm, ro = man.grad_mode_b(mp, nets[0], xi, dt, N, x0.astype(np.float64), mode)
    else:
        f = abi.fwd(cfg, theta, pack, x0)
        _, wY, wZ, wG = man.loss_cotangents_full(loss, f["Y"].astype(np.float64), f["gX"].astype(np.float64),
                                                 f["Zsum"].astype(np.float64), True)
        wY, wZ, wG = (np.asarray(w, np.float32) for w in (wY, wZ, wG))
        if inert:
            for w in (wY, wZ, wG):
                w[::7] = 0.0
        o, _ = abi.attached(cfg, theta, pack, x0, 0.0, wY, wZ, wG)
        gm, ro = man.grad_attached(mp, nets if outer else nets[0], xi, dt, N, x0.astype(np.float64),
                                   wY.astype(np.float64), wZ.astype(np.float64), wG.astype(np.float64), mode)
        for k in ("X", "Y", "Zsum", "gX"):           # the forward launch that produced the cotangents
            assert relerr(f[k], ro[k]) < TOL_PATH, ("forward launch", k, relerr(f[k], ro[k]))
    for k in ("X", "Y", "Zsum", "gX"):
        assert relerr(o[k], ro[k]) < TOL_PATH, ("attached launch", k, relerr(o[k], ro[k]))
    v = o["Zsum"].astype(np.float64) + o["gX"]
    assert o["stats"][3] == 0
    np.testing.assert_allclose(o["stats"][2], v.sum(), rtol=1e-10)
    check_grad(o["grad"], gm, grad_blocks(net, dims, n_sets), "%s d=%d %s" % (kind, d, loss))


# ------------------------------------------------------------------------------------------------ diffusion kernels
def _theta(dims, seed, scale=0.3):
    n = sum((sum(dims[:i + 1]) + 1) * dims[i + 1] for i in range(len(dims) - 1))
    return (scale * np.random.default_rng(seed).standard_normal(n) / np.sqrt(max(dims))).astype(np.float32)


def _ball(rng, K, d, r_lo=0.0, r_hi=1.0):
    z = rng.standard_normal((K, d))
    r = r_lo + (r_hi - r_lo) * rng.uniform(0, 1, (K, 1)) ** (1.0 / d)
    return (z / np.linalg.norm(z, axis=1, keepdims=True) * r).astype(np.float32)


def _chunked(fn, K, chunk):
    """Run the oracle over path chunks (one tape per step per chunk bounds its memory); the gradient is a per-path sum,
    the chunk's loss weight alpha_0 = K_chunk / K keeps w = 2 r / K."""
    parts = [fn(lo, min(K, lo + chunk), (min(K, lo + chunk) - lo) / K) for lo in range(0, K, chunk)]
    out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k not in ("grad", "K_count", "loss", "loss_boundary")}
    out["grad"] = sum(p["grad"] for p in parts)
    out["K_count"] = sum(p["K_count"] for p in parts)
    return out


_ORACLE = {}


def diffusion_case(abi, kind, d, arch, K, N, dt, noise, seed=7, chunk=1024):
    """GeneralSolver's kernels (heat: h = 0; allencahn: h = y - y^3, which adds the backward's V(X_n) pass) with t_0 in
    [0.9, 1): every tile mixes moving and stopped paths.  noise 'inject' feeds the Philox dump back as injected draws."""
    T = 1.0
    dims = [d + 1] + list(arch) + [1]
    theta = _theta(dims, seed)
    rng = np.random.default_rng(seed)
    X0 = _ball(rng, K, d)
    t0 = rng.uniform(0.9, 1.0, K).astype(np.float32)
    pid = L.PROBLEM_HEAT if kind == "heat" else L.PROBLEM_ALLEN_CAHN
    cfg = H.diffusion_cfg(K, d, N, dt, arch, noise=L.NOISE_PHILOX, seed=seed, offset=2, problem_id=pid)
    xs = abi.philox_dump(cfg)
    if noise == "inject":
        cfg = H.diffusion_cfg(K, d, N, dt, arch, noise=L.NOISE_INJECT, seed=seed, offset=2, problem_id=pid)
    pack = H.heat_pack(d)
    xin = xs if noise == "inject" else None
    f = abi.diff_fwd(cfg, T, theta, pack, X0, t0, xin)
    r = f["VE"].astype(np.float64) - f["Y"]
    w = 2 * r / K
    grad = abi.diff_bwd(cfg, T, theta, pack, X0, t0, xin, -w, w, -w)
    key = ("diff", kind, d, tuple(arch), K, N, dt, seed, xs.tobytes().__hash__())
    if key not in _ORACLE:
        net = man.Net("densenet", dims, theta.astype(np.float64))
        pde = None if kind == "heat" else man.ALLEN_CAHN
        X64, t64, x64 = X0.astype(np.float64), t0.astype(np.float64), xs.astype(np.float64)

        def part(lo, hi, a0):
            m = man.diffusion(man.Problem("heat", d), net, X64[lo:hi], t64[lo:hi], x64[:, lo:hi], dt, N, 1,
                              alpha=(a0, 0.0, 0.0), T=T, pde=pde)
            m["VE"] = net.forward(np.concatenate([m["X"], m["t"][:, None]], 1))[0][:, 0]
            m["V0"] = net.forward(np.concatenate([X64[lo:hi], t64[lo:hi, None]], 1))[0][:, 0]
            return m
        _ORACLE[key] = _chunked(part, K, chunk)
    m = _ORACLE[key]
    assert 0 < m["K_count"] < K * N and int(f["stats"][1]) == m["K_count"]
    assert relerr(f["X"], m["X"]) < TOL_END and relerr(f["t"], m["t"]) < TOL_END
    for k in ("Y", "VE", "V0"):
        assert relerr(f[k], m[k]) < TOL_PATH, (k, relerr(f[k], m[k]))
    assert f["stats"][3] == 0
    np.testing.assert_allclose(f["stats"][[0, 2]], [(r * r).sum(), r.sum()], rtol=1e-9)
    check_grad(grad, m["grad"], grad_blocks("densenet", dims), "diffusion %s %s" % (kind, noise))


def elliptic_case(abi, kind, d, arch, K, N, dt, seed=9, chunk=2048):
    """EllipticSolver's kernels on the unit ball ('sphere': h = expball_sin), a one-sided box ('box': h =
    exp-nonlinear, alpha = 1/2) and the committor annulus 1 < |x| < 2 ('committor': h = 0, sigma = I)."""
    dims = [d] + list(arch) + [1]
    theta = _theta(dims, seed)
    rng = np.random.default_rng(seed)
    pack = H.heat_pack(d)
    if kind == "sphere":
        ell, mp, X0 = H.elliptic_spec("expball_sin"), man.EllipticProblem("expball_sin", d), _ball(rng, K, d)
    elif kind == "box":
        ell = L.make_elliptic(L.DOMAIN_BOX, x_l=-1.0, x_r=1.0, one_boundary=True, h_id=L.H_EXP_NONLINEAR,
                              h_param=(0.5, 0, 0))
        mp = man.EllipticProblem("expball", d, alpha=0.5)
        mp.boundary, mp.one_boundary, mp.X_l, mp.X_r = "square", True, -1.0, 1.0
        X0 = rng.uniform(-1, 1, (K, d)).astype(np.float32)
    else:
        ell, mp, X0 = H.elliptic_spec("committor"), man.EllipticProblem("committor", d), _ball(rng, K, d, 1.02, 1.98)
        pack[d:2 * d] = 1.0
    cfg = H.elliptic_cfg(K, d, N, dt, arch, noise=L.NOISE_PHILOX, seed=seed, offset=1, k_offset=3)
    xs = abi.philox_dump(cfg)
    f = abi.diff_fwd(cfg, 1.0, theta, pack, X0, None, None, ell=ell)
    r = f["VE"].astype(np.float64) - f["Y"]
    w = 2 * r / K
    grad = abi.diff_bwd(cfg, 1.0, theta, pack, X0, None, None, -w, w, -w, ell=ell)
    key = ("ell", kind, d, tuple(arch), K, N, dt, seed, xs.tobytes().__hash__())
    if key not in _ORACLE:
        net = man.Net("densenet", dims, theta.astype(np.float64))
        X64, x64 = X0.astype(np.float64), xs.astype(np.float64)

        def part(lo, hi, a0):
            m = man.elliptic(mp, net, X64[lo:lo + 1], X64[lo:hi], x64[:, lo:hi], dt, N, alpha=(a0, 0.0))
            m["VE"] = m["r"] + m["Y"]
            return m
        _ORACLE[key] = _chunked(part, K, chunk)
    m = _ORACLE[key]
    assert 0 < m["K_count"] < K * N and int(f["stats"][1]) == m["K_count"]
    assert relerr(f["X"], m["X"]) < TOL_END
    for k in ("Y", "VE"):
        assert relerr(f[k], m[k]) < TOL_PATH, (k, relerr(f[k], m[k]))
    assert relerr(f["VL2"], m["V_L2"]) < (1e-4 if kind == "committor" else TOL_PATH), relerr(f["VL2"], m["V_L2"])
    assert f["stats"][3] == 0
    np.testing.assert_allclose(f["stats"][[0, 2]], [(r * r).sum(), r.sum()], rtol=1e-9)
    check_grad(grad, m["grad"], grad_blocks("densenet", dims), "elliptic %s" % kind)


# ------------------------------------------------------------------------------------------------ start points
def sample_case(abi, K, d, k_offset, seed=11, offset=4, radius=1.5, T=1.0):
    """diffusion_sample_kernel against its restatement (oracle/philox.py::ball_and_time)."""
    from oracle import philox as ph
    cfg = H.diffusion_cfg(K, d, 1, 0.01, (8,), noise=L.NOISE_PHILOX, k_offset=k_offset, seed=seed, offset=offset)
    X0, t0 = abi.sample(cfg, radius, T)
    Xr, tr = ph.ball_and_time(seed, offset, k_offset, K, d, radius, T)
    assert relerr(X0, Xr) < TOL_PATH and relerr(t0, tr) < TOL_PATH
    assert np.abs(np.linalg.norm(X0, axis=1) - np.linalg.norm(Xr, axis=1)).max() < TOL_PATH * radius
    return X0, t0


def sample_uniformity(X0, t0, radius, T):
    """(|X_0| / R)^d and t_0 / T are U(0, 1) if X_0 is uniform in the ball and t_0 uniform in [0, T): KS p-values."""
    from scipy import stats
    d = X0.shape[1]
    rad = (np.linalg.norm(X0.astype(np.float64), axis=1) / radius) ** d
    return stats.kstest(rad, "uniform").pvalue, stats.kstest(t0.astype(np.float64) / T, "uniform").pvalue


# ------------------------------------------------------------------------------------------ tensor-core rollout / gradient
P_TC = 128                      # paths per tile of rollout_tc_fwd_kernel (tensor-memory lanes)

# Shapes of the tensor-core kernels: (problem, d, network, hidden widths, N, dt).  The column groups per thread of the
# forward (TcGeom::ng) are 7 for c2 and d102, 4 for c3, 2 for lqgc7.
TC_SHAPES = {
    "c2": ("llgc", 100, "densenet", (30, 30), 10, 0.01),         # C2 / C5: LLGC d = 100, DenseNet [30, 30]
    "c3": ("dwm", 50, "mlp_tanh", (30, 30), 10, 0.005),          # C3: DoubleWell d = 50 (d_1 = 15, kappa = 5, eta = 3)
    "lqgc7": ("lqgc", 7, "densenet", (30, 30), 8, 0.02),         # d % 4 != 0
    "d102": ("llgc", 102, "densenet", (32, 32), 8, 0.01),        # all 512 tensor-memory columns
}


class TcCase:
    """Inputs of one tensor-core case: K paths from 0, the network, random-sign cotangents with every 7th path exactly
    zero, the kernels' Philox increments; `oracle()` is the fp64 rollout + gradient (man.grad_mode_a) on them."""

    def __init__(self, abi, shape, K, adaptive=True, wz=False, seed=5, offset=3, x0_per_path=False, y0=None):
        kind, d, net, arch, N, dt = TC_SHAPES[shape] if isinstance(shape, str) else shape
        self.shape, self.kind, self.d, self.net, self.N, self.K = shape, kind, d, net, N, K
        self.dt, self.adaptive, self.seed, self.offset = np.float32(dt), adaptive, seed, offset
        self.dims = [d + 1] + list(arch) + [d]
        self.mp, (self.pid, self.flags, self.pack), self.x0 = hjb_problem(kind, d)
        self.y0 = y0
        cfg = self.cfg()
        n_theta = abi.lib.pspde_theta_size(ctypes.byref(cfg))
        assert n_theta > 0, abi.lib.pspde_last_error()
        rng = np.random.default_rng(seed)
        self.theta = (0.1 * rng.standard_normal(n_theta)).astype(np.float32)
        self.wY = (rng.choice([-1.0, 1.0], K) * (0.5 + rng.uniform(0, 1, K)) / K).astype(np.float32)
        self.wZ = (rng.standard_normal(K) / K).astype(np.float32) if wz else None
        for w in (self.wY, self.wZ):
            if w is not None:
                w[::7] = 0.0
        self.xi_dump = abi.philox_dump(cfg)                          # (N, K, d)
        # u_L2 table of the diagnostic, mode 1: u*(x, t_n)_j = tab[2 n, j] + tab[2 n + 1, j] x_j
        self.table = (0.3 * rng.standard_normal((2 * N, d))).astype(np.float32)
        if x0_per_path:                                              # one start point per path around the problem's X_0
            self.x0 = (self.x0 + 0.5 * rng.standard_normal((K, d))).astype(np.float32)

    def cfg(self, K_local=None, k_offset=0, inject=False):
        strides = (self.d * (self.N + 1), self.N + 1, 1) if inject else (0, 0, 0)
        return L.make_cfg(self.K if K_local is None else K_local, self.d, self.N, self.dt, self.pid,
                          L.NET_DENSENET if self.net == "densenet" else L.NET_MLP_TANH, self.dims, L.TIME_FIRST,
                          adaptive=self.adaptive, k_offset=k_offset, problem_flags=self.flags,
                          noise_mode=L.NOISE_INJECT if inject else L.NOISE_PHILOX, seed=self.seed, offset=self.offset,
                          xi_strides=strides, x0_per_path=self.x0.ndim == 2)

    def xi_ref(self, lo=0, hi=None):
        """The Philox increments of paths [lo, hi) in the reference layout (K, d, N + 1), float32."""
        xi = np.zeros((self.K if hi is None else hi - lo, self.d, self.N + 1), np.float32)
        xi[:, :, 1:] = self.xi_dump[:, lo:hi].transpose(1, 2, 0)
        return xi

    def oracle(self, chunk=4096):
        """fp64: X_N, Y_N, g(X_N), Z_sum and u_L2 per path (u_l2), and the gradient of sum_k wY_k Y_N,k + wZ_k Z_sum,k."""
        key = ("tc", self.shape, self.K, self.adaptive, self.wZ is not None, self.seed, self.offset, self.x0.ndim, self.y0)
        if key in _ORACLE:
            return _ORACLE[key]
        net = man.Net(self.net, self.dims, self.theta.astype(np.float64))
        dt = float(self.dt)
        wZ = np.zeros(self.K) if self.wZ is None else self.wZ.astype(np.float64)
        x0 = self.x0.astype(np.float64)
        parts = []
        for lo in range(0, self.K, chunk):
            hi = min(self.K, lo + chunk)
            g, ro = man.grad_mode_a(self.mp, net, self.xi_ref(lo, hi).astype(np.float64), dt, self.N,
                                    x0[lo:hi] if x0.ndim == 2 else x0, self.wY[lo:hi].astype(np.float64), wZ[lo:hi],
                                    self.adaptive, "first", float(np.float32(self.y0 or 0.0)))
            parts.append(dict(grad=g, X=ro["X"], Y=ro["Y"], gX=ro["gX"], Zsum=ro["Zsum"], uL2=u_l2(self.table, ro, dt)))
        out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "grad"}
        out["grad"] = sum(p["grad"] for p in parts)
        _ORACLE[key] = out
        return out

    def blocks(self):
        return grad_blocks(self.net, self.dims)


def u_l2(table, ro, dt):
    """The u_L2 diagnostic of mode 1 (u*(x, t_n)_j = table[2 n, j] + table[2 n + 1, j] x_j) on an oracle rollout ro, as
    the forward sweeps sum it (solver.py:491-494): sum_n dt sum_j (-Z_n,j - u*(X_n+1, t_n)_j)^2 per path."""
    tab = table.astype(np.float64)
    ul = 0.0
    for n in range(len(ro["Z"])):
        u = tab[2 * n] + tab[2 * n + 1] * ro["path"][n + 1]
        ul = ul + dt * ((-ro["Z"][n] - u) ** 2).sum(1)
    return ul


def check_tc_forward(o, m, tol_end=TOL_END):
    """Per-path outputs of a tensor-core forward against the oracle, and its stats."""
    assert relerr(o["X"], m["X"]) < tol_end, ("X_N", relerr(o["X"], m["X"]))
    for k in ("Y", "gX", "Zsum"):
        assert relerr(o[k], m[k]) < TOL_PATH, (k, relerr(o[k], m[k]))
    check_stats(o)


def check_stats(o):
    """The stats vector (sum D, sum D^2, sum Z_sum + g, dropped paths; D = Y_N - g(X_N)) against a host recomputation
    from the per-path outputs it was reduced from."""
    D = o["Y"].astype(np.float64) - o["gX"]
    ref = np.array([D.sum(), (D * D).sum(), (o["Zsum"].astype(np.float64) + o["gX"]).sum(), 0.0])
    scale = np.array([np.abs(D).sum(), (D * D).sum(), np.abs(o["Zsum"].astype(np.float64) + o["gX"]).sum(), 1.0])
    assert np.all(np.abs(o["stats"] - ref) <= 1e-9 * scale), (o["stats"], ref)
