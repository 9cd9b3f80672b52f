"""Explicit-formula oracle (numpy) for the gradients of the path-space losses.

TEST INFRASTRUCTURE -- not product code (see oracle/ref_port.py for the rules).  Where ref_port.py restates the
reference *procedurally* (rollout + autograd), this file restates the closed-form gradient structure the CUDA
kernels implement, in float64 by default, so that (i) the derivations in DESIGN.md are pinned against the
reference fixtures and (ii) tests get condition-aware tolerances from a high-precision evaluation.

  Mode A  detached forward (solver.py:468-469): X is theta-independent, per-(k,n) VJPs only.
          cotangent on Z_n:  zeta = wY*(sqrt(dt)*xi_{n+1} + [not adaptive]*Z*dt) + wZ*Z*dt
  Mode B  attached forward, relative entropy (solver.py:180, :486): discrete adjoint lambda_n.
  Mode D  diffusion loss (solver.py:1076-1163), h == 0: value + x-tangent forward, reverse of both.

Parity pin: tests/test_oracle_golden.py checks all three against tests/golden/*.npz (reference outputs).
"""
import numpy as np


# ------------------------------------------------------------------ network spec
class Net:
    """kind 'densenet' (relu^2, dense concat; W (fan_in, out)) or 'mlp_tanh' (nn.Linear W (out, in))."""

    def __init__(self, kind, dims, theta, dtype=np.float64):
        self.kind, self.dims = kind, list(dims)
        self.W, self.b = [], []
        off = 0
        theta = np.asarray(theta, dtype=dtype)
        for i in range(len(dims) - 1):
            fan_in = sum(dims[:i + 1]) if kind == "densenet" else dims[i]
            n = fan_in * dims[i + 1]
            if kind == "densenet":
                self.W.append(theta[off:off + n].reshape(fan_in, dims[i + 1]))
            else:
                self.W.append(theta[off:off + n].reshape(dims[i + 1], fan_in).T)   # store as (in, out)
            off += n
            self.b.append(theta[off:off + dims[i + 1]])
            off += dims[i + 1]
        self.n_params = off
        assert off == theta.size, (off, theta.size)

    def act(self, pre):
        return np.maximum(pre, 0) ** 2 if self.kind == "densenet" else np.tanh(pre)

    def dact(self, pre, h):
        return 2 * np.maximum(pre, 0) if self.kind == "densenet" else 1 - h ** 2

    def d2act(self, pre, h):
        return 2.0 * (pre > 0) if self.kind == "densenet" else -2 * h * (1 - h ** 2)

    def forward(self, a0):
        """returns output and the tape [(a_l, pre_l, h_l)]."""
        a, tape = a0, []
        L = len(self.W)
        for l in range(L):
            pre = a @ self.W[l] + self.b[l]
            if l == L - 1:
                tape.append((a, pre, None))
                return pre, tape
            h = self.act(pre)
            tape.append((a, pre, h))
            a = np.concatenate([a, h], 1) if self.kind == "densenet" else h

    def vjp(self, tape, zeta, want_dx=False):
        """theta-gradient (flat, parameter order) of sum(out*zeta); optionally d/d a0."""
        L = len(self.W)
        gW, gb = [None] * L, [None] * L
        delta = zeta
        abar = None                                  # cotangent on the (concat) activation row
        for l in range(L - 1, -1, -1):
            a, pre, h = tape[l]
            if l < L - 1:
                if self.kind == "densenet":
                    hbar = abar[:, a.shape[1]:]
                    abar = abar[:, :a.shape[1]]
                else:
                    hbar, abar = abar, None
                delta = hbar * self.dact(pre, h)
            gW[l] = a.T @ delta
            gb[l] = delta.sum(0)
            contrib = delta @ self.W[l].T
            abar = contrib if abar is None else abar + contrib
        flat = []
        for l in range(L):
            flat.append((gW[l] if self.kind == "densenet" else gW[l].T).reshape(-1))
            flat.append(gb[l])
        g = np.concatenate(flat)
        return (g, abar) if want_dx else g

    # ---- forward-mode tangent + its reverse (diffusion loss)
    def forward_tangent(self, a0, da0):
        a, da, tape = a0, da0, []
        L = len(self.W)
        for l in range(L):
            pre = a @ self.W[l] + self.b[l]
            dpre = da @ self.W[l]
            if l == L - 1:
                tape.append((a, da, pre, dpre, None))
                return pre, dpre, tape
            h = self.act(pre)
            dh = self.dact(pre, h) * dpre
            tape.append((a, da, pre, dpre, h))
            if self.kind == "densenet":
                a, da = np.concatenate([a, h], 1), np.concatenate([da, dh], 1)
            else:
                a, da = h, dh

    def vjp_tangent(self, tape, ybar, dybar):
        """theta-gradient of sum(y*ybar + y'*dybar) for the pair (value y, tangent y')."""
        L = len(self.W)
        gW, gb = [None] * L, [None] * L
        pbar, dpbar = ybar, dybar
        abar = dabar = None
        for l in range(L - 1, -1, -1):
            a, da, pre, dpre, h = tape[l]
            if l < L - 1:
                if self.kind == "densenet":
                    hbar, dhbar = abar[:, a.shape[1]:], dabar[:, a.shape[1]:]
                    abar, dabar = abar[:, :a.shape[1]], dabar[:, :a.shape[1]]
                else:
                    hbar, dhbar, abar, dabar = abar, dabar, None, None
                d1 = self.dact(pre, h)
                dpbar = dhbar * d1
                pbar = hbar * d1 + dhbar * self.d2act(pre, h) * dpre
            gW[l] = a.T @ pbar + da.T @ dpbar
            gb[l] = pbar.sum(0)
            c, dc = pbar @ self.W[l].T, dpbar @ self.W[l].T
            abar = c if abar is None else abar + c
            dabar = dc if dabar is None else dabar + dc
        flat = []
        for l in range(L):
            flat.append((gW[l] if self.kind == "densenet" else gW[l].T).reshape(-1))
            flat.append(gb[l])
        return np.concatenate(flat)


# ------------------------------------------------------------------ problems (numpy)
class Problem:
    def __init__(self, kind, d, dtype=np.float64, A=None, B=None, eta_=None, kappa_=None):
        self.kind, self.d = kind, d
        I = np.eye(d, dtype=dtype)
        self.A = -I if A is None else np.asarray(A, dtype)
        self.B = I if B is None else np.asarray(B, dtype)
        if kind == "dwm":
            self.B = I
            self.eta_, self.kappa_ = np.asarray(eta_, dtype), np.asarray(kappa_, dtype)
        if kind == "heat":
            self.B = np.sqrt(dtype(2.0)) * I
        self.P, self.R, self.alpha = 0.5 * I, I, np.ones(d, dtype)

    def b(self, x):
        if self.kind in ("llgc", "lqgc"):
            return x @ self.A.T
        if self.kind == "dwm":
            return -4.0 * self.kappa_ * x * (x ** 2 - 1)
        return np.zeros_like(x)

    def Jb_T_vec(self, x, lam):          # J_b(x)^T lam, row convention
        if self.kind in ("llgc", "lqgc"):
            return lam @ self.A
        return -4.0 * self.kappa_ * (3 * x ** 2 - 1) * lam

    def f(self, x):
        return ((x @ self.P.T) * x).sum(1) if self.kind == "lqgc" else np.zeros(x.shape[0], x.dtype)

    def grad_f(self, x):
        return x @ (self.P + self.P.T) if self.kind == "lqgc" else np.zeros_like(x)

    def g(self, x):
        if self.kind == "llgc":
            return x @ self.alpha
        if self.kind == "lqgc":
            return ((x @ self.R.T) * x).sum(1)
        return (self.eta_ * (x - 1) ** 2).sum(1)

    def grad_g(self, x):
        if self.kind == "llgc":
            return np.tile(self.alpha, (x.shape[0], 1))
        if self.kind == "lqgc":
            return x @ (self.R + self.R.T)
        return 2 * self.eta_ * (x - 1)


def net_input(X, n, dt, time_mode):
    t = np.full((X.shape[0], 1), np.float32(n) * np.float32(dt), dtype=X.dtype)
    if time_mode == "first":
        return np.concatenate([t, X], 1)
    return X


def step_net(nets, n, dt, t_index=None, dt_net=None):
    """(network, time index, grid spacing) that step n evaluates: n on the step grid, or t_index[n] on a network grid of
    spacing dt_net (importance sampling on another grid: Solver.Z_n, solver.py:360-362, rollout_kernels.cuh's n_net /
    t_net).  In 'outer' mode (nets a list) the parameter set is that index clamped to [0, len(nets) - 1] (:352)."""
    n_net, dtn = (n, dt) if t_index is None else (int(t_index[n]), dt_net)
    if isinstance(nets, list):
        return nets[min(max(n_net, 0), len(nets) - 1)], n_net, dtn
    return nets, n_net, dtn


def start_states(X0, K, dtype):
    """X_0 of the K paths: one row for all (tiled) or one row per path (pspde_cfg::x0_per_path)."""
    X0 = np.asarray(X0, dtype)
    return np.tile(X0, (K, 1)) if X0.ndim == 1 else X0.copy()


# ------------------------------------------------------------------ HJB rollout (solver.py:440-489)
def rollout(problem, nets, xi, dt, N, X0, adaptive=True, y0=0.0, time_mode="first", t_index=None, dt_net=None):
    """nets: one Net (inner) or a list of Nets (outer). xi (K,d,N+1). X0 (d,) or (K, d). t_index / dt_net: see
    step_net. Returns dict with the X path and Fint = sum_n f(X_{n+1}) dt."""
    K = xi.shape[0]
    dtype = xi.dtype
    s = np.sqrt(dtype.type(dt))
    X = start_states(X0, K, dtype)
    Y = np.full(K, y0, dtype)
    Zsum = np.zeros(K, dtype)
    Fint = np.zeros(K, dtype)
    path, Zs = [X], []
    for n in range(N):
        net, n_net, dtn = step_net(nets, n, dt, t_index, dt_net)
        Z, _ = net.forward(net_input(X, n_net, dtn, time_mode))
        c = -Z if adaptive else np.zeros_like(Z)
        x = xi[:, :, n + 1]
        X = X + (problem.b(X) + c @ problem.B.T) * dt + (x @ problem.B.T) * s
        fX = problem.f(X)
        zz = (Z ** 2).sum(1)
        Y = Y + ((0.5 * zz + fX) + (Z * c).sum(1)) * dt + (Z * x).sum(1) * s
        Zsum = Zsum + (0.5 * zz + fX) * dt
        Fint = Fint + fX * dt
        path.append(X)
        Zs.append(Z)
    return dict(X=X, Y=Y, Zsum=Zsum, Fint=Fint, gX=problem.g(X), path=path, Z=Zs)


def loss_and_weights(loss_method, Y, gX, Zsum, adaptive=True):
    """Loss value and per-path cotangents (wY on Y_N, wZ on Z_sum) -- solver.py:164-192 differentiated by hand."""
    K = Y.shape[0]
    D = Y - gX
    zero = np.zeros_like(Y)
    if loss_method == "moment":
        return (D ** 2).mean(), 2 * D / K, zero
    if loss_method == "log-variance":
        return (D ** 2).mean() - D.mean() ** 2, 2 * (D - D.mean()) / K, zero
    if loss_method == "variance":
        E = np.exp(D)
        return E.var(ddof=1), 2 * (E - E.mean()) * E / (K - 1), zero
    if loss_method == "cross_entropy":
        E = np.exp(D) if adaptive else np.exp(-gX)
        return (Y * E).mean(), E / K, zero
    if loss_method == "relative_entropy":
        return (Zsum + gX).mean(), zero, np.full_like(Y, 1.0 / K)
    raise ValueError(loss_method)


def grad_mode_a(problem, nets, xi, dt, N, X0, wY, wZ, adaptive=True, time_mode="first", y0=0.0, t_index=None,
                dt_net=None):
    """SURVEY.md A.3 generalised: detached forward, one VJP per (k, n).  X0, t_index, dt_net: as in rollout."""
    dtype = xi.dtype
    s = np.sqrt(dtype.type(dt))
    ro = rollout(problem, nets, xi, dt, N, X0, adaptive, y0, time_mode, t_index, dt_net)
    outer = isinstance(nets, list)
    grads = [0.0] * (len(nets) if outer else 1)
    for n in range(N):
        net, n_net, dtn = step_net(nets, n, dt, t_index, dt_net)
        Z, tape = net.forward(net_input(ro["path"][n], n_net, dtn, time_mode))
        zeta = wY[:, None] * (s * xi[:, :, n + 1] + (0.0 if adaptive else 1.0) * Z * dt) + wZ[:, None] * Z * dt
        g = net.vjp(tape, zeta)
        i = min(max(n_net, 0), len(nets) - 1) if outer else 0
        grads[i] = grads[i] + g
    return np.concatenate([np.atleast_1d(g) for g in grads]), ro


def grad_mode_b(problem, net, xi, dt, N, X0, time_mode="first"):
    """SURVEY.md A.4: relative entropy, attached adaptive forward, discrete adjoint (w = 1/K)."""
    K = xi.shape[0]
    ro = rollout(problem, net, xi, dt, N, X0, True, 0.0, time_mode)
    lam = problem.grad_g(ro["X"]) / K
    grad = 0.0
    x_lo = 1 if time_mode == "first" else 0
    for n in range(N - 1, -1, -1):
        Xn = ro["path"][n]
        lam = lam + problem.grad_f(ro["path"][n + 1]) * dt / K
        Z, tape = net.forward(net_input(Xn, n, dt, time_mode))
        zeta = Z * dt / K - dt * (lam @ problem.B)
        g, dx = net.vjp(tape, zeta, want_dx=True)
        grad = grad + g
        lam = lam + dt * problem.Jb_T_vec(Xn, lam) + dx[:, x_lo:x_lo + problem.d]
    return grad, ro


def loss_cotangents_full(loss_method, Y, gX, Zsum, adaptive=True):
    """(loss, wY, wZ, wG): cotangents on Y_N, Z_sum and g(X_N) -- needed when X depends on theta (attached mode)."""
    K = Y.shape[0]
    loss, wY, wZ = loss_and_weights(loss_method, Y, gX, Zsum, adaptive)
    if loss_method == "relative_entropy":
        wG = np.full_like(Y, 1.0 / K)
    elif loss_method == "cross_entropy":
        E = np.exp(Y - gX) if adaptive else np.exp(-gX)
        wG = -Y * E / K
    else:                       # log-variance, moment, variance depend on D = Y - g only
        wG = -wY
    return loss, wY, wZ, wG


def grad_attached(problem, nets, xi, dt, N, X0, wY, wZ, wG, time_mode="first", y0=0.0):
    """Discrete adjoint for the attached adaptive forward process (c = -Z, not detached) and ANY loss given as
    per-path cotangents (wY on Y_N, wZ on Z_sum, wG on g(X_N)):
        lambda_N = wG grad g(X_N)
        n = N-1..0:  lambda += (wY + wZ) dt grad f(X_{n+1})
                     zeta = wY (-Z dt + sqrt(dt) xi) + wZ Z dt - dt (lambda B)
                     dtheta += J_theta' zeta ;  lambda += dt J_b' lambda + J_x' zeta
    (Y+ = Y + (f(X+) - |Z|^2/2) dt + Z.xi sqrt(dt), Zsum+ = Zsum + (|Z|^2/2 + f(X+)) dt, X+ = X + (b - BZ) dt + B xi sqrt(dt))."""
    dtype = xi.dtype
    s = np.sqrt(dtype.type(dt))
    ro = rollout(problem, nets, xi, dt, N, X0, True, y0, time_mode)
    outer = isinstance(nets, list)
    grads = [0.0] * (N if outer else 1)
    lam = wG[:, None] * problem.grad_g(ro["X"])
    for n in range(N - 1, -1, -1):
        net = nets[n] if outer else nets
        Xn = ro["path"][n]
        lam = lam + (wY + wZ)[:, None] * problem.grad_f(ro["path"][n + 1]) * dt
        Z, tape = net.forward(net_input(Xn, n, dt, time_mode))
        zeta = wY[:, None] * (-Z * dt + s * xi[:, :, n + 1]) + wZ[:, None] * Z * dt - dt * (lam @ problem.B)
        g, dx = net.vjp(tape, zeta, want_dx=True)
        grads[n if outer else 0] = grads[n if outer else 0] + g
        x_lo = 1 if time_mode == "first" else 0
        lam = lam + dt * problem.Jb_T_vec(Xn, lam) + dx[:, x_lo:x_lo + problem.d]
    return np.concatenate([np.atleast_1d(g) for g in grads]), ro


# ------------------------------------------------------------------ diffusion loss (solver.py:1062-1163, h == 0)
ALLEN_CAHN = dict(h=lambda y: y - y ** 3, h_y=lambda y: 1 - 3 * y ** 2, f=lambda x: 1 / (2 + 2 / 5 * (x ** 2).sum(1)))


def diffusion(problem, net, X0, t0, xis, dt, N, K_boundary, alpha=(1.0, 1.0, 1.0), T=1.0, pde=None):
    """Value and theta-gradient of the diffusion loss, unbounded domain, non-adaptive; net input is [X, t].
    pde = None: heat equation (h == 0, terminal |x|^2); pde = ALLEN_CAHN: h(y) = y - y^3, the value row of every
    active step then carries the cotangent w act h_y dt (as in `elliptic` below)."""
    dtype = X0.dtype
    K, d = X0.shape
    dt = dtype.type(np.float32(dt))
    s = np.sqrt(dt)
    Bt = problem.B.T
    # terminal-condition term on the first K_boundary interior samples (:1063-1064)
    aT = np.concatenate([X0[:K_boundary], np.full((K_boundary, 1), T, dtype)], 1)
    vT, tapeT = net.forward(aT)
    fT = (X0[:K_boundary] ** 2).sum(1) if pde is None else pde["f"](X0[:K_boundary])
    rT = vT[:, 0] - fT
    loss = alpha[1] * (rT ** 2).mean()
    grad = net.vjp(tapeT, (alpha[1] * 2 * rT / K_boundary)[:, None])
    # pass 1: values
    X, t = X0.copy(), t0.reshape(-1).copy()
    v0, tape0 = net.forward(np.concatenate([X, t[:, None]], 1))
    Y = v0[:, 0].copy()
    stopped = np.zeros(K, bool)
    steps = []
    K_count = 0
    for n in range(N):
        if not (~stopped).any():
            break
        act = (~stopped) & ((t.astype(np.float32) + np.float32(dt)) <= np.float32(T))
        v = (xis[n] @ Bt) * s                                      # direction B xi sqrt(dt)
        a0 = np.concatenate([X, t[:, None]], 1)
        da0 = np.concatenate([v, np.zeros((K, 1), dtype)], 1)
        y, dy, tape = net.forward_tangent(a0, da0)
        hy = np.zeros(K, dtype)
        if pde is not None:
            Y = Y - pde["h"](y[:, 0]) * dt * act
            hy = pde["h_y"](y[:, 0])
        Y = Y + dy[:, 0] * act
        steps.append((tape, act.copy(), hy))
        X = X + (problem.b(X) * dt + v) * act[:, None]
        t = t + dt * act
        K_count += int(act.sum())
        stopped |= ~act
    vE, tapeE = net.forward(np.concatenate([X, t[:, None]], 1))
    r = vE[:, 0] - Y
    loss = loss + alpha[0] * (r ** 2).mean()
    w = alpha[0] * 2 * r / K
    grad = grad + net.vjp(tapeE, w[:, None]) - net.vjp(tape0, w[:, None])
    for tape, act, hy in steps:
        grad = grad + net.vjp_tangent(tape, (w * act * hy * dt)[:, None], (-w * act)[:, None])
    return dict(loss=loss, grad=grad, K_count=K_count, X=X, t=t, Y=Y)


# ------------------------------------------------------------------ elliptic diffusion loss (solver.py:628-790)
class EllipticProblem:
    """numpy functors of the elliptic problems (problems.py:962-1064, :1614-1654): b = 0, sigma = sqrt(2) I,
    h(x, y) with its y-derivative, Dirichlet data g, exact solution v_true."""

    def __init__(self, kind, d, alpha=1.0, dtype=np.float64):
        self.kind, self.d, self.alpha, self.dtype = kind, d, float(alpha), dtype
        self.B = np.sqrt(dtype(2.0)) * np.eye(d, dtype=dtype)
        if kind == "helmholtz":
            self.boundary, self.one_boundary, self.X_l, self.X_r = "square", False, -1.0, 1.0
            self.a_1, self.a_2, self.k = 1.0, 4.0, 1.0
        elif kind == "committor":
            self.boundary, self.r_in, self.r_out = "two_spheres", 1.0, 2.0
            self.B = np.eye(d, dtype=dtype)
        else:
            self.boundary, self.boundary_distance = "sphere", 1.0

    def _ss(self, x):
        return np.sin(self.a_1 * np.pi * x[:, 0]) * np.sin(self.a_2 * np.pi * x[:, 1])

    def g(self, x):
        if self.kind == "committor":
            return (np.sqrt((x ** 2).sum(1)) > self.r_in).astype(x.dtype)
        return self._ss(x) if self.kind == "helmholtz" else np.exp(self.alpha * (x ** 2).sum(1))

    def v_true(self, x):
        if self.kind == "committor":
            a, c, d = self.r_in, self.r_out, self.d
            return (a ** 2 - np.sqrt((x ** 2).sum(1)) ** (2 - d) * a ** d) / (a ** 2 - c ** (2 - d) * a ** d)
        return self.g(x)

    def h(self, x, y):
        a, d, r2 = self.alpha, self.d, (x ** 2).sum(1)
        if self.kind == "expsphere":
            return -a * y * (4 * a * r2 + 2 * d)
        if self.kind == "expball":
            return -2 * a * y * (2 * a * r2 + d) + np.exp(2 * a * r2) - y ** 2
        if self.kind == "expball_sin":
            return -2 * a * y * (2 * a * r2 + d) + np.sin(np.exp(2 * a * r2) - y ** 2)
        if self.kind == "committor":
            return np.zeros(x.shape[0], x.dtype)
        c = (self.a_1 * np.pi) ** 2 + (self.a_2 * np.pi) ** 2 - self.k ** 2
        return self.k ** 2 * y + c * self._ss(x)

    def h_y(self, x, y):
        a, d, r2 = self.alpha, self.d, (x ** 2).sum(1)
        if self.kind == "expsphere":
            return -a * (4 * a * r2 + 2 * d)
        if self.kind == "expball":
            return -2 * a * (2 * a * r2 + d) - 2 * y
        if self.kind == "expball_sin":
            return -2 * a * (2 * a * r2 + d) - 2 * y * np.cos(np.exp(2 * a * r2) - y ** 2)
        if self.kind == "committor":
            return np.zeros(x.shape[0], x.dtype)
        return np.full(x.shape[0], self.k ** 2, dtype=x.dtype)

    def inside(self, X, X_prop):
        if self.boundary == "sphere":
            return np.sqrt((X ** 2).sum(1)) < self.boundary_distance          # solver.py:750-751: X, not the proposal
        if self.boundary == "two_spheres":
            r = np.sqrt((X ** 2).sum(1))
            return (r > self.r_in) & (r < self.r_out)                         # :752-753
        if self.one_boundary:
            return (X_prop <= self.X_r).all(1)
        return ((X_prop >= self.X_l) & (X_prop <= self.X_r)).all(1)


def elliptic(problem, net, Xb, X0, xis, dt, N, alpha=(1.0, 1.0), gb=None):
    """Value and theta-gradient of the elliptic diffusion loss (non-adaptive, Dirichlet term); net input is X.
        Y = V(X_0) + sum_n act_n (-h(X_n, V(X_n)) dt + grad V(X_n) . B xi_n sqrt(dt)),  r = V(X_end) - Y
        dL = sum_k w_k [dV(X_end) - dV(X_0) + sum_n act_n (h_y dt dV(X_n) - d(grad V(X_n) . v_n))],  w = 2 alpha_0 r / K
    i.e. per step the (value, tangent) pair gets the cotangents (w act h_y dt, -w act)."""
    dtype = X0.dtype
    K, d = X0.shape
    dt = dtype.type(np.float32(dt))
    s = np.sqrt(dt)
    Bt = problem.B.T
    vb, tapeb = net.forward(Xb)
    rb = vb[:, 0] - (problem.g(Xb) if gb is None else gb)      # gb: boundary data evaluated by the caller (fp32 indicator)
    loss_b = alpha[1] * (rb ** 2).mean()
    grad = net.vjp(tapeb, (alpha[1] * 2 * rb / Xb.shape[0])[:, None])
    X = X0.copy()
    v0, tape0 = net.forward(X)
    Y = v0[:, 0].copy()
    stopped = np.zeros(K, bool)
    V_L2 = np.zeros(K, dtype)
    steps, K_count = [], 0
    for n in range(N):
        if not (~stopped).any():
            break
        v = (xis[n] @ Bt) * s
        y, dy, tape = net.forward_tangent(X, v)
        sel = ~stopped
        V_L2 += (y[:, 0] - problem.v_true(X)) ** 2 * dt * sel
        X_prop = X + v * sel[:, None]
        act = problem.inside(X, X_prop) & ~stopped
        Y = Y + (-problem.h(X, y[:, 0]) * dt + dy[:, 0]) * act
        steps.append((tape, act.copy(), problem.h_y(X, y[:, 0])))
        X = np.where(act[:, None], X_prop, X)
        K_count += int(act.sum())
        stopped |= ~act
    vE, tapeE = net.forward(X)
    r = vE[:, 0] - Y
    loss = loss_b + alpha[0] * (r ** 2).mean()
    w = alpha[0] * 2 * r / K
    grad = grad + net.vjp(tapeE, w[:, None]) - net.vjp(tape0, w[:, None])
    for tape, act, hy in steps:
        grad = grad + net.vjp_tangent(tape, (w * act * hy * dt)[:, None], (-w * act)[:, None])
    return dict(loss=loss, loss_boundary=loss_b, grad=grad, K_count=K_count, X=X, Y=Y, V_L2=V_L2, r=r)
