"""Pins the oracle (oracle/ref_port.py, oracle/manual.py) to outputs of the UNMODIFIED reference
(tests/golden/*.npz, produced by tests/golden/make_golden.py in the build container)."""
import numpy as np
import pytest
import torch as pt

from conftest import HJB_TAGS, load_golden, relerr
from oracle import manual as man
from oracle import ref_port as orc

pt.set_num_threads(1)


def net_dims(g):
    d = g["d"]
    d_in = d if g["time_approx"] == "outer" else d + 1
    return [d_in, 30, 30, d]


def split_theta(g):
    """flat theta -> parameter list(s) in the oracle's layout."""
    dims = net_dims(g)
    kind = g["net"]
    shapes = []
    for i in range(3):
        fan_in = sum(dims[:i + 1]) if kind == "densenet" else dims[i]
        shapes += [(fan_in, dims[i + 1]) if kind == "densenet" else (dims[i + 1], fan_in), (dims[i + 1],)]
    per = sum(int(np.prod(s)) for s in shapes)
    n_nets = g["theta"].size // per
    nets, off = [], 0
    for _ in range(n_nets):
        ps = []
        for s in shapes:
            n = int(np.prod(s))
            ps.append(pt.tensor(g["theta"][off:off + n].reshape(s)))
            off += n
        nets.append(ps)
    return (nets if g["time_approx"] == "outer" else nets[0]), per


@pytest.mark.parametrize("tag", HJB_TAGS)
def test_port_matches_reference(tag):
    g = load_golden(tag)
    prob = orc.make_problem(g["kind"], g["d"], **g["pkw"])
    params, _ = split_theta(g)
    y0 = pt.tensor([g["y0"]], dtype=pt.float32) if g["learn_Y_0"] else None
    o = orc.hjb_iteration(prob, g["net"], params, pt.tensor(g["xi"]), g["delta_t"], g["N"], g["loss_method"],
                          g["time_approx"], g["adaptive"], g["detach_forward"], y0=y0)
    flatg = np.concatenate([q.reshape(-1).numpy() for q in o["grads"]])
    assert relerr(o["X"], g["X_N"]) < 1e-6
    assert relerr(o["Y"], g["Y_N"]) < 1e-6
    assert abs(float(o["loss"]) - g["loss"]) <= 1e-6 * abs(g["loss"])
    assert relerr(flatg, g["grad"]) < (1e-5 if not g["detach_forward"] else 1e-6)   # fp32 autograd order noise
    if g["learn_Y_0"]:
        assert abs(float(o["grad_y0"]) - g["grad_y0"]) < 1e-5 * abs(g["grad_y0"])


@pytest.mark.parametrize("tag", HJB_TAGS)
def test_manual_formulas_match_reference(tag):
    """fp64 closed-form gradients (modes A and B) vs the reference's fp32 autograd."""
    g = load_golden(tag)
    d, N, dt = g["d"], g["N"], g["delta_t"]
    dims = net_dims(g)
    kw = {}
    if g["kind"] in ("llgc", "lqgc"):
        kw = dict(A=g["A"], B=g["B"])
    if g["kind"] == "dwm":
        p32 = orc.make_problem("dwm", d, **g["pkw"])
        kw = dict(eta_=p32.eta_.numpy(), kappa_=p32.kappa_.numpy())
    prob = man.Problem(g["kind"], d, **kw)
    outer = g["time_approx"] == "outer"
    per = g["theta"].size // (N if outer else 1)
    nets = [man.Net(g["net"], dims, g["theta"][i * per:(i + 1) * per]) for i in range(N if outer else 1)]
    nets = nets if outer else nets[0]
    X0 = -np.ones(d) if g["kind"] == "dwm" else np.zeros(d)
    xi = g["xi"].astype(np.float64)
    tm = "none" if outer else "first"
    if g["detach_forward"]:
        ro = man.rollout(prob, nets, xi, dt, N, X0, g["adaptive"], g["y0"], tm)
        loss, wY, wZ = man.loss_and_weights(g["loss_method"], ro["Y"], ro["gX"], ro["Zsum"], g["adaptive"])
        grad, _ = man.grad_mode_a(prob, nets, xi, dt, N, X0, wY, wZ, g["adaptive"], tm, g["y0"])
        if g["learn_Y_0"]:
            assert abs(wY.sum() - g["grad_y0"]) < 1e-4 * abs(g["grad_y0"])
    elif g["loss_method"] == "relative_entropy":
        grad, ro = man.grad_mode_b(prob, nets, xi, dt, N, X0, tm)
        loss = (ro["Zsum"] + ro["gX"]).mean()
    else:   # attached forward process with a general loss: two-phase (forward -> cotangents -> adjoint)
        ro = man.rollout(prob, nets, xi, dt, N, X0, True, g["y0"], tm)
        loss, wY, wZ, wG = man.loss_cotangents_full(g["loss_method"], ro["Y"], ro["gX"], ro["Zsum"], True)
        grad, _ = man.grad_attached(prob, nets, xi, dt, N, X0, wY, wZ, wG, tm, g["y0"])
    assert relerr(ro["X"], g["X_N"]) < 2e-6
    assert relerr(ro["Y"], g["Y_N"]) < 5e-6
    # condition-aware tolerance on the scalar (SURVEY.md finding 9): eps32 * E[D^2] bounds the fp32 cancellation
    D = ro["Y"] - ro["gX"]
    tol = 1e-5 * abs(g["loss"]) + 4 * 6e-8 * float((D ** 2).mean()) if "variance" in g["loss_method"] \
        else 1e-5 * abs(g["loss"])
    assert abs(loss - g["loss"]) <= tol
    assert relerr(grad, g["grad"]) < 2e-5


def test_diffusion_small_port_and_manual():
    g = load_golden("diff_heat_d10_small")
    d, arch = g["d"], list(g["arch"])
    dims = [d + 1] + arch + [1]
    shapes, params, off = [], [], 0
    for i in range(len(dims) - 1):
        shapes += [(sum(dims[:i + 1]), dims[i + 1]), (dims[i + 1],)]
    for s in shapes:
        n = int(np.prod(s))
        params.append(pt.tensor(g["theta"][off:off + n].reshape(s)))
        off += n
    prob = orc.make_problem("heat", d, T=1)
    o = orc.diffusion_iteration(prob, params, pt.tensor(g["X0"]), pt.tensor(g["t0"]), pt.tensor(g["xis"]),
                                g["delta_t"], g["N"], g["K_boundary"])
    assert abs(float(o["loss"]) - g["loss"]) < 1e-6 * g["loss"]
    assert o["K_count"] == g["K_count"]
    assert relerr(np.concatenate([q.reshape(-1).numpy() for q in o["grads"]]), g["grad"]) < 1e-6
    # explicit forward-over-reverse formulas (fp64)
    net = man.Net("densenet", dims, g["theta"])
    m = man.diffusion(man.Problem("heat", d), net, g["X0"].astype(np.float64), g["t0"].astype(np.float64),
                      g["xis"].astype(np.float64), g["delta_t"], g["N"], g["K_boundary"])
    assert abs(m["loss"] - g["loss"]) < 1e-5 * g["loss"]
    assert m["K_count"] == g["K_count"]
    assert relerr(m["grad"], g["grad"]) < 2e-5


def test_diffusion_allen_cahn_port_and_manual():
    g = load_golden("diff_allencahn_d20")
    d, arch = int(g["d"]), [int(a) for a in g["arch"]]
    dims = [d + 1] + arch + [1]
    params, off = [], 0
    for i in range(len(dims) - 1):
        for s in ((sum(dims[:i + 1]), dims[i + 1]), (dims[i + 1],)):
            n = int(np.prod(s))
            params.append(pt.tensor(g["theta"][off:off + n].reshape(s)))
            off += n
    alpha, T = tuple(float(a) for a in g["alpha"]), float(g["T"])
    prob = orc.make_problem("allencahn", d, boundary_distance=7.0)
    o = orc.diffusion_iteration(prob, params, pt.tensor(g["X0"]), pt.tensor(g["t0"]), pt.tensor(g["xis"]),
                                g["delta_t"], int(g["N"]), int(g["K_boundary"]), alpha)
    assert abs(float(o["loss"]) - g["loss"]) < 1e-6 * g["loss"]
    assert o["K_count"] == g["K_count"]
    assert relerr(np.concatenate([q.reshape(-1).numpy() for q in o["grads"]]), g["grad"]) < 1e-6
    net = man.Net("densenet", dims, g["theta"])
    m = man.diffusion(man.Problem("heat", d), net, g["X0"].astype(np.float64), g["t0"].astype(np.float64),
                      g["xis"].astype(np.float64), g["delta_t"], int(g["N"]), int(g["K_boundary"]), alpha, T=T,
                      pde=man.ALLEN_CAHN)
    assert abs(m["loss"] - g["loss"]) < 1e-5 * g["loss"]
    assert m["K_count"] == g["K_count"]
    assert relerr(m["grad"], g["grad"]) < 2e-5


def test_diffusion_c4_shape_seeded():
    """C4 / G4 shape (d=50, DenseNet[256,256]); inputs regenerated from the seed (same torch build on every box)."""
    g = load_golden("diff_heat_d50_w256")
    d, K, N = g["d"], g["K"], g["N"]
    params = orc.densenet_init(d + 1, 1, list(g["arch"]), seed=g["seed"])
    pt.manual_seed(g["seed"])
    X0 = orc.sample_ball(K, d, 1.0)
    t0 = pt.rand(K, 1) * 1.0
    xis = pt.stack([pt.randn(K, d) for _ in range(N)])
    o = orc.diffusion_iteration(orc.make_problem("heat", d, T=1), params, X0, t0, xis, g["delta_t"], N,
                                g["K_boundary"])
    assert abs(float(o["loss"]) - g["loss"]) < 1e-6 * g["loss"]
    assert o["K_count"] == g["K_count"]
    flat = np.concatenate([q.reshape(-1).numpy() for q in o["grads"]])
    assert relerr(flat[g["grad_sample_idx"]], g["grad_sample"]) < 1e-6


@pytest.mark.parametrize("tag", ["is_llgc_d10_dense", "is_dwm_d4_mlp"])
def test_importance_sampling_port(tag):
    g = load_golden(tag)
    d = g["d"]
    g["time_approx"] = "inner"
    params, _ = split_theta(g)
    prob = orc.make_problem(g["kind"], d, **g["pkw"])
    N_solver = int(np.floor(g["T"] / g["solver_dt"]))
    m, v, r = orc.importance_sampling(prob, g["net"], params, pt.tensor(g["xis"]), g["is_dt"], g["solver_dt"],
                                      N_solver=N_solver)
    assert abs(m - g["mean"]) < 1e-5 * abs(g["mean"])
    assert abs(v - g["var"]) < 1e-4 * abs(g["var"])


@pytest.mark.parametrize("tag", ["is_llgc_d10_dense", "is_dwm_d4_mlp"])
def test_manual_rollout_on_network_grid(tag):
    """man.rollout with the network evaluated at t_index[n] dt_net (t_index[n] = ceil(n dt / dt_net), the fp32 division of
    Solver.Z_n) reproduces the reference's importance-sampling mean and variance, w = exp(Y_N - 2 Fint - g(X_N))."""
    g = load_golden(tag)
    d, dt, dt_net = g["d"], g["is_dt"], g["solver_dt"]
    g["time_approx"] = "inner"
    dims = net_dims(g)
    p32 = orc.make_problem(g["kind"], d, **g["pkw"])
    if g["kind"] == "dwm":
        prob = man.Problem("dwm", d, eta_=p32.eta_.numpy(), kappa_=p32.kappa_.numpy())
    else:
        prob = man.Problem(g["kind"], d, A=p32.A.numpy(), B=p32.B.numpy())
    N, K = g["xis"].shape[:2]
    xi = np.zeros((K, d, N + 1))
    xi[:, :, 1:] = g["xis"].transpose(1, 2, 0)
    t_index = [int(np.ceil(np.float32(n * dt) / np.float32(dt_net))) for n in range(N)]
    assert t_index != list(range(N))                  # a coarser (llgc) or finer (dwm) network grid: the remap matters
    ro = man.rollout(prob, man.Net(g["net"], dims, g["theta"]), xi, dt, N, p32.X_0.numpy(), True, 0.0, "first",
                     t_index, dt_net)
    w = np.exp(ro["Y"] - 2 * ro["Fint"] - ro["gX"])
    assert abs(w.mean() - g["mean"]) < 1e-5 * abs(g["mean"])
    assert abs(w.var(ddof=1) - g["var"]) < 1e-4 * abs(g["var"])


@pytest.mark.parametrize("tag", ["hjb_lqgc_d10_dense_lv", "hjb_lqgc_d10_outer_lv"])
def test_manual_extensions_reduce_to_the_pinned_oracle(tag):
    """The per-path X_0 and network-time arguments of man.rollout / man.grad_mode_a: a tiled X_0 and t_index = arange(N)
    with dt_net = dt give the one-row, step-grid result bit for bit."""
    g = load_golden(tag)
    d, N, dt = g["d"], g["N"], g["delta_t"]
    outer = g["time_approx"] == "outer"
    per = g["theta"].size // (N if outer else 1)
    nets = [man.Net(g["net"], net_dims(g), g["theta"][i * per:(i + 1) * per]) for i in range(N if outer else 1)]
    nets = nets if outer else nets[0]
    prob, tm = man.Problem(g["kind"], d, A=g["A"], B=g["B"]), "none" if outer else "first"
    xi = g["xi"].astype(np.float64)
    K = xi.shape[0]
    X0 = 0.1 * np.arange(d)
    wY, wZ = np.linspace(-1, 1, K) / K, np.linspace(0, 1, K) / K
    ref = man.grad_mode_a(prob, nets, xi, dt, N, X0, wY, wZ, g["adaptive"], tm, 0.5)
    for kw in (dict(X0=np.tile(X0, (K, 1))), dict(t_index=np.arange(N), dt_net=dt)):
        args = dict(X0=X0, t_index=None, dt_net=None)
        args.update(kw)
        got = man.grad_mode_a(prob, nets, xi, dt, N, args["X0"], wY, wZ, g["adaptive"], tm, 0.5, args["t_index"],
                              args["dt_net"])
        assert np.array_equal(got[0], ref[0])
        for k in ("X", "Y", "Zsum", "Fint", "gX"):
            assert np.array_equal(got[1][k], ref[1][k]), k


LOOPS = {
    "loop_G1": dict(kind="lqgc", d=10, pkw={}, net="densenet", ta="outer", K=200, dt=0.05, L=3, lr=1e-3,
                    loss="log-variance", detach=True),
    "loop_G1b": dict(kind="lqgc", d=10, pkw={}, net="densenet", ta="inner", K=200, dt=0.05, L=3, lr=1e-3,
                     loss="log-variance", detach=True),
    "loop_G3a": dict(kind="dwm", d=50, pkw=dict(d_1=15, d_2=35, T=1, eta=3, kappa=5), net="mlp_tanh", ta="inner",
                     K=256, dt=0.005, L=2, lr=0.05, loss="log-variance", detach=True),
    "loop_G3b": dict(kind="dwm", d=50, pkw=dict(d_1=15, d_2=35, T=1, eta=3, kappa=5), net="mlp_tanh", ta="inner",
                     K=256, dt=0.005, L=2, lr=0.05, loss="relative_entropy", detach=False),
}


@pytest.mark.parametrize("tag", sorted(LOOPS))
def test_training_loop_pins(tag):
    """Whole-loop pins (SURVEY.md Appendix B): torch CPU RNG + rollout + Adam reproduce the reference loss_log."""
    c = LOOPS[tag]
    g = load_golden(tag)
    prob = orc.make_problem(c["kind"], c["d"], **c["pkw"])
    N = int(np.floor(prob.T / c["dt"]))
    if c["net"] == "mlp_tanh":
        params = orc.mlp_init(c["d"] + 1, c["d"], seed=123)
    elif c["ta"] == "outer":
        params = [orc.densenet_init(c["d"], c["d"], seed=42) for _ in range(N)]
    else:
        params = orc.densenet_init(c["d"] + 1, c["d"], seed=42)
    ll = orc.hjb_train_loop(prob, c["net"], params, c["K"], c["dt"], c["L"], c["lr"], c["loss"], c["ta"],
                            True, c["detach"], seed=42)
    np.testing.assert_allclose(ll, g["loss_log"], rtol=2e-6)


def test_analytic_llgc_value():
    """V(0,0) = -(d/4)(1 - exp(-2T)) for A=-I, B=I, alpha=1 (BASELINE.md section 4): the optimal control
    u* = -exp(-(T-t)) makes D = Y_N - g(X_N) path-wise constant = -V(0,0) in the continuous limit."""
    d, T, dt = 10, 1.0, 0.001
    N = int(T / dt)
    rng = np.random.default_rng(0)
    xi = rng.standard_normal((64, d, N + 1))
    X = np.zeros((64, d))
    Y = np.zeros(64)
    for n in range(N):
        Z = np.exp(-(T - n * dt)) * np.ones((64, d))          # Z = -u*
        X = X + (-X - Z) * dt + xi[:, :, n + 1] * np.sqrt(dt)
        Y = Y + (-0.5 * (Z ** 2).sum(1)) * dt + (Z * xi[:, :, n + 1]).sum(1) * np.sqrt(dt)
    D = Y - X.sum(1)
    V00 = -(d / 4) * (1 - np.exp(-2 * T))
    assert abs(D.mean() - (-V00)) < 5e-3 * abs(V00)
    assert D.std() < 2e-2 * abs(V00)


# ---------------------------------------------------------------------------------------------- elliptic (row f4)
ELL_TAGS = ["ell_expsin_d10", "ell_expball_d5", "ell_expsphere_d4", "ell_helmholtz_d2", "ell_committor_d10"]


def ell_params(g):
    d, arch = int(g["d"]), [int(a) for a in g["arch"]]
    dims = [d] + arch + [1]
    params, off = [], 0
    for i in range(len(dims) - 1):
        for s in ((sum(dims[:i + 1]), dims[i + 1]), (dims[i + 1],)):
            n = int(np.prod(s))
            params.append(pt.tensor(g["theta"][off:off + n].reshape(s)))
            off += n
    return dims, params


@pytest.mark.parametrize("tag", ELL_TAGS)
def test_elliptic_port_and_manual(tag):
    """EllipticSolver iteration (solver.py:646-670, :687-790): the PyTorch-CPU restatement and the explicit fp64
    gradient formulas against the golden vectors generated from the reference."""
    g = load_golden(tag)
    d, kind = int(g["d"]), str(g["kind"])
    dims, params = ell_params(g)
    alpha = tuple(float(a) for a in g["alpha"])
    o = orc.elliptic_iteration(orc.make_problem(kind, d), params, pt.tensor(g["Xb"]), pt.tensor(g["X0"]),
                               pt.tensor(g["xis"]), g["delta_t"], int(g["N"]), alpha)
    assert abs(float(o["loss"]) - g["loss"]) < 1e-6 * g["loss"]
    assert o["K_count"] == g["K_count"]
    assert abs(float(o["V_L2"].mean()) - g["V_L2"]) < 1e-6 * g["V_L2"]
    assert relerr(np.concatenate([q.reshape(-1).numpy() for q in o["grads"]]), g["grad"]) < 2e-6
    assert 0 < int(o["stopped"].sum())                       # the exit logic is exercised
    net = man.Net("densenet", dims, g["theta"])
    gb = orc.make_problem(kind, d).g(pt.tensor(g["Xb"])).numpy().astype(np.float64)   # fp32 like the reference (committor: indicator)
    m = man.elliptic(man.EllipticProblem(kind, d), net, g["Xb"].astype(np.float64), g["X0"].astype(np.float64),
                     g["xis"].astype(np.float64), g["delta_t"], int(g["N"]), alpha, gb=gb)
    assert m["K_count"] == g["K_count"]
    assert abs(m["loss"] - g["loss"]) < 1e-5 * g["loss"]
    assert abs(m["V_L2"].mean() - g["V_L2"]) < 1e-5 * g["V_L2"]
    assert relerr(m["grad"], g["grad"]) < 2e-5
    assert relerr(m["X"], g["X_end"]) < 1e-6 and relerr(m["Y"], g["Y_end"]) < 1e-5


@pytest.mark.parametrize("tag,kind,d,N", [("loop_G5", "expball_sin", 50, 20), ("loop_G5b", "helmholtz", 2, 20),
                                          ("loop_G7", "committor", 10, 50)])
def test_elliptic_training_loop_pins(tag, kind, d, N):
    """Whole-loop pins: torch + numpy RNG order, rollout and Adam reproduce the reference's loss_log and K_log."""
    g = load_golden(tag)
    params = orc.densenet_init(d, 1, seed=42)
    ll, kc = orc.elliptic_train_loop(orc.make_problem(kind, d), params, 200, 50, N, 1e-3, 3, 1e-3, seed=42)
    np.testing.assert_allclose(ll, g["loss_log"], rtol=2e-6)
    assert kc == [int(v) for v in g["K_log"]]
