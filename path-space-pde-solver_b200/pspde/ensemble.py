"""SolverEnsemble: M independent ``Solver`` runs of one problem and one network geometry -- seeds, learning rates, initial
weights, L -- trained together, each phase of an iteration one launch for all members (include/pspde.h, "Ensembles").

The reference's notebooks train on a few hundred paths (K = 50 .. 256: one to four 64-path tiles, a few CTAs on a
148-SM B200); one iteration leaves almost all SMs idle and is latency bound.  Seeds, learning-rate and loss comparisons
and d sweeps are many such runs; the ensemble puts them on the idle SMs.  Member m computes what the same Solver computes
alone on the FP32-FMA kernels (PSPDE_FWD_PATH=simt PSPDE_BWD_PATH=simt): logs, parameters and Adam state bit for bit while
M * ceil(K / 64) <= #SMs.

    ens = pspde.SolverEnsemble([pspde.Solver('s%d' % s, problem, seed=s, K=200, L=500, detach_forward=True, ...)
                                for s in range(40)])
    ens.train()                     # every member's loss_log, u_L2_loss, ... as if trained alone

The members' parameters live in one [M][p] buffer (their module parameters, ``_theta`` and ``.grad`` are views of their
slice) and their flat Adam state in [M][p] buffers the same way, so ``member.z_n(x)``, ``member.Z_n``, ``save_networks``
and ``do_importance_sampling_me(problem, member, K)`` work on a member alone between or after iterations.
"""
import ctypes
import time

import numpy as np
import torch as pt

from . import _lib as L
from . import losses

# what every member must share (the kernels run one configuration)
_SHARED = ('K', 'delta_t_np', 'N', 'time_approx', 'loss_method', 'adaptive_forward_process', 'detach_forward', 'learn_Y_0',
           'u_l2_error_flag', 'blowup_bound', 'random_X_0', 'device')


def _pad(n, q=128):
    return (n + q - 1) // q * q


class SolverEnsemble:

    def __init__(self, solvers, verbose=True):
        self.members = list(solvers)
        self.verbose = verbose
        if not self.members:
            raise ValueError("an ensemble needs at least one Solver")
        s0 = self.members[0]
        for s in self.members:
            if s.noise != 'philox':
                raise NotImplementedError("ensembles draw their noise in the kernel: noise='philox' only")
            if s.process_group is not None:
                raise NotImplementedError("ensembles run on one GPU: process_group=None only")
            if (not s.detach_forward) and s.adaptive_forward_process:
                raise NotImplementedError("the attached forward process (detach_forward=False, adaptive) is not batched")
            if s.IS_variance_K > 0:
                raise NotImplementedError("IS_variance_K > 0 is not supported in an ensemble")
            if s.log_gradient or s.burgers_drift or s.compute_gradient_variance:
                raise NotImplementedError("log_gradient / burgers_drift / compute_gradient_variance are not supported")
            if s.loss_method not in losses.SUPPORTED:
                raise NotImplementedError("loss_method=%r is off the fused hot path" % s.loss_method)
            for a in _SHARED:
                if getattr(s, a) != getattr(s0, a):
                    raise ValueError("ensemble members must agree on %s (%r != %r)" % (a, getattr(s, a), getattr(s0, a)))
            if (s._net_id, s._dims) != (s0._net_id, s0._dims):
                raise ValueError("ensemble members must share the network spec")
        self._check_problems()
        self.M, self.K, self.N, self.d = len(self.members), s0.K, s0.N, s0.d
        self.lib = L.load()
        self.device = s0.device
        eng = s0._get_engine()                  # problem pack, fp32 dt, u_L2 table (validated like the member alone)
        self._eng0 = eng
        self._u_l2_on = s0._u_l2_on
        self.done = [False] * self.M
        self._homed = None
        f32 = dict(dtype=pt.float32, device=self.device)
        M, K, d = self.M, self.K, self.d
        self.Y_N, self.gX, self.Zsum, self.uL2 = (pt.zeros(M, K, **f32) for _ in range(4))
        self.X_N = pt.empty(M, K, d, **f32)
        self.stats = pt.zeros(M, 4, dtype=pt.float64, device=self.device)
        self.wY = pt.zeros(M, K, **f32)
        self.lv_out = pt.zeros(M, 3, dtype=pt.float64, device=self.device)
        self.seeds = pt.tensor(np.array([s.seed & (2 ** 64 - 1) for s in self.members], np.uint64).view(np.int64),
                               device=self.device)
        if s0.random_X_0:
            self.x0, self.x0_stride = pt.empty(M, K, d, **f32), K * d
        else:
            self.x0 = pt.stack([s.problem.X_0.detach().to(self.device, pt.float32).reshape(d) for s in self.members])
            self.x0_stride = d
        # rows padded to 512 bytes: the per-member sums below then see the alignment of a standalone buffer
        self._red = pt.zeros(M, _pad(K), dtype=pt.float64, device=self.device)
        self._red32 = pt.zeros(M, _pad(K), **f32)
        self._adam_table = pt.empty(M * ctypes.sizeof(L.pspde_adam_member), dtype=pt.uint8, device=self.device)
        self._adam_host = pt.empty(self._adam_table.numel(), dtype=pt.uint8, pin_memory=True)
        self.udiag = None
        if self._u_l2_on:
            u = L.pspde_udiag()
            src = eng.udiag
            u.mode, u.nx1, u.d1, u.xb, u.dx = src.mode, src.nx1, src.d1, src.xb, src.dx
            u.table, u.uL2, u.quirk_path = eng._utab.data_ptr(), self.uL2.data_ptr(), src.quirk_path
            self.udiag = u
        self.ens = L.pspde_ensemble(n_models=M, seeds=self.seeds.data_ptr(), theta_stride=0, x0_stride=self.x0_stride)
        self._home()
        nbytes = int(self.lib.pspde_ensemble_workspace_bytes(ctypes.byref(self.cfg(0)), ctypes.byref(self.ens)))
        if nbytes == 0:
            raise RuntimeError("libpspde: %s" % self.lib.pspde_last_error().decode())
        self.workspace = pt.empty(nbytes, dtype=pt.uint8, device=self.device)

    def _check_problems(self):
        """The members' problems must give the kernels the same functor pack and u_L2 table."""
        s0 = self.members[0]
        pid, flags, pack = s0.problem.functor_pack()
        tab0 = s0.problem.u_true_table(s0.N, s0.delta_t_np) if hasattr(s0.problem, 'u_true_table') else None
        for s in self.members[1:]:
            if s.problem is s0.problem:
                continue
            p2, f2, k2 = s.problem.functor_pack()
            if (p2, f2) != (pid, flags) or not pt.equal(k2.cpu(), pack.cpu()):
                raise ValueError("ensemble members must share the problem's functor pack")
            if s0.u_l2_error_flag:
                tab = s.problem.u_true_table(s.N, s.delta_t_np) if hasattr(s.problem, 'u_true_table') else None
                same = (tab is None) == (tab0 is None) and (tab is None or (
                    {k: v for k, v in tab.items() if k != 'table'} == {k: v for k, v in tab0.items() if k != 'table'}
                    and pt.equal(tab['table'].cpu(), tab0['table'].cpu())))
                if not same:
                    raise ValueError("ensemble members must share the problem's u_L2 table")

    # ------------------------------------------------------------------ parameters
    def _home(self):
        """Re-home every member's parameters in one [M][p] buffer and its flat Adam state in [M][p] buffers (the
        GeneralSolver._home_parameters pattern, one slice per member); y_0 of all members in one [M] buffer."""
        M, dev = self.M, self.device
        for s in self.members:
            s.update_Phis()                      # collects the current modules into the member's own flat buffer
        p = self.members[0]._theta.numel()
        self.p = p
        self.theta = pt.empty(M, p, dtype=pt.float32, device=dev)
        self.grad = pt.zeros(M, p, dtype=pt.float32, device=dev)
        self._grad_scratch = None
        self.exp_avg, self.exp_avg_sq = pt.zeros(M, p, dtype=pt.float32, device=dev), pt.zeros(M, p, dtype=pt.float32, device=dev)
        self.y0 = pt.zeros(M, dtype=pt.float32, device=dev)
        self._fa = []
        for m, s in enumerate(self.members):
            self.theta[m].copy_(s._theta.detach())
            th, g = self.theta[m], self.grad[m]
            off = 0
            for q in s._params:
                k = q.numel()
                q.data = th[off:off + k].view(q.shape)
                q.grad = g[off:off + k].view(q.shape)
                off += k
            s._theta = th.requires_grad_(True)
            s._theta.grad = g
            fa = s._flat_adam_state()
            if fa:
                self.exp_avg[m].copy_(fa['exp_avg'])
                self.exp_avg_sq[m].copy_(fa['exp_avg_sq'])
                off = 0
                for net in fa['nets']:
                    for q in net.parameters():
                        k, st = q.numel(), net.optim.state[q]
                        st['exp_avg'] = self.exp_avg[m, off:off + k].view(q.shape)
                        st['exp_avg_sq'] = self.exp_avg_sq[m, off:off + k].view(q.shape)
                        off += k
                fa['exp_avg'], fa['exp_avg_sq'] = self.exp_avg[m], self.exp_avg_sq[m]
            self._fa.append(fa)
            if s.learn_Y_0:
                self.y0[m:m + 1].copy_(s.y_0.Y_0.data.reshape(1))
                s.y_0.Y_0.data = self.y0[m:m + 1].view(s.y_0.Y_0.shape)
        self.ens.theta_stride = p
        self._homed = [(s._theta, [id(n) for n in s._nets()]) for s in self.members]

    def _check_homed(self):
        """Re-home when a member's parameters stopped being views of its slice (update_Phis, a replaced network or
        optimizer, a re-assigned y_0)."""
        for m, s in enumerate(self.members):
            th, nets = self._homed[m]
            if (s._theta is not th or [id(n) for n in s._nets()] != nets or s._flat_adam_state() is not self._fa[m]
                    or (s.learn_Y_0 and s.y_0.Y_0.data_ptr() != self.y0[m:m + 1].data_ptr())):
                self._home()
                return

    # ------------------------------------------------------------------ library calls
    def cfg(self, offset):
        e = self._eng0
        return L.make_cfg(self.K, self.d, self.N, e.dt, e.problem_id, e.net_id, e.dims, e.time_mode, adaptive=e.adaptive,
                          problem_flags=e.flags, noise_mode=L.NOISE_PHILOX, offset=offset,
                          x0_per_path=self.members[0].random_X_0, d_abs_max=e.blowup_bound)

    def _stream(self):
        return ctypes.c_void_p(pt.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _p(t):
        return None if t is None else ctypes.c_void_p(t.data_ptr())

    def _forward(self, cfg):
        y0 = self.y0 if self.members[0].learn_Y_0 else None
        rc = self.lib.pspde_ensemble_fwd(ctypes.byref(cfg), ctypes.byref(self.ens), self._p(self.theta), self._p(self._eng0.pack),
                                         self._p(self.x0), self._p(y0), self._p(self.X_N), self._p(self.Y_N), self._p(self.gX),
                                         self._p(self.Zsum), self._p(self.stats),
                                         None if self.udiag is None else ctypes.byref(self.udiag),
                                         self._p(self.workspace), self.workspace.numel(), self._stream())
        L.check(self.lib, rc)

    def _backward(self, cfg, wY, wZ, out):
        rc = self.lib.pspde_ensemble_bwd_detached(ctypes.byref(cfg), ctypes.byref(self.ens), self._p(self.theta),
                                                  self._p(self._eng0.pack), self._p(self.x0), self._p(wY), self._p(wZ),
                                                  self._p(out), self._p(self.workspace), self.workspace.numel(), self._stream())
        L.check(self.lib, rc)

    def _row_sums(self, x, buf):
        """Per-member sums of x [M][K], each over a 512-byte aligned row like a standalone run's buffer (same reduction)."""
        buf[:, :self.K].copy_(x)
        return [buf[m, :self.K].sum() for m in range(self.M)]

    # ------------------------------------------------------------------ one iteration
    def _draw_x0(self, l):
        for m, s in enumerate(self.members):       # exactly Solver.initialize_training_data's draw (k_lo = 0)
            gen = pt.Generator(device=self.device)
            gen.manual_seed((s.seed * 1000003 + l * 8191) % (2 ** 63))
            self.x0[m].copy_(pt.randn(self.K, self.d, device=self.device, generator=gen))

    def _adam(self, active):
        """Solver.optimization_step for every active member: the flat Adam of all members whose network optimizers are
        plain Adam with one setting and one step count in one launch, the other optimizers stepped one by one."""
        table = (L.pspde_adam_member * self.M)()
        rest = []
        for m in active:
            s, fa = self.members[m], self._fa[m]
            todo = s.Phis
            if fa:
                hyper = {s._adam_hyper(n.optim) for n in fa['nets']}
                steps = fa['step']
                if len(hyper) == 1 and None not in hyper and bool((steps == steps[0]).all()):
                    lr, beta1, beta2, eps = next(iter(hyper))
                    steps += 1
                    L.check(self.lib, self.lib.pspde_adam_member_make(lr, beta1, beta2, eps, int(float(steps[0])),
                                                                       ctypes.byref(table[m])))
                    todo = [phi for phi in s.Phis if all(phi is not n for n in fa['nets'])]
            rest += todo
        if any(table[m].step for m in active):
            # pinned staging: the previous iteration's copy has completed at its host sync
            self._adam_host.numpy()[:] = np.frombuffer(bytes(table), np.uint8)
            self._adam_table.copy_(self._adam_host, non_blocking=True)
            with pt.cuda.device(self.device):
                L.check(self.lib, self.lib.pspde_ensemble_adam(self.M, self.p, self.p, self._p(self.theta.data),
                                                               self._p(self.grad), self._p(self.exp_avg),
                                                               self._p(self.exp_avg_sq), self._p(self._adam_table),
                                                               self._stream()))
        for phi in rest:
            phi.optim.step()

    def train_step(self, l):
        """One iteration for every member that is not done and has l < its L: rollout, loss, backward and Adam, one
        launch per phase for all members; appends to each such member's logs what Solver.train_step appends."""
        t_0 = time.time()
        active = [m for m, s in enumerate(self.members) if not self.done[m] and l < s.L]
        if not active:
            return None
        self._check_homed()
        M, K = self.M, self.K
        s0 = self.members[0]
        with pt.cuda.device(self.device):
            for m in active:
                self.members[m]._iteration = l
            if s0.random_X_0:
                self._draw_x0(l)
            y0_before = self.y0.clone()
            cfg = self.cfg(l)
            all_active = len(active) == M
            if not all_active and self._grad_scratch is None:
                self._grad_scratch = pt.zeros_like(self.grad)
            gout = self.grad if all_active else self._grad_scratch
            for m in active:
                self.members[m]._ensure_grad_views()
            self._forward(cfg)
            if s0.loss_method in ('log-variance', 'moment'):
                L.check(self.lib, self.lib.pspde_ensemble_lv_cotangents(M, K, float(K), 1 if s0.loss_method == 'moment' else 0,
                                                                         self._p(self.Y_N), self._p(self.gX), self._p(self.stats),
                                                                         self._p(self.wY), self._p(self.lv_out), self._stream()))
                wY, wZ = self.wY, None
                loss, n_bad = self.lv_out[:, 0], self.lv_out[:, 1]
            else:
                # per-member cotangents with the host formulation on the member's slice, then one backward launch
                lv, nb = [], []
                wZ = None
                for m in range(M):
                    lo, w_y, w_z, _, n_b = losses.value_and_cotangents(s0.loss_method, self.Y_N[m], self.gX[m], self.Zsum[m],
                                                                       K, s0.adaptive_forward_process, None,
                                                                       stats=self.stats[m])
                    self.wY[m].copy_(w_y if w_y is not None else pt.zeros_like(self.wY[m]))
                    if w_z is not None:
                        if wZ is None:
                            wZ = pt.zeros_like(self.wY)
                        wZ[m].copy_(w_z)
                    lv.append(lo.double().reshape(()))
                    nb.append(n_b.double().reshape(()))
                wY = self.wY
                loss, n_bad = pt.stack(lv), pt.stack(nb)
            self._backward(cfg, wY, wZ, gout)
            if not all_active:
                idx = pt.tensor(active, device=self.device)
                self.grad.index_copy_(0, idx, gout.index_select(0, idx))
            if s0.learn_Y_0:
                sums = self._row_sums(wY, self._red32)
                for m in active:
                    self.members[m].y_0.Y_0.grad = sums[m].reshape(1)
            self._adam(active)
            u_l2 = pt.full((M,), float('nan'), dtype=pt.float64, device=self.device)
            if self._u_l2_on:
                u = self.uL2.double()
                kept = pt.isfinite(u) & pt.isfinite(self.Y_N)
                u_l2 = pt.stack(self._row_sums(pt.where(kept, u, pt.zeros_like(u)), self._red)) / K
            cols = [loss.double(), n_bad.double(), u_l2, y0_before.double()]
            if s0.metastability_logs is not None:
                target, epsilon = s0.metastability_logs
                cols.append(pt.stack([(pt.sqrt(pt.sum((self.X_N[m] - target) ** 2, 1)) < epsilon).float().sum().double()
                                      for m in range(M)]) / K)
            res = pt.stack(cols, 1).tolist()             # the only host sync of the iteration, for all members
        t_1 = time.time()
        for m in active:
            s, r = self.members[m], res[m]
            if s.learn_Y_0:
                s.Y_0_log.append(r[3])
            s.loss_log.append(r[0])
            s.nonfinite_log.append(int(r[1]))
            s.u_L2_loss.append(r[2])
            if s.metastability_logs is not None:
                s.particles_close_to_target.append(r[4])
            s.times.append(t_1 - t_0)
            s.path_steps_per_sec.append(s.K * s.N / max(t_1 - t_0, 1e-12))
            if l + 1 >= s.L:
                self.done[m] = True
            elif s.early_stopping_time is not None and l > s.early_stopping_time:
                if np.std(s.u_L2_loss[-s.early_stopping_time:]) / s.u_L2_loss[-1] < 0.02:
                    self.done[m] = True
        return [self.members[m].loss_log[-1] for m in active]

    def train(self):
        """Iterate until every member reached its L or its early-stopping rule fired; then save the logs of the members
        with save_results."""
        s0 = self.members[0]
        if self.verbose:
            print('ensemble of %d: d = %d, K = %d, delta_t = %.2e, %s, %s, %s'
                  % (self.M, self.d, self.K, s0.delta_t_np, s0.time_approx, s0.loss_method,
                     'adaptive' if s0.adaptive_forward_process else ''))
        l = 0
        while not all(self.done[m] or l >= s.L for m, s in enumerate(self.members)):
            out = self.train_step(l)
            if self.verbose and out and l % s0.print_every == 0:
                print('%d - %d active - loss min %.4e max %.4e - time/iter: %.2fs'
                      % (l, len(out), min(out), max(out), np.mean(s0.times[-s0.print_every:]) if s0.times else 0.0))
            l += 1
        for s in self.members:
            if s.save_results is True:
                s.save_logs()
