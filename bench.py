#!/usr/bin/env python
"""bench.py -- path-steps/sec per training iteration of the fused path-space rollout (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c1|c3|c3re|c4|c5]
                    [--dump-outputs DIR]

Workload (default): BASELINE.json configs[4], the configuration north_star's target is quoted on -- the large-batch
sweep, LLGC(d=100, off_diag=0, T=1), DenseNet(101 -> 30 -> 30 -> 100) 'inner', K = 2^20 trajectories per GPU,
delta_t = 0.005 (N = 200 steps), log-variance loss, detach_forward=True.  One "step" = one full training iteration:
in-kernel Philox noise, forward rollout, loss statistics, all-reduce of the statistics (N > 1), backward (checkpoint
rollout + gradient kernel), all-reduce of the gradient (N > 1), Adam.  Weak scaling: K per GPU is fixed, K_global =
N * 2^20.  The same line carries, as secondary blocks measured in the same process:
  "c2"        configs[1] (K = 2^16 per GPU, N = 100): ms per iteration, path-steps/s, kernel times
  "strong"    (N > 1) K_global = 2^20 fixed, sharded over the N ranks
  "accuracy"  the second half of the metric: configs[1] trained for a fixed budget, V(0,0) against the analytic
              -21.6166, rel. L2 error of V(.,0) over test points and of the control against u*(x,t) = -exp(-(T-t))
  "sharding_check"  per-path Y_N of 1024 global paths spread over all ranks, recomputed on rank 0 as one shard

Arms
  ours        the CUDA path through pspde.Solver (fails without a GPU: there is no CPU fallback)
  reference   the reference's CPU algorithm (oracle/ref_port.py: PyTorch eager + autograd + CPU randn, the exact
              procedure of solver.py:420-531) on the host cores, on a bounded sample of the same workload

--dump-outputs DIR (ours) writes what the last timed step computed as DIR/<name>.npy: loss (float64), the parameters
theta after the step's Adam update and their gradient grad (float32), and rank 0's per-path outputs (float32; Y_N, gX,
X_N, or V0, VE, Y, X_end, t_end for c4) on a fixed, seeded sample of at most 2^16 paths whose indices are path_index
(float64).  Inputs are seeded, so the same arguments give the same inputs on every run and build.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "path-space-pde-solver_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True  # the bench writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402
import torch as pt  # noqa: E402

METRIC = "path-steps/sec per train iter"
UNIT = "path-steps/s"
CPU_SAMPLE_K = 1 << 14          # SURVEY.md section 8(d): K_cpu = min(K, 2^14)
DUMP_PATHS = 1 << 16            # --dump-outputs: per-path outputs of at most this many paths (seeded sample)
DUMP_MAX_BYTES = 64 << 20

WORKLOADS = {
    # name: (problem kind, ctor kwargs, net, time_approx, K per GPU, delta_t, loss, detach, lr)
    "c2": dict(kind="llgc", pkw=dict(d=100, off_diag=0, T=1, seed=42), net="densenet", ta="inner", K=1 << 16,
               dt=0.01, loss="log-variance", detach=True, lr=1e-3,
               desc="C2: LLGC d=100 off_diag=0 T=1, DenseNet[101,30,30,100] inner, K=2^16/GPU, N=100, log-variance"),
    "c5": dict(kind="llgc", pkw=dict(d=100, off_diag=0, T=1, seed=42), net="densenet", ta="inner", K=1 << 20,
               dt=0.005, loss="log-variance", detach=True, lr=1e-3,
               desc="C5: LLGC d=100, DenseNet inner, K=2^20/GPU, N=200, log-variance"),
    # the rest of BASELINE configs[4]'s sweep K = 2^20 .. 2^24: 2^22 on one GPU; 2^21 per GPU = 2^24 over 8 GPUs
    "c5_k22": dict(kind="llgc", pkw=dict(d=100, off_diag=0, T=1, seed=42), net="densenet", ta="inner", K=1 << 22,
                   dt=0.005, loss="log-variance", detach=True, lr=1e-3,
                   desc="C5 sweep: LLGC d=100, DenseNet inner, K=2^22/GPU, N=200, log-variance"),
    "c5_k21": dict(kind="llgc", pkw=dict(d=100, off_diag=0, T=1, seed=42), net="densenet", ta="inner", K=1 << 21,
                   dt=0.005, loss="log-variance", detach=True, lr=1e-3,
                   desc="C5 sweep: LLGC d=100, DenseNet inner, K=2^21/GPU (2^24 over 8 GPUs), N=200, log-variance"),
    "c1": dict(kind="lqgc", pkw=dict(d=10), net="densenet", ta="outer", K=200, dt=0.05, loss="log-variance",
               detach=True, lr=1e-3, desc="C1: LQGC d=10, 100 x DenseNet[10,30,30,10] outer, K=200, N=100"),
    "c3": dict(kind="dwm", pkw=dict(d=50, d_1=15, d_2=35, T=1, eta=3, kappa=5), net="mlp", ta="inner", K=1 << 18,
               dt=0.005, loss="log-variance", detach=True, lr=0.05,
               desc="C3: DoubleWell_multidim d=50, MySequential, K=2^18/GPU, N=200, log-variance"),
    "c3re": dict(kind="dwm", pkw=dict(d=50, d_1=15, d_2=35, T=1, eta=3, kappa=5), net="mlp", ta="inner", K=1 << 18,
                 dt=0.005, loss="relative_entropy", detach=False, lr=0.05,
                 desc="C3: DoubleWell_multidim d=50, MySequential, K=2^18/GPU, N=200, relative entropy (attached)"),
    "c4": dict(kind="heat", pkw=dict(d=50, T=1), net="densenet", arch=[256, 256], K=1 << 18, K_boundary=50, N=25,
               dt=1e-3, loss="diffusion", lr=1e-3,
               desc="C4: HeatEquation d=50, GeneralSolver diffusion loss, DenseNet[51,256,256,1], K=2^18/GPU, N=25"),
}


def net_macs(dims, dense):
    """forward MACs M, hidden-cotangent MACs M_delta (SURVEY.md section 8d)."""
    L = len(dims) - 1
    if dense:
        M = sum(sum(dims[:i + 1]) * dims[i + 1] for i in range(L))
        Md = sum(sum(dims[1:i + 1]) * dims[i + 1] for i in range(1, L))
    else:
        M = sum(dims[i] * dims[i + 1] for i in range(L))
        Md = sum(dims[i] * dims[i + 1] for i in range(1, L))
    return M, Md


# ----------------------------------------------------------------------------------------------- reference arm
def run_reference(args, wl):
    """The reference's CPU procedure (torch eager, CPU randn, autograd, Adam) on a bounded sample."""
    from oracle import ref_port as orc
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    pt.set_num_threads(cores)
    d = wl["pkw"]["d"]
    kind = wl["kind"]
    pkw = {k: v for k, v in wl["pkw"].items() if k != "d"}
    prob = orc.make_problem(kind, d, **pkw)
    if kind == "heat":
        N, K_cpu = wl["N"], min(wl["K"], 2048)
        params = orc.densenet_init(d + 1, 1, wl["arch"], seed=42)
        times = []
        orc.diffusion_train_loop(prob, params, K_cpu, wl["K_boundary"], N, wl["dt"], args.warmup + args.steps, wl["lr"],
                                 seed=42, times=times)
        return _print_reference(args, wl, times, K_cpu, N, cores)
    N = int(np.floor(prob.T / wl["dt"]))
    K_cpu = min(wl["K"], CPU_SAMPLE_K)  # the reference pre-draws xi = randn(K, d, N+1) on the host: ~0.5 MB per path
    if wl["net"] == "mlp":
        params, net = orc.mlp_init(d + 1, d, seed=123), "mlp_tanh"
    elif wl["ta"] == "outer":
        params, net = [orc.densenet_init(d, d, seed=42) for _ in range(N)], "densenet"
    else:
        params, net = orc.densenet_init(d + 1, d, seed=42), "densenet"
    times = []
    orc.hjb_train_loop(prob, net, params, K_cpu, wl["dt"], args.warmup + args.steps, wl["lr"], wl["loss"], wl["ta"],
                       True, wl["detach"], seed=42, times=times)
    _print_reference(args, wl, times, K_cpu, N, cores)


def _print_reference(args, wl, times, K_cpu, N, cores):
    t = times[args.warmup:]
    ms = 1e3 * sum(t) / len(t)
    value = K_cpu * N / (ms * 1e-3)
    sample = "K=%d of %d trajectories per step, N=%d, %d timed iterations" % (K_cpu, wl["K"], N, len(t))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "K_global": wl["K"] * args.gpus, "K_per_gpu": wl["K"], "N": N, "d": wl["pkw"]["d"],
                       "noise": "torch CPU randn(K, d, N+1) per iteration (the reference's own, solver.py:381)",
                       "parallelism": "host threads: %d" % cores, "device": "cpu", "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ----------------------------------------------------------------------------------------------- our arm
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--id=%d" % index, "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); smax.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(smax), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=max(power))
        return out


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh)
    except OSError:
        return {}


def fma_peak_tflops(lib, dev):
    """FP32 FMA throughput of this GPU, measured live with the library's probe kernel (best of 5)."""
    sink = pt.zeros(4, device=dev)
    stream = ctypes.c_void_p(pt.cuda.current_stream(dev).cuda_stream)
    best = 0.0
    for _ in range(6):
        e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
        e0.record()
        flops = lib.pspde_fma_probe(20000, ctypes.c_void_p(sink.data_ptr()), stream)
        e1.record()
        e1.synchronize()
        best = max(best, flops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def fwd_roofline(flops_fwd, tf_ms, fma_peak, eng):
    """Forward kernel: on the tensor cores (tcgen05 kind::tf32, 3 passes per product for FP32 equivalence) when the
    network is in the tensor-core kernel's shape class, else FP32 FMA.  The tensor bound is the measured bf16 GEMM
    peak / 2 (TF32 runs at half the bf16 rate) / 3 (passes): FP32-equivalent TFLOP/s."""
    ach = flops_fwd / (tf_ms * 1e-3) / 1e12
    hid_max = 32 if eng.net_id == 0 else 31          # MySequential keeps a bias column per hidden segment
    tc_path = os.environ.get("PSPDE_FWD_PATH", "") != "simt" and len(eng.dims) == 4 \
        and max(eng.dims[1:3]) <= hid_max and eng.time_mode == 0 and not (eng.flags & 1)
    out = {"achieved": ach, "frac_of_fp32_fma_peak": ach / fma_peak}
    if tc_path:
        bf16 = measured_peaks().get("bf16_tflops")
        src = "MEASURED_PEAKS.json bf16_tflops (burst) / 2 / 3"
        if not bf16:
            bf16, src = 1590.0, "fallback 1.59 PFLOP/s bf16 / 2 / 3"
        out.update(kernel="rollout_tc_fwd_kernel (tcgen05.mma kind::tf32, 3xTF32, A from tensor memory)", bound="tensor",
                   peak=bf16 / 6.0, frac=ach / (bf16 / 6.0), peak_source=src)
    else:
        out.update(kernel="rollout_kernel<FWD>", bound="fp32_fma", peak=fma_peak, frac=ach / fma_peak)
    return out


def build_solver(wl, K_global, dev, u_l2=False, name="bench"):
    import pspde
    pkw = dict(wl["pkw"])
    d = pkw["d"]
    if wl["kind"] == "llgc":
        prob = pspde.LLGC(device=dev, **pkw)
    elif wl["kind"] == "lqgc":
        prob = pspde.LQGC(device=dev, **pkw)
    else:
        prob = pspde.DoubleWell_multidim(device=dev, **pkw)
    S = pspde.Solver(name, prob, lr=wl["lr"], L=1, K=K_global, delta_t=wl["dt"], loss_method=wl["loss"],
                     time_approx=wl["ta"], detach_forward=wl["detach"], early_stopping_time=None,
                     u_l2_error_flag=u_l2, verbose=False, seed=42, noise="philox", device=dev)
    if wl["net"] == "densenet" and wl["ta"] == "inner":
        S.z_n = pspde.DenseNet(d_in=d + 1, d_out=d, lr=wl["lr"], seed=42)
        S.update_Phis()
    return S


class Rig:
    """Per-process state of one bench run: device, ranks, the L2 flush buffer, barrier + max-over-ranks helpers."""

    def __init__(self):
        import torch.distributed as td
        self.td = td
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not pt.cuda.is_available():
            raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        pt.cuda.set_device(self.local)
        self.dev = pt.device("cuda", self.local)
        if self.world > 1:
            td.init_process_group("nccl", device_id=self.dev)
        self.flush = pt.empty(256 << 20, dtype=pt.uint8, device=self.dev)     # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.td.barrier()
        pt.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        t = pt.tensor([x], dtype=pt.float64, device=self.dev)
        if self.world > 1:
            self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.td.destroy_process_group()


def timed_steps(rig, S, first, steps):
    """EXACTLY `steps` training iterations, one CUDA-event pair each (L2 flushed and ranks aligned between them, outside
    the pairs); returns the sum of the per-step device times in ms, max over ranks."""
    ms = []
    for l in range(steps):
        rig.flush.fill_(l & 1)
        rig.barrier()
        e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
        e0.record()
        S.train_step(first + l)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    rig.barrier()
    return rig.max_over_ranks(sum(ms))


def dump_outputs(out_dir, whole, per_path):
    """--dump-outputs: `whole` (name -> tensor or number) as is, `per_path` (name -> tensor with one row per local path)
    on the paths of a sample that depends only on the number of paths, as out_dir/<name>.npy in float32 / float64."""
    K = next(iter(per_path.values())).shape[0]
    rows = np.arange(K) if K <= DUMP_PATHS else np.sort(np.random.default_rng(0).choice(K, DUMP_PATHS, replace=False))
    arrays = {name: np.asarray(v, dtype=np.float64) for name, v in whole.items() if not pt.is_tensor(v)}
    arrays.update({name: v.detach().cpu().numpy() for name, v in whole.items() if pt.is_tensor(v)})
    sel = pt.from_numpy(rows)
    arrays.update({name: v.detach()[sel.to(v.device)].cpu().numpy() for name, v in per_path.items()})
    arrays["path_index"] = rows.astype(np.float64)
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError("--dump-outputs: %s is %s, not float32 / float64" % (name, a.dtype))
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def timed_e2e(rig, S, eng, first, steps):
    """Wall clock of `steps` iterations through the public API with HOST inputs: the problem functor pack and x0 come from
    pinned host memory every step, the loss goes back to the host every step.  Returns (seconds max over ranks, h2d, d2h)."""
    pack_h = eng.pack.detach().cpu().pin_memory()
    x0_h = eng.x0.detach().cpu().pin_memory()
    rig.barrier()
    w0 = time.perf_counter()
    for l in range(steps):
        eng.pack.copy_(pack_h, non_blocking=True)
        eng.x0.copy_(x0_h, non_blocking=True)
        S.train_step(first + l)          # ends with the D2H read of (loss, n_bad, u_L2)
    rig.barrier()
    w1 = time.perf_counter()
    return rig.max_over_ranks(w1 - w0), int(pack_h.numel() * 4 + x0_h.numel() * 4), 24


def time_kernels(rig, S, eng, reps):
    """Kernel-level CUDA-event times (ms, medians) of the training forward and of the backward, on the launching stream."""
    from pspde.fused import Call
    tf, tb = [], []
    theta = S._theta.detach()
    wY = pt.randn(eng.K_local, device=rig.dev) / eng.K_global
    grad = pt.empty(eng.n_theta, device=rig.dev)
    for i in range(reps):
        c = Call(offset=1000 + i)
        rig.flush.fill_(i & 1)
        e = [pt.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        single = eng.forward(theta, None, c, keep_rows=True)   # the training forward (keeps its operand rows if a buffer exists)
        e[1].record()
        rig.flush.fill_(1 - (i & 1))
        e[2].record()
        if single:
            eng.grad_from_rows(theta, wY, c, grad)
        else:
            eng.backward_detached(theta, wY, None, c, grad)
        e[3].record()
        pt.cuda.synchronize(rig.dev)
        tf.append(e[0].elapsed_time(e[1])); tb.append(e[2].elapsed_time(e[3]))
    return statistics.median(tf), statistics.median(tb), single


def tc_shape_class(eng, env):
    hid_max = 32 if eng.net_id == 0 else 31          # MySequential keeps a bias column per hidden segment
    return os.environ.get(env, "") != "simt" and len(eng.dims) == 4 and max(eng.dims[1:3]) <= hid_max \
        and eng.time_mode == 0 and not (eng.flags & 1)


def detached_roofline(rig, lib, S, eng, N, clocks, workload):
    """Roofline of the dominant kernel of the detached (log-variance) step: the backward.  In the tensor-core shape class all of
    its multiply-adds -- the weight gradient and the hidden cotangents -- run on tcgen05 kind::tf32 in 3 passes, so the bound
    is the tensor pipe: FP32-equivalent peak = measured bf16 GEMM peak / 2 (TF32 rate) / 3 (passes).  The FP32-FMA-equivalent
    fraction (what the same algorithmic FLOPs would be of the CUDA-core peak) is kept as a note."""
    from pspde import _lib
    M, Md = net_macs(eng.dims, eng.net_id == _lib.NET_DENSENET)
    flops_fwd = 2.0 * M * eng.K_local * N                  # forward kernel: one network evaluation per path-step
    flops_bwd = 2.0 * (M + Md) * eng.K_local * N           # backward: weight gradient + hidden cotangents
    tf, tb, single = time_kernels(rig, S, eng, 5)          # (a recomputed forward inside the backward is NOT counted)
    fma_peak = fma_peak_tflops(lib, rig.dev)
    nominal = 148 * 128 * 2 * ((clocks or {}).get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
    peaks = measured_peaks()
    bf16 = peaks.get("bf16_tflops")
    tsrc = "MEASURED_PEAKS.json bf16_tflops (burst) / 2 / 3"
    if not bf16:
        bf16, tsrc = 1590.0, "fallback 1.59 PFLOP/s bf16 (B200_PROFILING.md) / 2 / 3"
    tpeak = bf16 / 6.0
    ach = flops_bwd / (tb * 1e-3) / 1e12
    prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
            prof = json.load(fh)
    except OSError:
        pass
    ckpt_path = tc_shape_class(eng, "PSPDE_BWD_PATH")
    cols = 0
    if ckpt_path:
        s0 = (eng.d + 2 + 7) // 8 * 8
        cols = s0 + 64                       # [a0 | h1 | h2]; zeta is regenerated from the Philox key in the gradient kernel
    row_bytes = 4.0 * cols * eng.K_local * N
    kept = (eng.ckpt.numel() / eng._ckpt_need) if (ckpt_path and single and eng.ckpt is not None) else 0.0
    if ckpt_path and single:
        kernel = ("single-rollout step: the training forward (rollout_tc_fwd_kernel<CKPT>, 'fwd') keeps the operand rows "
                  "[a0|h1|h2] of its tiles in HBM; backward = grad_tc_kernel over those rows (TMA-fed, zeta regenerated from "
                  "Philox, hidden cotangents and weight gradient on tcgen05 kind::tf32 3xTF32) + reduce; tiles the buffer does "
                  "not hold (rows_kept_fraction < 1) go through the wave-checkpointed backward inside 'bwd'")
    elif ckpt_path:
        kernel = ("wave-checkpointed backward = per wave of 148 x 2 tiles: rollout_tc_fwd_kernel<CKPT> (tensor-core rollout "
                  "that leaves the operand rows [a0|h1|h2] in a K-independent workspace) + grad_tc_kernel (TMA-fed, zeta "
                  "regenerated from Philox, hidden cotangents and weight gradient on tcgen05 kind::tf32 3xTF32); timed together")
    else:
        kernel = "rollout_kernel<BWD> (detached backward, FP32-FMA recompute)"
    key = workload if (single or not ckpt_path) else workload + "_two_rollout_step"      # profiles/roofline_traffic.json
    roof = {"bound": "tensor" if ckpt_path else "fp32_fma", "kernel": kernel, "achieved": ach,
            "peak": tpeak if ckpt_path else fma_peak, "unit": "TFLOP/s", "frac": ach / (tpeak if ckpt_path else fma_peak),
            "peak_source": tsrc if ckpt_path else "fp32 FMA probe measured live in this run",
            "algorithmic_flops_per_path_step": 2.0 * (M + Md),
            "fma_equivalent": {"peak": fma_peak, "frac": ach / fma_peak, "nominal_peak": nominal, "frac_of_nominal": ach / nominal,
                               "note": "the same algorithmic FLOPs against the FP32 CUDA-core peak (probe measured live; "
                                       "MEASURED_PEAKS.json has no fp32 figure)"},
            "traffic": prof.get(key, {}).get("bwd_dram_bytes_per_launch"),
            "kernel_ms": {"fwd": tf, "bwd": tb},
            "single_rollout": bool(ckpt_path and single), "rows_kept_fraction": kept,
            "bwd_checkpoint": {"algorithmic_bytes_per_step": row_bytes * 2,         # written once, read once
                               "gbs_over_bwd": row_bytes * (2.0 - kept) / (tb * 1e-3) / 1e9,
                               "gbs_over_fwd": row_bytes * kept / (tf * 1e-3) / 1e9,
                               "hbm_peak_gbs_measured": peaks.get("hbm_gbs")} if ckpt_path else None,
            "fwd": fwd_roofline(flops_fwd, tf, fma_peak, eng),
            "step": {"algorithmic_flops_per_path_step": 2.0 * (2 * M + Md),
                     "achieved": (flops_fwd + flops_bwd) / ((tf + tb) * 1e-3) / 1e12,
                     "frac_of_tensor_bound": (flops_fwd + flops_bwd) / ((tf + tb) * 1e-3) / 1e12 / tpeak,
                     "frac_of_fp32_fma_peak": (flops_fwd + flops_bwd) / ((tf + tb) * 1e-3) / 1e12 / fma_peak},
            "hbm_peak_gbs_measured": peaks.get("hbm_gbs")}
    return roof


def attached_roofline(rig, lib, S, eng, N):
    """Attached (relative-entropy) step: one launch of rollout_attached_kernel = forward sweep + adjoint sweep, FP32 FMA.
    Algorithmic FLOPs per path-step: 2 (2M + M_delta + M_x), M_x = the input-Jacobian product J_x' zeta (= M for these nets)."""
    from pspde import _lib
    from pspde.fused import Call
    M, Md = net_macs(eng.dims, eng.net_id == _lib.NET_DENSENET)
    flops = 2.0 * (3 * M + Md) * eng.K_local * N
    theta = S._theta.detach()
    grad = pt.empty(eng.n_theta, device=rig.dev)
    ts = []
    for i in range(4):
        rig.flush.fill_(i & 1)
        e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
        e0.record(); eng.attached(theta, Call(offset=1000 + i), grad); e1.record()
        pt.cuda.synchronize(rig.dev)
        ts.append(e0.elapsed_time(e1))
    t = statistics.median(ts[1:])
    peak = fma_peak_tflops(lib, rig.dev)
    ach = flops / (t * 1e-3) / 1e12
    return {"bound": "fp32_fma", "kernel": "rollout_attached_kernel (forward sweep + adjoint sweep with state checkpoints, one launch)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "peak_source": "fp32 FMA probe measured live in this run (MEASURED_PEAKS.json has no fp32 figure)",
            "algorithmic_flops_per_path_step": 2.0 * (3 * M + Md), "traffic": None, "kernel_ms": {"attached": t},
            "hbm_peak_gbs_measured": measured_peaks().get("hbm_gbs")}


def cpu_port_baseline(wl, N, K_cpu, iters, threads):
    """oracle/ref_port.py (the reference's CPU procedure: torch eager + autograd + CPU randn) on `threads` host threads."""
    from oracle import ref_port as orc
    pt.set_num_threads(threads)
    d = wl["pkw"]["d"]
    pkw = {k: v for k, v in wl["pkw"].items() if k != "d"}
    prob = orc.make_problem(wl["kind"], d, **pkw)
    if wl["net"] == "mlp":
        params, net = orc.mlp_init(d + 1, d, seed=123), "mlp_tanh"
    elif wl["ta"] == "outer":
        params, net = [orc.densenet_init(d, d, seed=42) for _ in range(N)], "densenet"
    else:
        params, net = orc.densenet_init(d + 1, d, seed=42), "densenet"
    times = []
    orc.hjb_train_loop(prob, net, params, K_cpu, wl["dt"], iters, wl["lr"], wl["loss"], wl["ta"], True, wl["detach"],
                       seed=42, times=times)
    tt = times[1:] if len(times) > 1 else times
    return K_cpu * N / (sum(tt) / len(tt)), len(tt)


def eager_gpu_baseline(wl, N, K_gpu, iters, dev):
    """The same eager procedure (oracle/ref_port.py) with its tensors on the B200 -- the reference's own device='cuda' mode
    (solver.py:36): noise drawn on the host and copied (:381), one aten kernel per operation, autograd tape in HBM."""
    from oracle import ref_port as orc
    d = wl["pkw"]["d"]
    pkw = {k: v for k, v in wl["pkw"].items() if k != "d"}
    prob = orc.make_problem(wl["kind"], d, **pkw)
    if wl["net"] == "mlp":
        params, net = orc.mlp_init(d + 1, d, seed=123), "mlp_tanh"
    elif wl["ta"] == "outer":
        params, net = [orc.densenet_init(d, d, seed=42) for _ in range(N)], "densenet"
    else:
        params, net = orc.densenet_init(d + 1, d, seed=42), "densenet"
    orc.to_device(prob, params, dev)
    times = []
    orc.hjb_train_loop(prob, net, params, K_gpu, wl["dt"], iters, wl["lr"], wl["loss"], wl["ta"], True, wl["detach"],
                       seed=42, times=times, device=dev)
    tt = times[1:] if len(times) > 1 else times
    return K_gpu * N / (sum(tt) / len(tt)), len(tt)


def cpu_baseline_block(wl, N, dev=None):
    cores = os.cpu_count() or 1
    K_cpu = min(wl["K"], CPU_SAMPLE_K)
    v, n = cpu_port_baseline(wl, N, K_cpu, 3, cores)
    K1 = min(wl["K"], 1024)
    v1, n1 = cpu_port_baseline(wl, N, K1, 2, 1)
    pt.set_num_threads(cores)
    eager = None
    if dev is not None:
        try:
            vg, ng = eager_gpu_baseline(wl, N, K_cpu, 4, dev)
            eager = {"value": vg, "unit": UNIT, "device": pt.cuda.get_device_name(dev),
                     "sample": "K=%d, N=%d, %d timed iterations after 1 warm-up; PyTorch eager on the GPU (the reference's "
                               "device='cuda' mode: host randn + H2D, aten kernels, autograd), context only" % (K_cpu, N, ng)}
        except Exception as e:                     # context only: never fail the bench line over it
            eager = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
        pt.cuda.empty_cache()
    return {"torch_eager_gpu": eager, "value": v, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "K=%d of %d trajectories, N=%d, %d timed iterations after 1 warm-up (torch CPU eager + autograd + CPU "
                      "randn, the reference's procedure)" % (K_cpu, wl["K"], N, n),
            "one_thread": {"value": v1, "unit": UNIT, "cores": 1,
                           "sample": "K=%d, N=%d, %d timed iteration(s) after 1 warm-up" % (K1, N, n1)}}


def accuracy_block(rig, iters):
    """Second half of BASELINE.json's metric on configs[1] (LLGC d=100, K=2^16 global, N=100, lr=1e-3, log-variance): train for a
    fixed budget, then (reference: problems.py:51-65 u_true / v_true, utilities.py:440-472 compute_test_error)
      V(0,0)      -mean(Y_N - g(X_N)) of the last training batch against -(d/4)(1 - exp(-2T)) = -21.6166
      u           sqrt(u_L2 / int |u*|^2 dt): the device diagnostic of solver.py:491-494 relative to the analytic control
      V(.,0)      64 test points x ~ 0.5 N(0, I): one forward rollout of 1024 controlled paths from each,
                  V^(x) = -mean(Y_N - g(X_N)), against LLGC.v_true(x, 0)"""
    from pspde.fused import Call
    wl = dict(WORKLOADS["c2"])
    S = build_solver(wl, wl["K"], rig.dev, u_l2=True, name="accuracy")
    d, T = S.d, float(S.T)
    V00 = -(d / 4.0) * (1.0 - np.exp(-2.0 * T))
    u_norm2 = d * (1.0 - np.exp(-2.0 * T)) / 2.0                 # int_0^T |u*(t)|^2 dt, u* = -exp(-(T-t)) 1
    eng = S._get_engine()
    trace = []
    t0 = time.perf_counter()
    for l in range(iters):
        S.train_step(l)
        if l + 1 in (100, 300, 1000, 3000) and l + 1 < iters:     # convergence trace (the last batch's statistics)
            st = eng.stats.clone()
            if rig.world > 1:
                rig.td.all_reduce(st)
            trace.append({"iteration": l + 1, "loss": S.loss_log[-1], "V00_rel_err": abs(-(st[0].item() / S.K) - V00) / abs(V00),
                          "u_rel_L2_err": float(np.sqrt(max(S.u_L2_loss[-1], 0.0) / u_norm2))})
    pt.cuda.synchronize(rig.dev)
    train_s = time.perf_counter() - t0
    stats = eng.stats.clone()
    if rig.world > 1:
        rig.td.all_reduce(stats)
    est = -(stats[0].item() / S.K)
    out = {"workload": wl["desc"], "iterations": iters, "train_seconds": train_s, "loss_first": S.loss_log[0],
           "loss_last": S.loss_log[-1], "V00": est, "V00_exact": V00, "V00_rel_err": abs(est - V00) / abs(V00),
           "u_rel_L2_err": float(np.sqrt(max(S.u_L2_loss[-1], 0.0) / u_norm2)), "u_L2_first": S.u_L2_loss[0],
           "u_L2_last": S.u_L2_loss[-1], "trace": trace}
    # V(.,0) on test points: per-path starts, one forward launch on this rank's shard of the 64 x 1024 paths
    n_pts, per = 64, 1024
    g = pt.Generator().manual_seed(7)
    pts = 0.5 * pt.randn(n_pts, d, generator=g)
    lo, hi = S._k_lo, S._k_hi
    idx = pt.arange(lo, hi) // per                              # test point of each local path (K_global = 64 * 1024)
    x0_saved, per_path_saved = eng.x0, eng.x0_per_path
    eng.set_x0(pts[idx].to(rig.dev))
    eng.forward(S._theta.detach(), None, Call(offset=10 ** 6))
    D = (eng.Y_N - eng.gX).double()
    sums = pt.zeros(n_pts, dtype=pt.float64, device=rig.dev).index_add_(0, idx.to(rig.dev), D)
    if rig.world > 1:
        rig.td.all_reduce(sums)
    eng.x0, eng.x0_per_path = x0_saved, per_path_saved
    v_hat = -(sums / per).cpu().numpy()
    v_ref = np.asarray(S.problem.v_true(pts, 0.0)).reshape(-1)
    out["V_rel_L2_err"] = float(np.linalg.norm(v_hat - v_ref) / np.linalg.norm(v_ref))
    out["V_test_points"] = "%d points x ~ 0.5 N(0, I), %d controlled paths each (Philox), against LLGC.v_true(x, 0)" % (n_pts, per)
    return out


def sharding_check(rig, wl):
    """Per-path results must not depend on the number of ranks (dist.py): K_global = wl K is sharded over the ranks, every
    rank runs the forward rollout of its shard at the initial theta, the Y_N of 1024 global paths i * K / 1024 (spread over all
    ranks) are gathered on rank 0 and compared BIT-EXACTLY with a one-shard recomputation of the same K on rank 0
    (reference: per-path Y_N of solver.py:164-168).  The sha256 of the sample is comparable across runs at different N."""
    import hashlib
    from pspde.fused import Call
    K = wl["K"]
    S = build_solver(wl, K, rig.dev, name="shard")
    eng = S._get_engine()
    theta = S._theta.detach()
    eng.forward(theta, None, Call(offset=0))
    stride = K // 1024
    lo, hi = S._k_lo, S._k_hi
    first = (lo + stride - 1) // stride * stride
    local = eng.Y_N[pt.arange(first, hi, stride, device=rig.dev) - lo].contiguous()
    sample = pt.zeros(1024, dtype=pt.float32, device=rig.dev)
    sample[first // stride: first // stride + local.numel()] = local
    if rig.world > 1:
        rig.td.all_reduce(sample)                  # disjoint supports, zeros elsewhere: the sum is a gather
    out = None
    if rig.rank == 0:
        from pspde.fused import RolloutEngine
        one = RolloutEngine(S.problem, S._net_id, S._dims, eng.time_mode, K, S.N, S.delta_t_np, adaptive=True, k_offset=0,
                            K_global=K, seed=S.seed, device=rig.dev)
        one.forward(theta, None, Call(offset=0))
        ref = one.Y_N[::stride].contiguous()
        out = {"sample": "Y_N of the 1024 global paths i * K / 1024, K_global = %d over %d rank(s), iteration 0, initial theta"
                         % (K, rig.world),
               "sha256": hashlib.sha256(sample.cpu().numpy().tobytes()).hexdigest(),
               "matches_one_shard": bool(pt.equal(sample, ref))}
        del one
    del S, eng
    pt.cuda.empty_cache()
    return out


def run_ours(args, wl):
    from pspde import _lib
    rig = Rig()
    rank, world, dev = rig.rank, rig.world, rig.dev
    lib = _lib.load()
    K_global = wl["K"] * world
    S = build_solver(wl, K_global, dev)
    N, d = S.N, S.d
    eng = S._get_engine()

    for l in range(args.warmup):
        S.train_step(l)
    rig.barrier()
    sampler = ClockSampler(rig.local) if rank == 0 else None
    launches0 = lib.pspde_launch_count()
    # ---- timed region A: device-timed steps
    total_ms = timed_steps(rig, S, args.warmup, args.steps)
    launches = lib.pspde_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": [S.loss_log[-1]], "theta": S._theta, "grad": S._theta.grad},
                     {"Y_N": eng.Y_N, "gX": eng.gX, "X_N": eng.X_N})
    ms_per_step = total_ms / args.steps
    value = K_global * N * args.steps / (total_ms * 1e-3)
    # ---- timed region B: end to end through the public API with host inputs
    e2e_s, h2d, d2h = timed_e2e(rig, S, eng, args.warmup + args.steps, args.steps)
    e2e_value = K_global * N * args.steps / e2e_s
    clocks = sampler.stop() if sampler else None

    # ---- roofline of the dominant kernel (rank 0 reports; every rank runs it so that nobody waits in a collective)
    roof = detached_roofline(rig, lib, S, eng, N, clocks, args.workload) if wl["detach"] else attached_roofline(rig, lib, S, eng, N)
    final_loss = S.loss_log[-1]
    del S, eng
    pt.cuda.empty_cache()

    extra = {}
    if args.workload == "c5" and not args.headline_only:
        # ---- configs[1] in the same process
        w2 = WORKLOADS["c2"]
        S2 = build_solver(w2, w2["K"] * world, dev)
        for l in range(3):
            S2.train_step(l)
        ms2 = timed_steps(rig, S2, 3, args.steps) / args.steps
        r2 = detached_roofline(rig, lib, S2, S2._get_engine(), S2.N, clocks, "c2")
        extra["c2"] = {"workload": w2["desc"], "K_global": w2["K"] * world, "ms_per_step": ms2,
                       "value": w2["K"] * world * S2.N / (ms2 * 1e-3), "unit": UNIT, "kernel_ms": r2["kernel_ms"],
                       "roofline_frac": r2["frac"], "single_rollout": r2["single_rollout"]}
        del S2
        pt.cuda.empty_cache()
        # ---- strong scaling: K_global fixed at one GPU's batch
        if world > 1:
            S3 = build_solver(wl, wl["K"], dev)
            for l in range(3):
                S3.train_step(l)
            ms3 = timed_steps(rig, S3, 3, args.steps) / args.steps
            extra["strong"] = {"K_global": wl["K"], "ms_per_step": ms3, "value": wl["K"] * S3.N / (ms3 * 1e-3), "unit": UNIT}
            del S3
            pt.cuda.empty_cache()
        extra["sharding_check"] = sharding_check(rig, wl)
        extra["accuracy"] = accuracy_block(rig, args.accuracy_iters)

    if rank != 0:
        rig.close()
        return

    # ---- CPU baseline beside it (rank 0, N=1 only): the oracle port on the host cores, bounded sample
    cpu = cpu_baseline_block(wl, N, dev) if (world == 1 and not args.no_cpu_baseline) else None

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "K_global": K_global, "K_per_gpu": wl["K"], "N": N, "d": d,
                       "noise": "in-kernel Philox4x32-10", "parallelism": "trajectory-sharded dp%d" % world,
                       "l2": "256 MiB buffer written between timed steps (outside the per-step CUDA-event pairs); "
                             "the kernels' working set is on-chip"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "how": "pspde.Solver.train_step through the C ABI, wall clock, problem functor pack + x0 copied "
                           "from pinned host memory and (loss, n_bad, u_L2) read back every step"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "final_loss": final_loss}
    line.update(extra)
    emit(line)
    rig.close()


def run_ours_c4(args, wl):
    """BASELINE config 4: one GeneralSolver iteration (device-side sampling, forward rollout with the directional
    derivative of V, loss, backward rollout, terminal-condition term, Adam) per step."""
    import torch.distributed as td
    import pspde
    from pspde import _lib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not pt.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    pt.cuda.set_device(local)
    dev = pt.device("cuda", local)
    if world > 1:
        td.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    d, N = wl["pkw"]["d"], wl["N"]
    K_global = wl["K"] * world
    prob = pspde.HeatEquation(device=dev, **wl["pkw"])
    G = pspde.GeneralSolver(prob, "bench", seed=42, delta_t=wl["dt"], N=N, lr=wl["lr"], L=1, K=K_global,
                            K_boundary=wl["K_boundary"], verbose=False, device=dev)
    G.V = pspde.DenseNet(d_in=d + 1, d_out=1, lr=wl["lr"], arch=wl["arch"], seed=42)
    eng = G._get_engine()
    flush = pt.empty(256 << 20, dtype=pt.uint8, device=dev)

    def barrier():
        if world > 1:
            td.barrier()
        pt.cuda.synchronize(dev)

    for l in range(args.warmup):
        G.train_step(l)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = lib.pspde_launch_count()
    step_ms = []
    for l in range(args.steps):
        flush.fill_(l & 1)
        barrier()
        e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
        e0.record()
        G.train_step(args.warmup + l)
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    barrier()
    launches = lib.pspde_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": [G.loss_log[-1]], "theta": G._theta, "grad": G._theta.grad},
                     {"V0": eng.V0, "VE": eng.VE, "Y": eng.Y, "X_end": eng.X_end, "t_end": eng.t_end})
    t = pt.tensor([sum(step_ms)], dtype=pt.float64, device=dev)
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    total_ms = float(t.item())
    value = K_global * N * args.steps / (total_ms * 1e-3)
    pack_h = eng.pack.detach().cpu().pin_memory()
    barrier()
    w0 = time.perf_counter()
    for l in range(args.steps):
        eng.pack.copy_(pack_h, non_blocking=True)
        G.train_step(args.warmup + args.steps + l)
    barrier()
    w1 = time.perf_counter()
    t = pt.tensor([w1 - w0], dtype=pt.float64, device=dev)
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    e2e_value = K_global * N * args.steps / float(t.item())
    clocks = sampler.stop() if sampler else None
    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return
    # kernel-level timing + roofline (FP32 FMA bound; value and tangent rows: 2 network rows per path-step)
    M, Md = net_macs(eng.dims, True)
    theta = G._theta.detach()
    X0, t0 = eng.sample(1.0, 12345)
    w = pt.randn(eng.K_local, device=dev) / K_global
    grad = pt.empty(eng.n_theta, device=dev)
    tf, tb = [], []
    for i in range(4):
        flush.fill_(i & 1)
        e = [pt.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(); eng.forward(theta, X0, t0, None, 12345); e[1].record()
        flush.fill_(1 - (i & 1))
        e[2].record(); eng.backward(theta, X0, t0, None, 12345, -w, w, -w, grad); e[3].record()
        pt.cuda.synchronize(dev)
        if i:
            tf.append(e[0].elapsed_time(e[1])); tb.append(e[2].elapsed_time(e[3]))
    tf, tb = statistics.median(tf), statistics.median(tb)
    peak = fma_peak_tflops(lib, dev)
    ps = eng.K_local * N
    flops_fwd, flops_bwd = 4.0 * M * ps, 4.0 * (M + Md) * ps
    ach = flops_bwd / (tb * 1e-3) / 1e12
    roof = {"bound": "fp32_fma", "kernel": "diffusion_kernel<BWD> (reverse of the value/tangent pair + weight gradient, recompute)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "peak_source": "fp32 FMA probe measured live in this run (MEASURED_PEAKS.json has no fp32 figure)",
            "traffic": None, "kernel_ms": {"fwd": tf, "bwd": tb},
            "fwd": {"achieved": flops_fwd / (tf * 1e-3) / 1e12, "frac": flops_fwd / (tf * 1e-3) / 1e12 / peak},
            "step": {"algorithmic_flops_per_path_step": 4.0 * (2 * M + Md),
                     "achieved": (flops_fwd + flops_bwd) / ((tf + tb) * 1e-3) / 1e12,
                     "frac": (flops_fwd + flops_bwd) / ((tf + tb) * 1e-3) / 1e12 / peak},
            "hbm_peak_gbs_measured": measured_peaks().get("hbm_gbs")}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import ref_port as orc
        cores = os.cpu_count() or 1
        pt.set_num_threads(cores)
        K_cpu = 1024
        params = orc.densenet_init(d + 1, 1, wl["arch"], seed=42)
        times = []
        orc.diffusion_train_loop(orc.make_problem("heat", d, T=1), params, K_cpu, wl["K_boundary"], N, wl["dt"], 3,
                                 wl["lr"], seed=42, times=times)
        tt = times[1:]
        cpu = {"value": K_cpu * N / (sum(tt) / len(tt)), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "K=%d of %d points, N=%d, 2 timed iterations after 1 warm-up (torch CPU eager, autograd with "
                         "create_graph per step: the reference's procedure)" % (K_cpu, wl["K"], N)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "K_global": K_global, "K_per_gpu": wl["K"], "N": N, "d": d,
                       "noise": "device-side Philox4x32-10 (initial points and increments)",
                       "parallelism": "trajectory-sharded dp%d" % world,
                       "l2": "256 MiB buffer written between timed steps; weights (371 KB) are re-read from L2 every tile-step by design"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(pack_h.numel() * 4), "d2h_bytes_per_step": 32,
                    "how": "pspde.GeneralSolver.train_step through the C ABI, wall clock, problem functor pack copied from "
                           "pinned host memory and (loss, K_count) read back every step"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "final_loss": G.loss_log[-1]}
    emit(line)
    if world > 1:
        td.destroy_process_group()


_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner comes out of a plain printf
    whenever NCCL_DEBUG is VERSION or WARN, whatever NCCL_DEBUG_FILE says): keep a private handle on the real stdout for the
    JSON line and point file descriptor 1 at stderr for everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the c2 / strong / sharding / accuracy blocks")
    ap.add_argument("--accuracy-iters", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif wl["kind"] == "heat":
        run_ours_c4(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
