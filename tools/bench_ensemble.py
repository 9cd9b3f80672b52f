"""Ensemble throughput: ms per SolverEnsemble iteration for M members against one standalone Solver iteration.

Two notebook-sized configurations: C1 (LQGC d = 10, 'outer' DenseNet, K = 200, log-variance) and an 'inner'
DoubleWell_multidim d = 50 with MySequential at K = 256.  The standalone iteration is timed with its natural kernels and
forced onto the FP32-FMA kernels the ensemble runs (PSPDE_FWD_PATH / PSPDE_BWD_PATH=simt); the ensemble for each M.
CUDA events around `iters` warmed iterations (each ends in the iteration's host sync).  Prints one JSON line with the GPU
name and power limit read in the same run; --out also writes it to a file.

    python tools/bench_ensemble.py --iters 30 --out bench_ensemble.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "path-space-pde-solver_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch as pt  # noqa: E402

CONFIGS = {
    "c1": dict(problem="lqgc", pkw=dict(d=10), ta="outer", K=200, dt=0.05, lr=1e-3),
    "dwm50_inner": dict(problem="dwm", pkw=dict(d=50, d_1=15, d_2=35, T=1, eta=3, kappa=5), ta="inner", K=256, dt=0.005,
                        lr=0.05),
}


def solver(cfg, seed, L):
    import pspde
    prob = pspde.LQGC(device="cuda", **cfg["pkw"]) if cfg["problem"] == "lqgc" else \
        pspde.DoubleWell_multidim(device="cuda", **cfg["pkw"])
    return pspde.Solver("bench", prob, lr=cfg["lr"], L=L, K=cfg["K"], delta_t=cfg["dt"], loss_method="log-variance",
                        time_approx=cfg["ta"], detach_forward=True, early_stopping_time=None, verbose=False, seed=seed)


def timed(step, warmup, iters):
    for l in range(warmup):
        step(l)
    e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
    e0.record()
    for l in range(warmup, warmup + iters):
        step(l)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_info():
    name = pt.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        power = out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--models", default="1,8,37,74,148")
    ap.add_argument("--configs", default="c1,dwm50_inner")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import pspde
    if not pt.cuda.is_available():
        raise SystemExit("bench_ensemble.py needs a CUDA device")
    L = args.warmup + args.iters + 1
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, iters=args.iters, warmup=args.warmup, configs={})
    for key in args.configs.split(","):
        cfg = CONFIGS[key]
        row = {}
        for label, env in (("standalone_natural_ms", None), ("standalone_fma_ms", "simt")):
            for v in ("PSPDE_FWD_PATH", "PSPDE_BWD_PATH"):
                if env:
                    os.environ[v] = env
                else:
                    os.environ.pop(v, None)
            s = solver(cfg, 42, L)
            row[label] = timed(s.train_step, args.warmup, args.iters)
        for v in ("PSPDE_FWD_PATH", "PSPDE_BWD_PATH"):
            os.environ.pop(v, None)
        row["ensemble"] = {}
        for M in (int(m) for m in args.models.split(",")):
            ens = pspde.SolverEnsemble([solver(cfg, 1000 + m, L) for m in range(M)], verbose=False)
            ms = timed(ens.train_step, args.warmup, args.iters)
            row["ensemble"][str(M)] = dict(ms_per_iter=ms, member_iters_per_s=M / ms * 1e3,
                                           speedup_vs_sequential_natural=M * row["standalone_natural_ms"] / ms,
                                           speedup_vs_sequential_fma=M * row["standalone_fma_ms"] / ms)
            del ens
            pt.cuda.empty_cache()
        res["configs"][key] = row
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
