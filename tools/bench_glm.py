"""Throughput and efficiency of KLHR / KLHRSINH on Bayesian logistic regression, fp64.

Logistic regression is the first target whose line restriction is a sum over the N observations: every evaluation
recomputes X theta and X rho row by row (2 D FMAs, one exp, one log1p per observation), and for D <= 16 the sinh
family's exact gradient clip adds one full lp_grad per evaluation.  For each (N, K, sampler): 65 536 chains on
synthetic data (seeded), --warmup adapting draws, then
  - chain-draws/s over a steady-state window timed with CUDA events (sized from a probe to hold about --seconds),
  - evaluations per draw (grad_evals over the window) and acceptance,
  - observation terms per second, chain-draws/s x evals/draw x N (the clip's extra lp_grad not counted),
  - the kernel that ran (klhr_launch_info),
  - ESS per chain-draw (min and median over coordinates) from a separate run(..., chain_stats=True) pass.
The GPU's name and power limit are read in the same run.  One JSON line per case on stdout.

    python tools/bench_glm.py [--chains 65536] [--seconds 1.0] [--warmup 200] [--ess-draws 200] [--n 100,1000,10000]
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import klhr_b200 as kb  # noqa: E402
from bench_hier import gpu_identity, kernel_name  # noqa: E402
from klhr_b200.diagnostics import chain_summary  # noqa: E402
from oracle.glm_models import synthetic  # noqa: E402


def case(N, K, cls, chains, seconds, warmup, ess_draws, seed):
    data = synthetic(N, K, seed=1000 + N + K, scale=1.0 / np.sqrt(K), beta=np.ones(K))
    model = kb.BSModel(stan_file="logistic_regression.stan", data=data)
    s = getattr(kb, cls)(model, seed=seed, chains=chains, warmup=warmup)
    s.run(warmup)
    torch.cuda.synchronize()
    kind, info = kernel_name(model, s._fit)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 2
    e0.record()
    s.run(n)
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) / 1e3 / n
    n = max(2, int(np.ceil(seconds / per)))
    acc0 = s._accept_count.clone()
    ev0 = s.grad_evals
    e0.record()
    s.run(n)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3
    acc = float((s._accept_count - acc0).double().sum()) / (n * chains)
    evals = (s.grad_evals - ev0) / (n * chains)
    s1, s2 = s.run(ess_draws, chain_stats=True)
    epd = chain_summary(s1, s2, ess_draws)["ess_per_draw"].cpu().numpy()
    rate = n * chains / t
    return dict(N=N, K=K, D=K + 1, sampler=cls, dtype="float64", chains=chains, warmup=warmup, timed_draws=n,
                timed_seconds=round(t, 4), chain_draws_per_s=rate, accept=acc, evals_per_draw=evals,
                obs_terms_per_s=rate * evals * N, kernel=kind, threads_per_cta=info["threads"],
                smem_bytes=info["smem"], regs=info["regs"], ess_draws=ess_draws,
                ess_per_chain_draw_min=float(epd.min()), ess_per_chain_draw_median=float(np.median(epd)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--chains", type=int, default=65_536)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--ess-draws", type=int, default=200)
    ap.add_argument("--n", default="100,1000,10000")
    ap.add_argument("--k", default="4,24")
    ap.add_argument("--samplers", default="KLHR,KLHRSINH")
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_glm needs a CUDA device")
    gpu, power = gpu_identity()
    for N in map(int, args.n.split(",")):
        for K in map(int, args.k.split(",")):
            for cls in args.samplers.split(","):
                t0 = time.time()
                r = case(N, K, cls, args.chains, args.seconds, args.warmup, args.ess_draws, args.seed)
                r.update(gpu=gpu, power_limit_and_max_sm_clock=power, wall_s=round(time.time() - t0, 1))
                print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
