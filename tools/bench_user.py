"""What a user-written target costs against the hand-written built-in model of the same density, fp64.

For each built-in target with a restatement in tests/user_targets (eight schools non-centered, logistic regression
MODERATE, ARMA(1,1) MODERATE) and each sampler, the built-in model and the CudaModel run on the same seed and
configuration: --chains chains, --warmup adapting draws, then
  - chain-draws/s over a steady-state window timed with CUDA events (sized from a probe to hold about --seconds),
  - evaluations per draw and acceptance over that window,
  - ESS per chain-draw (min and median over coordinates) from a separate run(..., chain_stats=True) pass,
  - the kernel that ran (klhr_launch_info).
The GPU's name and power limit are read in the same run.  One JSON line per (target, sampler, model); the user
lines carry user_over_builtin, the ratio of the two chain-draw rates.

    python tools/bench_user.py [--chains 65536] [--seconds 1.0] [--warmup 200] [--ess-draws 200]
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import klhr_b200 as kb  # noqa: E402
from bench_hier import gpu_identity, kernel_name  # noqa: E402
from klhr_b200.diagnostics import chain_summary  # noqa: E402
from oracle import glm_models, ts_models  # noqa: E402
from oracle.hier_models import EIGHT_SCHOOLS_DATA  # noqa: E402

TARGETS = ROOT / "tests" / "user_targets"
CASES = {  # name: (user source, built-in Stan program, data, dim)
    "eight_schools_noncentered": ("eight_schools_noncentered.cuh", "eight_schools_noncentered", EIGHT_SCHOOLS_DATA, 10),
    "logistic_regression": ("logistic_regression.cuh", "logistic_regression", glm_models.MODERATE, 3),
    "arma11": ("arma11.cuh", "arma11", ts_models.MODERATE, 4),
}


def measure(model, cls, chains, seconds, warmup, ess_draws, seed):
    import numpy as np
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
    n = max(2, int(np.ceil(seconds / (e0.elapsed_time(e1) / 1e3 / n))))
    acc0, ev0, d0 = s._accept_count.clone(), s.grad_evals, s._draw
    e0.record()
    s.run(n)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3
    n = s._draw - d0                    # draws the window ran (a window closure can add one)
    s1, s2 = s.run(ess_draws, chain_stats=True)
    epd = chain_summary(s1, s2, ess_draws)["ess_per_draw"].cpu().numpy()
    return dict(chain_draws_per_s=n * chains / t, evals_per_draw=(s.grad_evals - ev0) / (n * chains),
                accept=float((s._accept_count - acc0).double().sum()) / (n * chains), timed_draws=n,
                timed_seconds=round(t, 4), kernel=kind, regs=info["regs"],
                ess_per_chain_draw_min=float(epd.min()), ess_per_chain_draw_median=float(np.median(epd)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--chains", type=int, default=65_536)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--ess-draws", type=int, default=200)
    ap.add_argument("--targets", default=",".join(CASES))
    ap.add_argument("--samplers", default="KLHR,KLHRSINH")
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_user needs a CUDA device")
    gpu, power = gpu_identity()
    for name in args.targets.split(","):
        src, stan, data, dim = CASES[name]
        for cls in args.samplers.split(","):
            rates = {}
            for which, model in (("builtin", kb.BSModel(stan_file=f"{stan}.stan", data=data)),
                                 ("user", kb.CudaModel(TARGETS / src, data, dim))):
                t0 = time.time()
                r = dict(target=name, model=which, sampler=cls, D=dim, dtype="float64", chains=args.chains,
                         warmup=args.warmup, ess_draws=args.ess_draws)
                r.update(measure(model, cls, args.chains, args.seconds, args.warmup, args.ess_draws, args.seed))
                rates[which] = r["chain_draws_per_s"]
                if which == "user":
                    r["user_over_builtin"] = rates["user"] / rates["builtin"]
                r.update(gpu=gpu, power_limit_and_max_sm_clock=power, wall_s=round(time.time() - t0, 1))
                print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
