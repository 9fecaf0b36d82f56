"""Throughput and efficiency of KLHR / KLHRSINH on eight schools (non-centered and centered), fp64.

For each (target, sampler): 262 144 chains on the classic data, the default 1000-draw warm-up, then
  - chain-draws/s over a steady-state window timed with CUDA events (the window is sized from a probe to hold at
    least --seconds of work; the launch shape was warmed by the warm-up and the probe),
  - the acceptance of that window (the change of the sampler's accept counts over it), evaluations per draw
    (grad_evals over it), and the kernel that ran (klhr_launch_info: threads per CTA, shared memory, registers),
  - ESS per chain-draw of every coordinate (min and median) from a separate run(..., chain_stats=True) pass, and the
    per-coordinate z-scores of that pass against the exact posterior (oracle/hier_truth.py).
The GPU's name and power limit are read in the same run.  One JSON line per case on stdout.

    python tools/bench_hier.py [--chains 262144] [--seconds 1.0] [--ess-draws 1000]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import klhr_b200 as kb  # noqa: E402
from klhr_b200.diagnostics import chain_summary  # noqa: E402
from oracle.hier_truth import posterior_moments  # noqa: E402
from oracle.hier_models import EIGHT_SCHOOLS_DATA  # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unavailable ({e})"
    return name, out


def kernel_name(model, fit):
    info = kb.launch_info(model, fit, dtype=torch.float64, free_running=True, accumulate=False)
    D = model.dim()
    kind = ("chain kernel, thread-per-chain D-phase" if D <= 16 else "chain kernel, octet D-phase") \
        if info["threads"] == 32 else "octet kernel"
    return kind, info


def case(name, cls, chains, seconds, ess_draws, seed):
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=EIGHT_SCHOOLS_DATA)
    s = getattr(kb, cls)(model, seed=seed, chains=chains, warmup=1000)
    s.run(1000)                                          # the default warm-up
    torch.cuda.synchronize()
    kind, info = kernel_name(model, s._fit)
    # probe: size the window to at least `seconds` of work
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    s.run(n)
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) / 1e3 / n
    n = max(20, int(np.ceil(1.25 * seconds / per)))      # margin: the probe's rate includes its own ramp-up
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
    summ = chain_summary(s1, s2, ess_draws)
    mean, var = posterior_moments(EIGHT_SCHOOLS_DATA["y"], EIGHT_SCHOOLS_DATA["sigma"])[
        "noncentered" if name.endswith("noncentered") else "centered"]
    zm = (summ["mean"].cpu().numpy() - mean) / summ["mcse_mean"].cpu().numpy()
    zv = (summ["var"].cpu().numpy() - var) / summ["mcse_var"].cpu().numpy()
    epd = summ["ess_per_draw"].cpu().numpy()
    return dict(target=name, sampler=cls, dtype="float64", chains=chains, warmup=1000, timed_draws=n,
                timed_seconds=round(t, 4), chain_draws_per_s=n * chains / t, accept=acc, evals_per_draw=evals,
                kernel=kind, threads_per_cta=info["threads"], smem_bytes=info["smem"], regs=info["regs"],
                ess_draws=ess_draws, ess_per_chain_draw_min=float(epd.min()),
                ess_per_chain_draw_median=float(np.median(epd)),
                z_mean=[round(float(v), 2) for v in zm], z_var=[round(float(v), 2) for v in zv],
                parameters=model.parameter_names())


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--chains", type=int, default=262_144)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--ess-draws", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_hier needs a CUDA device")
    gpu, power = gpu_identity()
    for name in ("eight_schools_noncentered", "eight_schools_centered"):
        for cls in ("KLHR", "KLHRSINH"):
            t0 = time.time()
            r = case(name, cls, args.chains, args.seconds, args.ess_draws, args.seed)
            r.update(gpu=gpu, power_limit_and_max_sm_clock=power, wall_s=round(time.time() - t0, 1))
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
