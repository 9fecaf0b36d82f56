#!/usr/bin/env python
"""Benchmark of the KLHR hot path (BASELINE.json metric: chain-draws/sec, ESS/sec, % roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[1]): stan/ill-normal, D = 100 diagonal Gaussian, 65 536 chains per GPU,
Gaussian line family, fp64, reference warm-up schedule [50, 150, 350, 1000] run (and timed separately) before the
timed region.  One "step" = every chain advanced by --draws-per-step KLHR draws (one `klhr_run` launch).  N > 1
shards chains over ranks (weak scaling, no collective in the step).

The JSON line also carries
  peaks     FP64 / FP32 FMA, FP64 DMMA and Philox+Box-Muller normals per second measured in this process with the
            micro-kernels of csrc/klhr_probe.cu (BASELINE.md section 3: the vector peaks are not in MEASURED_PEAKS.json);
  roofline  the slower of (FP64 flops executed / measured FP64 peak) and (HBM bytes / measured HBM peak), plus the
            direction-normal rate against its measured ceiling (the resource the kernel actually runs against);
  adapt     the warm-up phase: wall time of the 1000 adaptation draws including the pooled all-reduce at each of the
            4 window closures (the only collective of the path) -- max over ranks;
  e2e       the metric through the public sampler API from pinned HOST buffers; e2e_sample: MCMCBase.sample's own
            contract (every draw returned, mcmc.py:31-37) streamed to pinned host memory;
  configs   BASELINE.json configs[2..4] (funnel + sinh-arcsinh family, dense corr-normal D = 256, arK T = 10 000)
            measured the same way, --steps timed steps each, with its roofline and its adaptation phase (c5 is the
            config whose closure all-reduce runs over every rank of --gpus N).

`--dump-outputs DIR` writes, on rank 0, what the last timed step of each workload left to its caller -- the chain states
(`<tag>_theta.npy`, chains x D, the sampler's dtype) and the per-chain accept counts (`<tag>_accept_count.npy`,
float64) -- for comparing two builds output for output: every input derives from a fixed seed, so the same arguments
give the same inputs.  At most 64 MB in all: a workload whose arrays exceed its share keeps a fixed, seeded sample of
chains (the same chains in both of its files).

`--impl reference` times the reference's own CPU implementation of the same step (the SciPy-BFGS single-chain port in
oracle/ref_port.py, one process per chain on all host cores, like reference run_experiments:27) -- /root/reference
itself is pure Python and is not present on the GPU box, so `cpu_baseline.kind` is "port".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "chain_draws_per_sec"
UNIT = "chain-draws/s"
SEED = 20261018


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=65_536, help="chains per GPU")
    ap.add_argument("--dim", type=int, default=100)
    ap.add_argument("--draws-per-step", type=int, default=1000)
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--adapt-warmup", type=int, default=1000, help="sampler warm-up draws (timed separately)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only (skip configs c3..c5)")
    ap.add_argument("--profile-region", default="", choices=["", "c2", "c3", "c3_dims11", "c4", "c5"],
                    help="cudaProfilerStart/Stop around the first timed launch of that config (ncu --profile-from-start off)")
    ap.add_argument("--ref-draws-per-step", type=int, default=400)
    ap.add_argument("--ref-procs", type=int, default=0, help="0 = all host cores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of each workload to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# =============================================================================== CPU reference arm
def _ref_worker(conn, dim, seed, adapt_warmup):
    """One OS process = one chain of the reference algorithm (oracle port, SciPy BFGS)."""
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"                     # one core per chain; avoids BLAS oversubscription
    import numpy as np  # noqa: F401
    from oracle.bsmodel import BSModel
    from oracle.ref_port import ChainSampler
    model = BSModel(stan_file="stan/ill-normal.stan", data={"D": dim})
    s = ChainSampler(model, family="gauss", seed=seed, warmup=adapt_warmup)
    for _ in range(adapt_warmup):
        s.draw()
    conn.send("ready")
    while True:
        n = conn.recv()
        if n <= 0:
            break
        t0 = time.perf_counter()
        for _ in range(n):
            s.draw()
        conn.send(time.perf_counter() - t0)
    conn.close()


class RefPool:
    def __init__(self, procs, dim, adapt_warmup):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.conns, self.procs = [], []
        for i in range(procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_ref_worker, args=(b, dim, SEED + i, adapt_warmup), daemon=True)
            p.start()
            self.conns.append(a)
            self.procs.append(p)
        for c in self.conns:
            assert c.recv() == "ready"

    def step(self, n):
        t0 = time.perf_counter()
        for c in self.conns:
            c.send(n)
        for c in self.conns:
            c.recv()
        return time.perf_counter() - t0

    def close(self):
        for c in self.conns:
            c.send(0)
        for p in self.procs:
            p.join(timeout=10)


def cpu_baseline(dim, draws, procs, adapt_warmup, steps=1, warmup=0):
    procs = procs or (os.cpu_count() or 1)
    pool = RefPool(procs, dim, adapt_warmup)
    try:
        for _ in range(warmup):
            pool.step(max(1, draws // 4))
        times = [pool.step(draws) for _ in range(steps)]
    finally:
        pool.close()
    total = sum(times)
    return dict(value=procs * draws * steps / total, unit=UNIT, cores=procs, kind="port",
                sample=f"{procs} processes x 1 chain (oracle/ref_port.py, SciPy BFGS, analytic NumPy model "
                       f"shim; BridgeStan absent), {adapt_warmup} warm-up draws untimed, then "
                       f"{steps} x {draws} draws each, wall clock"), total / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, sec_per_step = cpu_baseline(args.dim, args.ref_draws_per_step, args.ref_procs, args.adapt_warmup,
                                    steps=args.steps, warmup=args.warmup)
    line = {
        "metric": METRIC, "value": cb["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"stan/ill-normal D={args.dim} KLHR Gaussian line fit, one chain per host core",
                   "chains": cb["cores"], "draws_per_step": args.ref_draws_per_step},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# =============================================================================== clocks
class ClockSampler:
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.rows = None
        try:
            import shutil
            exe = shutil.which("nvidia-smi") or "nvidia-smi"
            # full path + close_fds=False: CPython then starts the child with posix_spawn instead of fork -- a fork()
            # makes every later multi-threaded LAPACK call of this process hang when the bench runs under ncu
            # (tools/dev/t_ncu.py reproduces it)
            self.proc = subprocess.Popen(
                [exe, f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(gpu_index)], stdout=self.tmp, stderr=subprocess.DEVNULL, close_fds=False)
            import atexit
            atexit.register(self._kill)                  # never leave the sampler behind if the bench dies
        except OSError:
            pass

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()

    def stop(self):
        import datetime
        if self.proc is None:
            self.rows = []
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        rows = []
        for r in Path(self.tmp.name).read_text().splitlines():
            f = r.split(",")
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), [x.strip().lower().startswith("active") for x in f[4:8]]))
            except ValueError:
                continue
        os.unlink(self.tmp.name)
        self.rows = rows

    def window(self, t_begin, t_end):
        """Median SM clock and active throttle reasons over the samples stamped inside [t_begin, t_end]
        (time.time() stamps); all samples if the window holds none (a region shorter than the 50 ms period)."""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        rows = self.rows or []
        inside = [r for r in rows if t_begin - 0.05 <= r[0] <= t_end + 0.05]
        use = inside or rows
        if not use:
            return out
        sm = sorted(r[1] for r in use)
        reasons = sorted({self.NAMES[k] for r in use for k in range(4) if r[3][k]})
        out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=use[-1][2], reasons=reasons, samples=len(inside),
                   samples_total=len(rows))
        return out


# =============================================================================== B200 arm
def ark_series(T=10_000, K=5):
    """BASELINE.md section 4 config 5: y_t = 0.2 + sum_k beta_k y_{t-6+k} + 0.5 eps_t, seeded, 500 burn-in dropped."""
    import numpy as np
    beta = np.array([0.05, -0.10, 0.15, -0.20, 0.60])
    rng = np.random.default_rng(20261018)
    eps = rng.normal(size=T + 500)
    y = np.zeros(T + 500)
    for t in range(K, T + 500):
        y[t] = 0.2 + beta @ y[t - K:t] + 0.5 * eps[t]
    return y[500:]


DUMP_MB = {"c2": 55, "c3": 2, "c3_dims11": 2, "c4": 2, "c5": 2}    # shares of the <= 64 MB --dump-outputs writes


def last_step_outputs(tag, sampler):
    """`<tag>_theta` and `<tag>_accept_count` of `sampler` as host arrays (the sampler's dtype / float64); a sampler
    whose two arrays exceed the workload's share of DUMP_MB keeps the same fixed, seeded sample of chains in both."""
    import numpy as np
    import torch
    theta, acc = sampler._theta, sampler._accept_count
    rows = DUMP_MB[tag] * 10 ** 6 // (theta.shape[1] * theta.element_size() + 8)
    if theta.shape[0] > rows:
        idx = np.sort(np.random.default_rng(SEED).choice(theta.shape[0], rows, replace=False))
        idx = torch.as_tensor(idx, device=theta.device)
        theta, acc = theta[idx], acc[idx]
    return {f"{tag}_theta": theta.cpu().numpy(), f"{tag}_accept_count": acc.double().cpu().numpy()}


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import klhr_b200 as kb
    from klhr_b200 import engine
    from klhr_b200.diagnostics import chain_summary

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    # started first: nvidia-smi can take a second to spin up on a fresh box, and only samples stamped inside the
    # timed regions are used
    clocks = ClockSampler(local) if rank == 0 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    B, D, S, K, W = args.chains, args.dim, args.draws_per_step, args.steps, args.warmup
    rb = 8 if dtype == torch.float64 else 4
    launches = [0]                                   # klhr_run launches inside timed regions (gpu_launches)
    dumps = None
    if args.dump_outputs and rank == 0:
        dumps = {}
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)

    trace_on = bool(os.environ.get("KLHR_BENCH_TRACE"))
    t_start = time.time()

    def trace(msg):                                  # progress on stderr (KLHR_BENCH_TRACE=1): where a run under a profiler spends its time
        if trace_on and rank == 0:
            print(f"[bench +{time.time() - t_start:7.1f}s] {msg}", file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # ---------------------------------------------------------------- peaks (micro-kernels, this process, this GPU)
    peaks = {
        "fp64_fma_tflops": 2e-12 * engine.peak_probe("fp64_fma", dev),
        "fp32_fma_tflops": 2e-12 * engine.peak_probe("fp32_fma", dev),
        "fp64_dmma_tflops": 16e-12 * engine.peak_probe("fp64_dmma", dev),
        "normals_per_s": engine.peak_probe("normals", dev),
        "how": "csrc/klhr_probe.cu, 8 CTAs x 256 threads per SM, best of 5 launches, CUDA events; normals = "
               "Philox4x32-10 + fp32 Box-Muller exactly as in the step kernels",
    }
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        hbm_peak, hbm_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    peaks["hbm_gbs"] = hbm_peak
    prof = {}
    pp = ROOT / "profiles" / "ncu_counts.json"          # per-chain-draw instruction / flop / DRAM counts from ncu captures
    if pp.exists():
        prof = json.loads(pp.read_text())

    def adapt_phase(make_sampler, n):
        """The warm-up: n adaptation draws incl. the pooled all-reduce + host eigendecomposition at each closure.
        Timed twice on two identically configured samplers: the first pass is the process's first use of these
        kernels, of LAPACK and of the NCCL communicator (lazy module loading, allocator growth: reported as
        `cold_phase_s`); the second is the phase itself (`phase_s`), like every other timed region after warm-up."""
        out = []
        sampler = None
        for k_pass in range(2):
            del sampler
            trace(f"adaptation pass {k_pass}")
            sampler = make_sampler()
            barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sampler.run(n)
            torch.cuda.synchronize()
            out.append(max_over_ranks(time.perf_counter() - t0))
        return sampler, out[1], out[0]

    def timed_steps(sampler, draws, k, w, do_flush, tag=""):
        """k launches of `draws` draws, each bracketed by CUDA events on the launching stream; max over ranks of
        the summed device time.  Returns (total_ms, wall window)."""
        trace(f"timed steps {tag or '-'}: {w} warm-up + {k} x {draws} draws")
        for _ in range(w):
            sampler.run(draws)
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        barrier()
        torch.cuda.synchronize()
        w0 = time.time()
        for i in range(k):
            if do_flush:
                flush.zero_()                      # L2 flush between timed iterations
            prof_this = bool(tag) and args.profile_region == tag and i == 0
            if prof_this:
                torch.cuda.synchronize()
                torch.cuda.profiler.start()
            evs[i][0].record()
            sampler.run(draws)                     # ONE klhr_run launch: all chains x `draws` draws
            evs[i][1].record()
            if prof_this:
                torch.cuda.synchronize()
                torch.cuda.profiler.stop()
        torch.cuda.synchronize()
        barrier()
        w1 = time.time()
        launches[0] += k
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in evs)), (w0, w1)

    def fp64_roofline(name, value_per_gpu, hbm_bytes_per_draw, peak_tflops, peak_name, kernel, note, alg_flops=None):
        """Slower of FP64 and HBM (north star); flops per chain-draw are COUNTED by ncu on the same kernel and
        configuration (profiles/ncu_counts.json: (dadd + dmul + 2 dfma [+ 512 dmma]) / chain-draws)."""
        c = prof.get(name, {})
        flops = c.get("fp64_flops_per_draw")
        out = {"kernel": kernel, "hbm_bytes_per_chain_draw": hbm_bytes_per_draw,
               "hbm_gbs_achieved": hbm_bytes_per_draw * value_per_gpu / 1e9, "hbm_frac": hbm_bytes_per_draw * value_per_gpu / 1e9 / hbm_peak,
               "fp64_flops_per_chain_draw": flops, "warp_instructions_per_chain_draw": c.get("warp_inst_per_draw"),
               "issue_active_pct": c.get("issue_active_pct"), "traffic": c.get("dram_bytes_per_launch"),
               "traffic_launch": c.get("launch"), "counts_source": "profiles/ncu_counts.json (ncu --set full, same kernel and shape)" if c else None,
               "note": note}
        if flops:
            ach = flops * value_per_gpu / 1e12
            t_f, t_b = flops / (peak_tflops * 1e12), hbm_bytes_per_draw / (hbm_peak * 1e9)
            out.update(bound="fp64" if t_f >= t_b else "hbm", achieved=ach if t_f >= t_b else out["hbm_gbs_achieved"],
                       peak=peak_tflops if t_f >= t_b else hbm_peak, unit="TFLOP/s" if t_f >= t_b else "GB/s",
                       frac=(ach / peak_tflops) if t_f >= t_b else out["hbm_frac"], peak_source=f"measured in this run ({peak_name})" if t_f >= t_b else hbm_src)
        else:
            out.update(bound="hbm", achieved=out["hbm_gbs_achieved"], peak=hbm_peak, unit="GB/s", frac=out["hbm_frac"],
                       peak_source=hbm_src)
        if alg_flops:        # SURVEY 8(d)'s per-unit figure next to the flops the kernel really executes
            out["algorithmic_flops_per_chain_draw"] = alg_flops
            out["algorithmic_tflops"] = alg_flops * value_per_gpu / 1e12
            out["algorithmic_frac"] = alg_flops * value_per_gpu / 1e12 / peak_tflops
        return out

    # =============================================================== headline: ill-normal D = 100 (configs[1])
    model = kb.BSModel(stan_file="stan/ill-normal.stan", data={"D": D}, device=dev)
    sampler, adapt_s, adapt_cold_s = adapt_phase(
        lambda: kb.KLHR(model, seed=SEED, chains=B, warmup=args.adapt_warmup, windowsize=50, windowscale=2,
                        dtype=dtype, device=dev), args.adapt_warmup)     # windows close at 50,150,350,1000 (+ all-reduce)
    total_ms, (wall0, wall1) = timed_steps(sampler, S, K, W, True, "c2")
    if dumps is not None:
        dumps.update(last_step_outputs("c2", sampler))          # before the e2e arm moves the chains on
    value = world * B * S * K / (total_ms * 1e-3)
    info = kb.launch_info(model, sampler._fit, dtype=dtype, free_running=True, accumulate=False, device=dev)

    # ---------------------------------------------------------------- end-to-end arm (host buffers)
    # Every step: H2D of the step's start state from pinned host memory, S draws through the public
    # sampler API, D2H of the final state and the accept counts.  Two device state buffers and three
    # streams pipeline the copies of step k +- 1 under the kernel of step k (steps are independent
    # jobs: each starts from the host start state), so PCIe time overlaps compute.
    start_host = torch.empty(B, D, dtype=dtype).pin_memory()
    start_host.copy_(sampler._theta)
    out_host = [torch.empty(B, D, dtype=dtype).pin_memory() for _ in range(2)]
    acc_host = [torch.empty(B, dtype=torch.int64).pin_memory() for _ in range(2)]
    bufs = [sampler._theta, torch.empty_like(sampler._theta)]
    s_in, s_run, s_out = torch.cuda.Stream(dev), torch.cuda.current_stream(dev), torch.cuda.Stream(dev)

    def e2e_steps(n):
        ev_in = [torch.cuda.Event() for _ in range(n)]
        ev_run = [torch.cuda.Event() for _ in range(n)]
        ev_out = [torch.cuda.Event() for _ in range(n)]
        for k in range(n):
            buf = bufs[k % 2]
            with torch.cuda.stream(s_in):
                if k >= 2:
                    s_in.wait_event(ev_out[k - 2])               # buffer free again once step k-2 was read back
                buf.copy_(start_host, non_blocking=True)         # H2D of the step's start state
                ev_in[k].record(s_in)
            s_run.wait_event(ev_in[k])
            sampler.swap_state(buf)
            sampler.run(S)                                       # public sampler API, one launch
            ev_run[k].record(s_run)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_run[k])
                out_host[k % 2].copy_(buf, non_blocking=True)    # D2H of the step's result
                acc_host[k % 2].copy_(sampler._accept_count, non_blocking=True)
                ev_out[k].record(s_out)
        torch.cuda.synchronize()

    e2e_steps(min(W, 2))
    barrier()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_steps(K)
    e1.record()
    torch.cuda.synchronize()
    barrier()
    launches[0] += K
    sampler.swap_state(bufs[0])
    e2e_value = world * B * S * K / (max_over_ranks(e0.elapsed_time(e1)) * 1e-3)

    # ---------------------------------------------------------------- e2e of MCMCBase.sample's own contract
    # sample(M) returns EVERY draw (mcmc.py:31-37): 800 B per chain-draw must cross PCIe, which bounds the
    # host-visible rate; the rows are streamed to pinned host memory in chunks, D2H of chunk k-1 under the kernel
    # of chunk k (KLHR.sample(out=...)).
    M_rows = 17
    rows_host = torch.empty(M_rows, B, D, dtype=dtype).pin_memory()
    sampler.sample(M_rows, thin=1, out=rows_host, chunk_rows=4)          # warm-up (allocations, first touch)
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sampler.sample(M_rows, thin=1, out=rows_host, chunk_rows=4)
    torch.cuda.synchronize()
    samp_s = max_over_ranks(time.perf_counter() - t0)
    launches[0] += 4
    e2e_sample = {"value": world * B * (M_rows - 1) / samp_s, "unit": UNIT, "rows": M_rows, "thin": 1,
                  "d2h_bytes_per_call": M_rows * B * D * rb, "d2h_gbs_per_gpu": M_rows * B * D * rb / samp_s / 1e9,
                  "bound": f"PCIe D2H: {D * rb} B per chain-draw",
                  "api": "KLHR.sample(M, thin=1, out=pinned host tensor): every draw returned (mcmc.py:31-37), chunks of 4 rows "
                         "double-buffered on the device, D2H on a copy stream under the next chunk's kernel; host wall clock"}
    del rows_host

    # ---------------------------------------------------------------- ESS per draw (diagnostic pass)
    ess = None
    if not args.no_ess:
        S_ess = max(S, 2000)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        s1, s2 = sampler.run(S_ess, chain_stats=True)
        a1.record()
        torch.cuda.synchronize()
        summ = chain_summary(s1, s2, S_ess)
        truth = torch.arange(1, D + 1, dtype=torch.float64, device=dev) ** 2 / D      # var_i = i^2 / D
        zmean = (summ["mean"].abs() / summ["mcse_mean"]).max()
        zvar = ((summ["var"] - truth).abs() / summ["mcse_var"]).max()
        ess_min = float(summ["ess"].min())
        ms = a0.elapsed_time(a1)
        # ESS per draw is a property of the chains (all kernels draw the same streams); the pass that
        # measures it needs per-chain sums and therefore runs on the accumulating octet kernel, so
        # ESS/sec of the production path = ESS per chain-draw x the timed chain-draws/sec
        ess = {"min_ess_per_sec": (ess_min / (B * S_ess)) * value, "min_ess_per_draw": ess_min / (B * S_ess),
               "min_ess_per_sec_of_stats_pass": world * ess_min / (ms * 1e-3),
               "draws_per_chain": S_ess, "estimator": "between-chain variance of chain means, B independent chains",
               "max_abs_z_mean": float(zmean), "max_abs_z_var": float(zvar),
               "acceptance": sampler.acceptance_probability}
        del s1, s2

    kernel_name = ("klhr::lane_kernel (csrc/klhr_lane.cuh)" if info["threads"] in (32, 64) and info["smem"] > 30000 else
                   "klhr::tile_kernel (csrc/klhr_tile.cuh)" if info["threads"] == 32 else "klhr::step_kernel (csrc/klhr_step.cuh)")
    n_gen = lane_normals_generated(D)
    roof = fp64_roofline(
        "c2", value / world, (2 * D * rb + 16) / S, peaks["fp64_fma_tflops"], "peaks.fp64_fma_tflops", kernel_name,
        f"S = {S} draws are fused per launch with theta resident in shared memory: HBM sees one read and one write of "
        f"theta per LAUNCH, i.e. (2 D {rb} + 16) / S bytes per chain-draw (SURVEY 8d); the FP64 side counts the flops the "
        "kernel executes (closed-form quadratic fit, not the reference-equivalent 14 evaluations); neither is what "
        "bounds the kernel -- see `normals`")
    roof["normals"] = {"generated_per_chain_draw": n_gen, "used_per_chain_draw": D,
                       "achieved_per_s": n_gen * value / world, "peak_per_s": peaks["normals_per_s"],
                       "frac": n_gen * value / world / peaks["normals_per_s"],
                       "note": "the D direction normals per chain-draw (klhr.py:143-153) are the dominant instruction stream; "
                               "peak = the same Philox4x32-10 + Box-Muller code alone at full occupancy"}
    roof["draws_fused_per_launch"] = S

    line = None
    cfg_lines = {}
    # =============================================================== configs[2..4]
    if not args.no_configs:
        def run_config(tag, workload, make_sampler, draws, hbm_bytes_per_draw, peak_tflops, peak_name, kernel, note, extra=None,
                       alg_flops=None):
            smp, a_s, a_cold = adapt_phase(make_sampler, 1000)
            a_draws = world * smp.chains * 1000
            t_ms, (c0_, c1_) = timed_steps(smp, draws, K, max(W, 3), False, tag)
            if dumps is not None:
                dumps.update(last_step_outputs(tag, smp))
            val = world * smp.chains * draws * K / (t_ms * 1e-3)
            trace(f"{tag}: timed steps done")
            ev0 = int(smp._evals_total.item())
            smp.run(draws)
            evals = (int(smp._evals_total.item()) - ev0) / (smp.chains * draws)
            trace(f"{tag}: evaluation count done")
            out = {"workload": workload, "value": val, "unit": UNIT, "ms_per_step": t_ms / K, "steps": K,
                   "draws_per_step": draws, "chains_per_gpu": smp.chains, "acceptance": smp.acceptance_probability,
                   "line_evaluations_per_draw": evals,
                   "adapt": {"draws": 1000, "closures": smp._windowedadaptation.closures, "phase_s": a_s, "cold_phase_s": a_cold,
                             "chain_draws_per_s": a_draws / a_s, "frac_of_steady_state": a_draws / a_s / val},
                   "roofline": fp64_roofline(tag, val / world, hbm_bytes_per_draw / draws, peak_tflops, peak_name, kernel, note, alg_flops),
                   "window": (c0_, c1_), "inputs": "state (chains x D fp64) larger than L2" if smp.chains * smp.D * 8 > 126e6
                   else "state smaller than L2; kernels keep it on-chip for the whole launch, so no flush is needed between steps"}
            if extra:
                out.update(extra(smp))
            del smp
            torch.cuda.empty_cache()
            return out

        fm = kb.BSModel(stan_file="stan/funnel.stan", data={"D": 1}, device=dev)
        cfg_lines["c3"] = run_config(
            "c3", "stan/funnel dims=2 (stan/funnel.json), KLHRSINH sinh-arcsinh line fit, overrelaxed=False, 262144 chains/GPU, fp64",
            lambda: kb.KLHRSINH(fm, seed=SEED, chains=262_144, warmup=1000, overrelaxed=False, device=dev), 20,
            2 * 2 * 8 + 16, peaks["fp64_fma_tflops"], "peaks.fp64_fma_tflops", "klhr::chain_kernel (csrc/klhr_chain.cuh)",
            "thread-per-chain 4-parameter Newton fit on the O(1) line restriction; bound by fp64 arithmetic incl. exp/log",
        )
        fm11 = kb.BSModel(stan_file="stan/funnel.stan", data={"D": 10}, device=dev)
        cfg_lines["c3_dims11"] = run_config(
            "c3_dims11", "stan/funnel dims=11 (the 10-D funnel of write_experiments.py:127), KLHRSINH sinh-arcsinh line fit, overrelaxed=False, "
                         "262144 chains/GPU, fp64",
            lambda: kb.KLHRSINH(fm11, seed=SEED, chains=262_144, warmup=1000, overrelaxed=False, device=dev), 20,
            2 * 11 * 8 + 16, peaks["fp64_fma_tflops"], "peaks.fp64_fma_tflops", "klhr::chain_kernel (csrc/klhr_chain.cuh)",
            "as c3; the elementwise gradient clip walks the 11 components only when its bound trips")
        trace("c4: building the model (precision, Cholesky factor, packing)")
        cm = kb.BSModel(stan_file="stan/corr-normal.stan", data={"N": 256, "rho": 0.9}, device=dev)
        trace("c4: model built")
        cfg_lines["c4"] = run_config(
            "c4", "stan/corr-normal D=256 dense precision (Sigma_ij = 0.9^|i-j|), KLHR Gaussian line fit, 16384 chains/GPU, fp64",
            lambda: kb.KLHR(cm, seed=SEED, chains=16_384, warmup=1000, device=dev), 100,
            2 * 256 * 8 + 16, peaks["fp64_dmma_tflops"], "peaks.fp64_dmma_tflops", "klhr::dense_ws_kernel (csrc/klhr_densews.cuh + klhr_densek.cuh, DMMA)",
            "V = L' rho (P = L L') for the 32 chains of a CTA on mma.sync.m8n8k4.f64 (8 tensor warps), w = L' theta carried along, directions / fit / move on 8 producer warps: the "
            "triangular product executes ~D^2 flops per chain-draw where P rho needs 2 D^2 = 131 kflop (SURVEY 8d, `algorithmic_*`)",
            alg_flops=2 * 256 * 256)
        ak = kb.BSModel(stan_file="stan/arK.stan", data={"K": 5, "T": 10_000, "y": ark_series().tolist()}, device=dev)

        def ark_extra(smp):
            s1_, s2_ = smp.run(200, chain_stats=True)
            mean = chain_summary(s1_, s2_, 200)["mean"].cpu().numpy()
            if world > 1:
                mt = torch.as_tensor(mean, device=dev)
                dist.all_reduce(mt)
                mean = (mt / world).cpu().numpy()
            return {"posterior_mean": [round(float(x), 4) for x in mean],
                    "generating_values": [0.2, 0.05, -0.10, 0.15, -0.20, 0.60, round(float(np.log(0.5)), 4)]}
        cfg_lines["c5"] = run_config(
            "c5", f"stan/arK K=5 T=10000 synthetic (BASELINE.md 4.5), KLHR Gaussian line fit, 131072 chains/GPU "
                  f"({world * 131_072} chains over {world} GPU(s)), pooled windowed-adaptation all-reduce at 4 closures",
            lambda: kb.KLHR(ak, seed=SEED, chains=131_072, warmup=1000, device=dev), 100,
            2 * 7 * 8 + 16, peaks["fp64_fma_tflops"], "peaks.fp64_fma_tflops", "klhr::chain_kernel (csrc/klhr_chain.cuh)",
            "line restriction through the Gram matrix X'X (6x6), X'y, y'y: ~100 flop per evaluation instead of 2.6e5 for the "
            "direct T-loop (SURVEY 8a M6); the adaptation phase contains the only collective of the path", ark_extra)

    if clocks:
        clocks.stop()
    if rank == 0:
        clk = clocks.window(wall0, wall1)
        for c in cfg_lines.values():
            c["clocks"] = clocks.window(*c.pop("window"))
        adapt_draws = world * B * args.adapt_warmup
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"stan/ill-normal D={D} diagonal Gaussian, {B} chains/GPU, KLHR Gaussian "
                                   f"line fit, {S} draws per step (one launch)",
                       "chains_per_gpu": B, "global_chains": world * B, "dim": D, "draws_per_step": S,
                       "adapt_warmup_draws": args.adapt_warmup, "windows": sampler._windowedadaptation.closures,
                       "parallelism": f"chains sharded over {world} GPU(s), no collective in the step; one all-reduce of "
                                      "pooled moment / PCA sums per window closure (inside `adapt`)",
                       "l2": "256 MB memset between timed steps (state 52 MB < 126 MB L2); excluded from "
                             "ms_per_step by per-step CUDA events", "seed": SEED, "launch": info},
            "clocks": clk,
            "peaks": peaks,
            "adapt": {"draws": args.adapt_warmup, "closures": sampler._windowedadaptation.closures, "phase_s": adapt_s,
                      "cold_phase_s": adapt_cold_s,
                      "chain_draws_per_s": adapt_draws / adapt_s, "frac_of_steady_state": adapt_draws / adapt_s / value,
                      "contains": "adaptation launches, pooled moment/PCA accumulation, 4 x all-reduce(SUM, fp64) of "
                                  f"(2 + 4 D + D^2) doubles = {(2 + 4 * D + D * D) * 8} B over {world} rank(s), host eigh; wall clock, max over ranks"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * D * rb,
                    "d2h_bytes_per_step": B * D * rb + B * 8,
                    "api": "KLHR.run(draws_per_step) from a pinned host start state, final state + accept counts "
                           "read back every step; copies of neighbouring steps overlap the kernel (2 buffers, 3 streams)"},
            "e2e_sample": e2e_sample,
            "gpu_launches": launches[0],
            "roofline": roof,
            "ess": ess,
            "configs": cfg_lines,
        }
        if world == 1 and not args.no_cpu_baseline:
            cb, _ = cpu_baseline(D, 2000, args.ref_procs, args.adapt_warmup)
            line["cpu_baseline"] = cb
        for name, a in (dumps or {}).items():
            np.save(Path(args.dump_outputs) / f"{name}.npy", a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def lane_normals_generated(D):
    """Direction normals the lane kernel draws per chain-draw (csrc/klhr_lane.cuh): 16 per trip of its sweep (4 Philox
    blocks; trip t covers the 4 coordinate quads at 32 (t // 2) + 4 (t % 2) + 8 r); a last trip of ONE quad (D mod 32 in
    1..4, kTail) is split between the chain's two lanes instead and draws only the 4 cosine-branch normals it needs."""
    rem = D % 32
    return 32 * (D // 32) + (4 if 1 <= rem <= 4 else (32 if rem > 4 else 0))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
