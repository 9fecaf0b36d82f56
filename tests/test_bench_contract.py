"""bench.py contract on the CPU: the reference arm (`--impl reference`: the SciPy-BFGS port of the reference's step, one
process per chain) prints ONE JSON line with the keys the driver reads, and the GPU arm refuses to run without a device
instead of falling back."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dim", "6", "--ref-draws-per-step", "15", "--adapt-warmup", "60", "--ref-procs", "2"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "chain_draws_per_sec" and line["unit"] == "chain-draws/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 2
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True,
                         text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_dump_outputs_fit_their_share_and_keep_a_fixed_sample_of_chains():
    """`--dump-outputs`: every workload's arrays fit its share of DUMP_MB (64 MB in all, .npy headers included); a larger
    sampler keeps a seeded sample of chains, the same in theta and the accept counts and the same run after run."""
    import types
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    assert sum(bench.DUMP_MB.values()) < 64
    B, D = 4096, 256
    smp = types.SimpleNamespace(_theta=torch.arange(B * D, dtype=torch.float64).reshape(B, D),
                                _accept_count=torch.arange(B))
    out = bench.last_step_outputs("c4", smp)
    th, acc = out["c4_theta"], out["c4_accept_count"]
    assert th.dtype == acc.dtype == np.float64 and th.nbytes + acc.nbytes <= bench.DUMP_MB["c4"] * 10 ** 6
    assert 0 < len(acc) < B and th.shape == (len(acc), D) and len(np.unique(acc)) == len(acc)
    assert np.array_equal(th[:, 0] / D, acc)                           # the same chains in both files
    again = bench.last_step_outputs("c4", smp)
    assert all(np.array_equal(out[k], again[k]) for k in out)
    small = types.SimpleNamespace(_theta=torch.ones(64, 100, dtype=torch.float32), _accept_count=torch.zeros(64, dtype=torch.int64))
    out = bench.last_step_outputs("c2", small)                          # under its share: every chain
    assert out["c2_theta"].dtype == np.float32 and out["c2_theta"].shape == (64, 100) and out["c2_accept_count"].shape == (64,)
    # the headline workload at its default size is written whole
    assert 65_536 * (100 * 8 + 8) <= bench.DUMP_MB["c2"] * 10 ** 6
    ref = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert ref.returncode != 0 and "--dump-outputs needs --impl b200" in ref.stderr


def test_normals_accounting_follows_the_lane_kernels_element_map():
    """`roofline.normals.generated_per_chain_draw` against a walk of the lane kernel's sweep (csrc/klhr_lane.cuh): trip t
    covers the coordinate quads at e = 32 (t // 2) + 4 (t % 2) + 8 r, r = 0..3, and draws 16 normals whatever part of it
    lies below D; a last trip of a single quad is split between the chain's two lanes and draws 4 (kTail)."""
    sys.path.insert(0, str(ROOT))
    import bench
    for D in range(1, 300):
        trips = [t for t in range(2 * (D // 32 + 1)) if 32 * (t // 2) + 4 * (t % 2) < D]
        rem = D % 32
        tail = 1 <= rem <= 4
        assert len(trips) == 2 * (D // 32) + (2 if rem > 4 else (1 if rem else 0))
        if tail:
            last = trips.pop()
            quads = [r for r in range(4) if 32 * (last // 2) + 4 * (last % 2) + 8 * r < D]
            assert quads == [0]                                    # one quad: coordinates D - rem .. D - 1
        assert bench.lane_normals_generated(D) == 16 * len(trips) + (4 if tail else 0)
        assert bench.lane_normals_generated(D) >= D
