"""Helpers shared by the GPU parity tests (CUDA path through the C ABI vs the oracle)."""
import numpy as np
import torch

import klhr_b200 as kb
from oracle import batched, stan_models


def device():
    return torch.device("cuda", 0)


def up(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=device()).contiguous()


def fit_pair(family, dtype=torch.float64, **kw):
    """(klhr_b200.FitConfig, oracle FitConfig) with identical settings."""
    if family == "subsinh":
        family = "sinh"
        kw = dict(kw, fix_d=True)
    if family == "sinh":
        base = dict(family="sinh", tol=1e-10, scale_clip=300.0, n2=48, kmax=32)
        base["grad_clip"] = 1e15 if kw.get("fix_d") else kw.get("scale_clip", 300.0)   # klhr_sinh.py:158-161 / sub_klhr_sinh.py:152-154
    else:
        base = dict(family="gauss")
    base.update(kw)
    k = kb.FitConfig(**base).for_dtype(dtype)
    o = batched.FitConfig(**{f: getattr(k, f) for f in
                             ("family", "N", "initscale", "tol", "scale_clip", "n1", "n2", "nb", "kmax", "fix_d", "grad_clip", "gtol1",
                              "gtol2", "step_cap", "c1", "basin")})
    if dtype == torch.float32:
        o.eps = float(np.finfo(np.float32).eps)
    return k, o


# replay tapes of the unmodified reference (tests/golden) by line family
GAUSS_TAPES = ["normal_d2_klhr", "normal_d2_klhr_method2", "illnormal_d100_klhr",
               "illnormal_d100_klhr_tight", "corrnormal_n50_klhr", "ar1_n100_klhr",
               "funnel_d2_klhr", "funnel_d2_klhr_tight", "funnel_d11_klhr_tight",
               "ark_t200_klhr_tight", "rosenbrock_d4_klhr_tight", "earnings_klhr_tight",
               "illnormal_d20_klhr_scaledir"]
SINH_TAPES = ["funnel_d2_sinh", "funnel_d2_sinh_tight", "ark_t200_sinh", "rosenbrock_d4_sinh", "earnings_sinh",
              "funnel_d2_sinh_scaledir_method1",
              "funnel_d2_subsinh_tight", "rosenbrock_d4_subsinh"]     # subsinh: SUBKLHRSINH, d = 1 (sub_klhr_sinh.py)

DIAG_MODELS = ("normal", "ill-normal")     # targets the tile kernel covers (csrc/klhr_tile.cuh)


def replay_both(model_name, data, family, theta, rho, z_init, z_prop, u, init4=None,
                dtype=torch.float64, xw=None, **fitkw):
    """Run the CUDA replay step and the batched oracle on the same inputs."""
    force_octet = fitkw.pop("force_octet", False)
    kfit, ofit = fit_pair(family, dtype, **fitkw)
    kfit.force_octet = force_octet
    if xw is not None:
        kfit.x, kfit.w = np.array(xw[0]), np.array(xw[1])
    model = kb.BSModel(stan_file=f"stan/{model_name}.stan", data=data, device=device())
    th = up(theta, dtype)
    tr = kb.step_replay(model, kfit, th, up(rho, dtype), up(z_init, dtype), up(z_prop, dtype), up(u, dtype),
                        init4=up(init4, dtype) if init4 is not None else None)
    torch.cuda.synchronize()
    gpu = dict(eta=tr.eta[0].double().cpu().numpy(), zp=tr.zp[0].double().cpu().numpy(),
               r=tr.r[0].double().cpu().numpy(), accept=tr.accept[0].cpu().numpy().astype(bool),
               evals=tr.evals[0].cpu().numpy(), theta=th.double().cpu().numpy())
    om = stan_models.make_model(model_name, data)
    if dtype == torch.float32:   # the oracle sees the same rounded inputs
        f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32).astype(np.float64)
        theta, rho, z_init, z_prop, u, init4 = map(f32, (theta, rho, z_init, z_prop, u, init4))
    ref = batched.step(om, np.asarray(theta, dtype=np.float64), np.asarray(rho, dtype=np.float64),
                       np.asarray(z_init, dtype=np.float64), np.asarray(z_prop, dtype=np.float64),
                       np.asarray(u, dtype=np.float64), ofit, init4=init4,
                       xw=(kfit.x, kfit.w))
    return gpu, ref


def _pad(D, rb):
    """pad_dim of csrc/klhr_step.cuh."""
    mod = 16 if rb == 8 else 32
    p = -(-D // mod) * mod + 8
    return p - mod if p - mod >= D else p


def assert_kernel(model, kfit, dtype, want, accumulate=False, free_running=True):
    """The launch plan of ``want`` (csrc: launch_lane / launch_tile_typed / chain_smem_bytes / plan_step /
    densek_smem_bytes / launch_densews_nt) is the one the dispatcher picks for this model, fit and dtype."""
    info = kb.launch_info(model, kfit, dtype=dtype, free_running=free_running, accumulate=accumulate, device=device())
    D, rb, t, sm = model.dim(), 8 if dtype == torch.float64 else 4, info["threads"], info["smem"]
    ok = {
        "lane": t == 64,
        "tile": t == 32 and sm == ((D + 1) & ~1) * rb + 32 * _pad(D, 4) * 4 + D * 4,
        "chain_serial": D <= 16 and t == 32 and sm == (64 * (D | 1) + D) * rb,
        "chain_octet": D > 16 and t == 32 and sm == (36 * _pad(D, rb) + D) * rb,
        "octet": t % 32 == 0 and sm == ((4 if accumulate else 2) * (t // 8) * _pad(D, rb) + 2 * D) * rb,
        "dense_ws": t == 512,
        "dense": t == 256 and sm == 2 * 32 * (D + 4) * 8 + 8 * 4 * (D // 64) * 64 * 8 + (8 * 32 * 2 + 6 * 32) * 8 + D * 4,
    }[want]
    assert ok, (want, info)


def rel_errors(gpu, ref, family):
    """Dimensionless errors: m and zp in units of the fitted scale s, log-parameters absolute."""
    s = np.exp(np.clip(ref["eta"][:, 1], -300, 300))
    em = np.abs(gpu["eta"][:, 0] - ref["eta"][:, 0]) / np.maximum(s, np.abs(ref["eta"][:, 0]))
    es = np.abs(gpu["eta"][:, 1:] - ref["eta"][:, 1:]).max(axis=1)
    ez = np.abs(gpu["zp"] - ref["zp"]) / np.maximum(s, np.abs(ref["zp"]))
    fin = np.isfinite(ref["r"]) & np.isfinite(gpu["r"])
    er = np.where(fin, np.abs(gpu["r"] - ref["r"]) / np.maximum(1.0, np.abs(ref["r"])), 0.0)
    er = np.where(fin | (np.isnan(ref["r"]) & np.isnan(gpu["r"])) | (ref["r"] == gpu["r"]), er, np.inf)
    return em, es, ez, er
