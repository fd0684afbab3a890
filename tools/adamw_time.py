"""End of a training micro-step on GPT-2-Medium-shaped fp32 parameters (290 tensors, 355 M elements, ~10 GB per update
pass: far beyond L2): global-norm clip + AdamW, four ways, timed in one process, alternating, after warm-up:

    torch_foreach   torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW() (foreach, the default on CUDA)
    torch_fused     torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW(fused=True)
    pgica_two_call  NaNSafeGradientNorm (norm + in-place clip kernels) + FusedAdamW.step()
    pgica_fused     FusedAdamW.clip_and_step (norm pass + one update pass that applies the clip factor)

plus the update kernel alone (FusedAdamW.step()).  Rates are algorithmic bytes over time: 28 B per element for the
update (p, g, m, v read; p, m, v written), 4 B more for the norm pass of clip_and_step; the HBM fraction uses the
project's measured peak (bench.peaks() convention, 6.54 TB/s).  Then K = 20 steps from the same state with a cosine
LambdaLR, FusedAdamW and torch's fused AdamW side by side, each step started from the same state; prints the largest
error / (c 2^-24 S) of each against the fp64 step (S, c as in tests/test_fused_adamw.py) and of their difference
against twice that bound.

    python tools/adamw_time.py [--reps 5] [--out profiles/adamw_time.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from preference_guided_image_captioning_alignment_b200 import FusedAdamW, NaNSafeGradientNorm  # noqa: E402

HBM_PEAK_GBS = 6539.9  # measured (SURVEY.md peaks table)
U, C = 2.0 ** -24, 4.0
SHAPES = [(50257, 1024), (1024, 1024)] + [
    s for _ in range(24) for s in ((1024, 3072), (3072,), (1024, 1024), (1024,), (1024, 4096), (4096,), (4096, 1024),
                                   (1024,), (1024,), (1024,), (1024,), (1024,))]
HP = dict(lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
MAX_NORM = 1.0


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def make_arm(kind, dev, gen):
    params = []
    for s in SHAPES:
        p = torch.nn.Parameter(torch.randn(*s, generator=gen, device=dev) * 0.02)
        p.grad = torch.randn(*s, generator=gen, device=dev) * 1e-3
        params.append(p)
    if kind == "torch_foreach":
        opt = torch.optim.AdamW(params, **HP)
    elif kind == "torch_fused":
        opt = torch.optim.AdamW(params, fused=True, **HP)
    else:
        opt = FusedAdamW(params, **HP)
    clipper = NaNSafeGradientNorm(MAX_NORM)

    def step():
        if kind in ("torch_foreach", "torch_fused"):
            torch.nn.utils.clip_grad_norm_(params, MAX_NORM)
            opt.step()
        elif kind == "pgica_two_call":
            clipper(params)
            opt.step()
        elif kind == "pgica_fused":
            opt.clip_and_step(MAX_NORM)
        else:  # update kernel alone
            opt.step()
    return params, opt, step


def time_ms(step, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def accuracy(dev, K=20):
    """K steps of FusedAdamW and torch fused AdamW, each from the same state, cosine LambdaLR: largest error/bound of
    each against the fp64 step from that state, and of their difference against the sum of both bounds."""
    gen = torch.Generator(device=dev).manual_seed(3)
    a = [torch.nn.Parameter(torch.randn(*s, generator=gen, device=dev) * 0.02) for s in SHAPES]
    b = [torch.nn.Parameter(p.detach().clone()) for p in a]
    oa, ob = FusedAdamW(a, **HP), torch.optim.AdamW(b, fused=True, **HP)
    cos = lambda k: 0.5 * (1 + math.cos(math.pi * k / K))
    sa = torch.optim.lr_scheduler.LambdaLR(oa, cos)
    sb = torch.optim.lr_scheduler.LambdaLR(ob, cos)
    worst = {k: {"p": 0.0, "m": 0.0, "v": 0.0} for k in ("fused_adamw", "torch_fused", "difference")}
    b1, b2 = HP["betas"]
    wd, eps = HP["weight_decay"], HP["eps"]
    for k in range(K):
        for p, q in zip(a, b):
            g = torch.randn(p.shape, generator=gen, device=dev) * 1e-3
            p.grad, q.grad = g, g.clone()
        if k > 0:  # the same state on both sides before the step
            for p, q in zip(a, b):
                q.data.copy_(p.data)
                for key in ("exp_avg", "exp_avg_sq"):
                    ob.state[q][key].copy_(oa.state[p][key])
        before = [(p.detach().double(), p.grad.double(), oa.state[p]["exp_avg"].double() if k else torch.zeros_like(p, dtype=torch.float64),
                   oa.state[p]["exp_avg_sq"].double() if k else torch.zeros_like(p, dtype=torch.float64)) for p in a]
        step_lr = oa.param_groups[0]["lr"]
        oa.step()
        ob.step()
        sa.step()
        sb.step()
        s1 = k + 1.0
        bc1, bc2 = 1 - b1 ** s1, 1 - b2 ** s1
        for (p0, g, m0, v0), p, q in zip(before, a, b):
            m1 = b1 * m0 + (1 - b1) * g
            v1 = b2 * v0 + (1 - b2) * g * g
            kk = step_lr / (bc1 * (v1.sqrt() / math.sqrt(bc2) + eps))
            S = {"m": b1 * m0.abs() + (1 - b1) * g.abs(), "v": v1}
            S["p"] = (1 - step_lr * wd) * p0.abs() + kk * S["m"]
            pairs = {"p": (p, q), "m": (oa.state[p]["exp_avg"], ob.state[q]["exp_avg"]),
                     "v": (oa.state[p]["exp_avg_sq"], ob.state[q]["exp_avg_sq"])}
            for key, (x, y) in pairs.items():
                bound = C * U * S[key]
                ref = {"p": (1 - step_lr * wd) * p0 - kk * m1, "m": m1, "v": v1}[key]
                for name, val in (("fused_adamw", x), ("torch_fused", y)):
                    err = (val.double() - ref).abs()
                    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
                    worst[name][key] = max(worst[name][key], float(r.max()))
                err = (x.double() - y.double()).abs()
                r = torch.where(err == 0, torch.zeros_like(err), err / (2 * bound))
                worst["difference"][key] = max(worst["difference"][key], float(r.max()))
        del before
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="alternating rounds over the arms")
    ap.add_argument("--iters", type=int, default=10, help="steps per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "adamw_time.json"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = gpu_info()
    n = sum(math.prod(s) for s in SHAPES)
    arms = ["torch_foreach", "torch_fused", "pgica_two_call", "pgica_fused", "update_kernel_only"]
    times = {k: [] for k in arms}
    gen = torch.Generator(device=dev).manual_seed(0)
    built = {k: make_arm(k, dev, gen) for k in arms}  # ~6 GB each: parameters, gradients, moments
    for k in arms:
        for _ in range(3):
            built[k][2]()
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for k in arms:
            times[k].append(time_ms(built[k][2], args.iters))
    del built
    torch.cuda.empty_cache()
    ms = {k: min(v) for k, v in times.items()}
    upd_bytes, clip_step_bytes = 28 * n, 32 * n
    res = {
        "gpu": info, "tensors": len(SHAPES), "elements": n, "reps": args.reps, "iters_per_window": args.iters,
        "ms_min": ms, "ms_all": times,
        "update_kernel": {"algorithmic_bytes": upd_bytes, "gb_per_s": upd_bytes / ms["update_kernel_only"] / 1e6,
                          "frac_of_measured_hbm_peak": upd_bytes / ms["update_kernel_only"] / 1e6 / HBM_PEAK_GBS},
        "clip_and_step": {"algorithmic_bytes": clip_step_bytes, "gb_per_s": clip_step_bytes / ms["pgica_fused"] / 1e6,
                          "frac_of_measured_hbm_peak": clip_step_bytes / ms["pgica_fused"] / 1e6 / HBM_PEAK_GBS},
        "speedup_clip_and_step_vs_torch_fused": ms["torch_fused"] / ms["pgica_fused"],
        "hbm_peak_gbs": HBM_PEAK_GBS,
    }
    res["max_err_over_bound_20_steps"] = accuracy(dev)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
