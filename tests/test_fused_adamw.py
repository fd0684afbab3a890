"""FusedAdamW (optim.py, csrc/adamw.cu): the fused AdamW step, with and without the folded NaN-safe global-norm clip.

The reference is `adamw_ref` below, the fp64 recurrence of torch's AdamW (decoupled weight decay) with the clip factor
and the non-finite skip, applied to the same fp32 inputs the kernel read.  `bound_ratio` compares element by element
against the bound derived in its docstring; every check prints its largest error/bound ratio, and the same check is
shown to pass torch's own AdamW(fused=True) and to reject planted faults.

CPU tests (not marked gpu) check the oracle against torch.optim.AdamW in float64, the bound against an fp32 emulation of
the kernel's operation sequence and against planted faults, and the optimizer's host-side checks.
"""
import io
import math
import warnings

import numpy as np
import pytest
import torch

U = 2.0 ** -24  # unit roundoff of fp32 round-to-nearest
C = 4.0
CHUNK = 32768  # elements per block of adamw_update_kernel
GPT2_MEDIUM_SHAPES = [(50257, 1024), (1024, 1024)] + [
    s for _ in range(24) for s in ((1024, 3072), (3072,), (1024, 1024), (1024,), (1024, 4096), (4096,), (4096, 1024),
                                   (1024,), (1024,), (1024,), (1024,), (1024,))]


# --------------------------------------------------------------------------------------------------------- oracle
def adamw_ref(p, g, m, v, step, lr, beta1, beta2, eps, weight_decay, coef=1.0, finite=True, fault=None):
    """One AdamW step in fp64 from fp32 inputs (torch/optim/adam.py::_single_tensor_adam, decoupled weight decay):
        g' = fl32(coef * g),  s1 = step + 1,  bc1 = 1 - beta1^s1,  bc2 = 1 - beta2^s1,  a = 1 - lr*wd
        m' = beta1*m + (1-beta1)*g'           v' = beta2*v + (1-beta2)*g'^2
        d  = sqrt(v')/sqrt(bc2) + eps         k = lr / (bc1 * d)            p' = a*p - k*m'
    A non-finite global norm (finite=False) leaves everything as it was.  Also returns the magnitude sums of the terms
    of each recurrence (bound_ratio's S):
        S_m = beta1|m| + (1-beta1)|g'|        S_v = beta2 v + (1-beta2) g'^2 (= v')
        S_p = a|p| + k (beta1|m| + (1-beta1)|g'|) = a|p| + k S_m     (p' = a p - k beta1 m - k (1-beta1) g')
    `fault` plants a bug for the checker to find: "bc_step" (bias corrections with s instead of s + 1), "no_wd" (weight
    decay dropped), "no_clip" (clip factor not applied)."""
    p, g, m, v = (np.asarray(x, dtype=np.float64) for x in (p, g, m, v))
    if not finite:
        return dict(p=p, m=m, v=v, step=step, S_p=np.abs(p), S_m=np.abs(m), S_v=np.abs(v))
    # the clipped gradient as an in-place clip stores it (one fp32 product), which the fused clip reproduces bit for bit
    gc = g if fault == "no_clip" or coef == 1.0 else (np.float32(g) * np.float32(coef)).astype(np.float64)
    s1 = float(step) + (0.0 if fault == "bc_step" else 1.0)
    bc1, bc2 = 1.0 - beta1 ** s1, 1.0 - beta2 ** s1
    a = 1.0 if fault == "no_wd" else 1.0 - lr * weight_decay
    m1 = beta1 * m + (1.0 - beta1) * gc
    v1 = beta2 * v + (1.0 - beta2) * gc * gc
    with np.errstate(divide="ignore", invalid="ignore"):
        k = lr / (bc1 * (np.sqrt(v1) / math.sqrt(bc2) + eps))
        p1 = a * p - k * m1
    S_m = beta1 * np.abs(m) + (1.0 - beta1) * np.abs(gc)
    S_v = beta2 * np.abs(v) + (1.0 - beta2) * gc * gc
    return dict(p=p1, m=m1, v=v1, step=float(step) + 1.0, S_p=a * np.abs(p) + np.abs(k) * S_m, S_m=S_m, S_v=S_v)


def bound_ratio(x, ref, S, c=C):
    """Largest |x - x64| / (c * 2^-24 * S_x) over the elements (0 where both sides are 0; inf for a non-finite error).

    Derivation.  Every fp32 operation returns fl(r) = r (1 + d) with |d| <= u = 2^-24, and so does rounding a double
    value once to fp32.  The kernel forms m' and v' as short fp32 sequences, with fp32 scalars (double values rounded
    once), from the fp32 inputs and g' = fl(coef g), which the reference takes as given (it is what an in-place clip
    stores, and the fused clip reproduces it bit for bit):
      m' = fma(w, fl(g' - m), m),  w = fl(1 - beta1) < 1/2
      v' = fma(fl(fl(1 - beta2) g'), g', fl(fl(beta2) v))
    Expand each output into the terms of its exact recurrence (adamw_ref).  A rounding perturbs the terms it touches by
    at most u times their magnitude:
      m: w (1 + d_w)(g' - m)(1 + d_s) + m, rounded:  |err| <= 2u w (|g'| + |m|) + u |m'|.  As w <= beta1,
         w |m| <= beta1 |m|, so |err| <= 2u S_m + u S_m = 3u S_m.
      v: the term (1-beta2) g'^2 carries two roundings (scalar, product), beta2 v two (scalar, product), the fma one
         of |v'| <= S_v:  |err| <= 3u S_v.
    So c = 4 holds for m and v in the worst case, with one unit to spare.  p' is evaluated in double from the fp32 p,
    m', v' and double scalars, and rounded once, so its error is what m' and v' carry in plus that last rounding:
      p: k m' with |m' - m'_64| <= 3u S_m; sqrt halves the relative error of v' (<= 3u) in the denominator, which moves
         k by <= 1.5u; the rounding of p' adds u |p'| <= u S_p:  |err| <= (3 + 1.5) u k S_m + u S_p <= 5.5u S_p.
    For p, c = 4 is therefore not a worst case: it takes the roundings of m', v' and p' to reach their extreme values
    with the same sign in one element.  They are independent and spread over [-u, u], and the measured ratio over 16 M
    random elements (emulated, see emulate_kernel_f32; CPU test below) is 0.55 for p, 0.51 for m and 0.69 for v.
    The double-precision p update is what makes c = 4 hold: formed in fp32, the update term passes about nine further
    roundings (sqrt, two scalars, fma, quotient, step size, final fma), and the same emulation reaches a ratio of 1.03.
    torch's AdamW(fused=True) computes m and v in double and passes the same check.  Errors in the inputs are not
    counted: the reference starts from the very fp32 values the kernel read.
    """
    x = np.asarray(x, dtype=np.float64)
    err = np.abs(x - ref)
    bound = c * U * np.asarray(S, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / bound)
    r = np.where(np.isfinite(r), r, np.inf)
    return float(r.max()) if r.size else 0.0


def emulate_kernel_f32(p, g, m, v, step, lr, beta1, beta2, eps, weight_decay, coef=1.0):
    """The kernel's operation sequence (adamw_elem in csrc/adamw.cu) in numpy: m and v in fp32 (an fma is one rounding
    of the exact fp64 result: a product of two fp32 values is exact in fp64), the update of p in double, rounded once."""
    f = np.float32
    fma = lambda a, b, c: (np.float64(a) * np.float64(b) + np.float64(c)).astype(f)
    s1 = float(step) + 1.0
    step_size, rsbc2 = lr / (1.0 - beta1 ** s1), 1.0 / math.sqrt(1.0 - beta2 ** s1)
    w1, b2, omb2 = f(1.0 - beta1), f(beta2), f(1.0 - beta2)
    gc = (g * f(coef)).astype(f)
    m1 = fma(w1, (gc - m).astype(f), m)
    v1 = fma((omb2 * gc).astype(f), gc, (v * b2).astype(f))
    den = np.sqrt(v1.astype(np.float64)) * rsbc2 + eps
    p2 = (p.astype(np.float64) * (1.0 - lr * weight_decay) - step_size * (m1.astype(np.float64) / den)).astype(f)
    return p2, m1, v1


def random_state(n, seed, step_scale=1.0):
    """p ~ N(0, 1), g ~ N(0, 0.1^2) with sign-mixed m ~ N(0, 0.05^2) and v ~ (0.1 N)^2 (nonzero moments)."""
    rng = np.random.default_rng(seed)
    f = np.float32
    p = rng.standard_normal(n).astype(f)
    g = (0.1 * rng.standard_normal(n)).astype(f)
    m = (0.05 * rng.standard_normal(n)).astype(f)
    v = ((0.1 * rng.standard_normal(n)) ** 2).astype(f)
    return p, g, m, v


HP = dict(lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.01)
FAULTS = ("bc_step", "no_wd", "no_clip", "chunk")
COEF = float(np.float32(0.37))  # a clip factor < 1, as the fp32 value the norm kernel would hand over


def check_against_ref(out, inp, step, hp, coef=1.0, finite=True, label=""):
    """ratios (p, m, v) of the fp32 results `out` against the oracle from the fp32 inputs `inp` (all numpy)."""
    ref = adamw_ref(*inp, step, **hp, coef=coef, finite=finite)
    return tuple(bound_ratio(o, ref[k], ref["S_" + k]) for o, k in zip(out, ("p", "m", "v")))


def planted(inp, step, hp, coef, fault):
    """The oracle's own result rounded to fp32, with one planted fault."""
    if fault == "chunk":
        ref = adamw_ref(*inp, step, **hp, coef=coef)
        out = [ref[k].astype(np.float32) for k in ("p", "m", "v")]
        lo = CHUNK if len(inp[0]) > CHUNK else 0
        for o, x in zip(out, (inp[0], inp[2], inp[3])):
            o[lo:lo + CHUNK] = x[lo:lo + CHUNK]  # one chunk left un-updated
        return out
    ref = adamw_ref(*inp, step, **hp, coef=coef, fault=fault)
    return [ref[k].astype(np.float32) for k in ("p", "m", "v")]


# --------------------------------------------------------------------------------------------------------- CPU tests
def test_oracle_matches_torch_adamw_fp64():
    """adamw_ref against torch.optim.AdamW(foreach=False) in float64 on the CPU: 5 steps, two param groups."""
    torch.manual_seed(0)
    shapes = [(7, 5), (13,), (4, 4, 3)]
    params = [torch.nn.Parameter(torch.randn(*s, dtype=torch.float64)) for s in shapes]
    groups = [dict(params=params[:2], lr=3e-3, weight_decay=0.05, betas=(0.9, 0.999), eps=1e-8),
              dict(params=params[2:], lr=1e-2, weight_decay=0.0, betas=(0.8, 0.99), eps=1e-6)]
    opt = torch.optim.AdamW(groups, foreach=False)
    state = [dict(p=p.detach().numpy().copy(), m=np.zeros(p.shape), v=np.zeros(p.shape), step=0.0) for p in params]
    for it in range(5):
        grads = [torch.randn(*s, dtype=torch.float64) for s in shapes]
        for p, g in zip(params, grads):
            p.grad = g
        opt.step()
        for gi, group in enumerate(groups):
            for p in group["params"]:
                i = next(j for j, q in enumerate(params) if q is p)
                st = state[i]
                r = adamw_ref(st["p"], grads[i].numpy(), st["m"], st["v"], st["step"], group["lr"], group["betas"][0],
                              group["betas"][1], group["eps"], group["weight_decay"])
                st.update(p=r["p"], m=r["m"], v=r["v"], step=r["step"])
    for i, p in enumerate(params):
        ts = opt.state[p]
        for got, want in ((p.detach().numpy(), state[i]["p"]), (ts["exp_avg"].numpy(), state[i]["m"]),
                          (ts["exp_avg_sq"].numpy(), state[i]["v"])):
            assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max()
        assert float(ts["step"]) == state[i]["step"] == 5.0


@pytest.mark.parametrize("step", [0, 1, 999, 1_000_000])
def test_bound_admits_fp32_kernel_sequence(step):
    """The fp32 emulation of the kernel's operation sequence stays within the bound, with a clip factor < 1."""
    inp = random_state(1 << 20, seed=step)
    out = emulate_kernel_f32(*inp, step, **HP, coef=COEF)
    rp, rm, rv = check_against_ref(out, inp, step, HP, coef=COEF)
    print(f"\nstep {step}: fp32 emulation, max error/bound  p {rp:.3f}  m {rm:.3f}  v {rv:.3f}")
    assert max(rp, rm, rv) <= 1.0


@pytest.mark.parametrize("step", [0, 999])
def test_bound_rejects_planted_faults(step):
    n = 3 * CHUNK + 5
    inp = random_state(n, seed=10 + step)
    good = planted(inp, step, HP, COEF, fault="none")
    assert max(check_against_ref(good, inp, step, HP, coef=COEF)) <= 1.0
    for fault in FAULTS:
        r = check_against_ref(planted(inp, step, HP, COEF, fault), inp, step, HP, coef=COEF)
        print(f"\nstep {step}: planted fault {fault}: error/bound  p {r[0]:.3g}  m {r[1]:.3g}  v {r[2]:.3g}")
        assert max(r) > 1.0, fault


@pytest.mark.parametrize("kwargs,name", [
    (dict(amsgrad=True), "amsgrad"), (dict(maximize=True), "maximize"), (dict(capturable=True), "capturable"),
    (dict(differentiable=True), "differentiable"), (dict(foreach=True), "foreach"), (dict(fused=True), "fused"),
    (dict(lr=torch.tensor(1e-3)), "lr"), (dict(betas=(torch.tensor(0.9), 0.999)), "betas")])
def test_constructor_rejects_unsupported_options(kwargs, name):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    with pytest.raises(ValueError, match=name):
        FusedAdamW([torch.nn.Parameter(torch.zeros(4))], **kwargs)


def test_constructor_rejects_parameter_kinds():
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    for dt in (torch.float16, torch.bfloat16, torch.float64):
        with pytest.raises(ValueError, match="fp32"):
            FusedAdamW([torch.nn.Parameter(torch.zeros(4, dtype=dt))])
    with pytest.raises(ValueError, match="sparse"):
        FusedAdamW([torch.nn.Parameter(torch.zeros(4, 4).to_sparse())])
    with pytest.raises(ValueError, match="amsgrad"):
        FusedAdamW([dict(params=[torch.nn.Parameter(torch.zeros(4))], amsgrad=True)])


def test_cpu_parameters_raise_at_step():
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    from preference_guided_image_captioning_alignment_b200._lib import PgicaError
    p = torch.nn.Parameter(torch.zeros(8))
    p.grad = torch.ones(8)
    opt = FusedAdamW([p])
    with pytest.raises(PgicaError):
        opt.step()


def test_param_group_keys_match_torch_adamw():
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    groups = lambda: [dict(params=[torch.nn.Parameter(torch.zeros(3))]),
                      dict(params=[torch.nn.Parameter(torch.zeros(2))], lr=0.1, weight_decay=0.0)]
    ours, theirs = FusedAdamW(groups(), lr=1e-3), torch.optim.AdamW(groups(), lr=1e-3)
    assert [sorted(g) for g in ours.param_groups] == [sorted(g) for g in theirs.param_groups]
    assert [{k: v for k, v in g.items() if k != "params"} for g in ours.param_groups] == \
           [{k: v for k, v in g.items() if k != "params"} for g in theirs.param_groups]


# --------------------------------------------------------------------------------------------------------- GPU tests
SIZES = [1, 3, 4, 4097, 32769, 1 << 20]
STEPS = [0, 1, 999, 1_000_000]
GROUP_HP = [dict(lr=1e-3, weight_decay=0.01), dict(lr=3e-4, weight_decay=0.1)]


def _t(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def _np(t):
    return t.detach().float().cpu().numpy().copy()


def build_problem(dev, seed=0):
    """Params over two groups, numel in SIZES (+ one leaf carved at element offset 3 of a flat buffer, its gradient at
    offset 1), random nonzero moments, per-tensor step counts from STEPS.  -> (params, groups, state, grads)."""
    params, grads, state = [], [], {}
    sizes = SIZES + [4097 + 40]
    for i, n in enumerate(sizes):
        p, g, m, v = random_state(n, seed=100 * seed + i)
        if i == len(sizes) - 1:
            flat, gflat = torch.zeros(n + 8, device=dev), torch.zeros(n + 8, device=dev)
            flat[3:3 + n] = _t(p, dev)
            gflat[1:1 + n] = _t(g, dev)
            param = torch.nn.Parameter(flat[3:3 + n])
            assert param.is_leaf and param.data_ptr() % 16 == 12
            param.grad = gflat[1:1 + n]
        else:
            param = torch.nn.Parameter(_t(p, dev))
            param.grad = _t(g, dev)
        params.append(param)
        state[i] = dict(step=float(STEPS[i % len(STEPS)]), exp_avg=_t(m, dev), exp_avg_sq=_t(v, dev))
    groups = [dict(params=params[0::2], **GROUP_HP[0]), dict(params=params[1::2], **GROUP_HP[1])]
    return params, groups, state


def load_state(opt, params, state, dev):
    for i, p in enumerate(params):
        s = state[i]
        opt.state[p] = dict(step=torch.tensor(s["step"], dtype=torch.float32, device=dev),
                            exp_avg=s["exp_avg"].clone(), exp_avg_sq=s["exp_avg_sq"].clone())


def snapshot(opt, params):
    return [(_np(p), _np(p.grad), _np(opt.state[p]["exp_avg"]), _np(opt.state[p]["exp_avg_sq"]),
             float(opt.state[p]["step"])) for p in params]


def hp_of(opt, p):
    g = next(g for g in opt.param_groups if any(q is p for q in g["params"]))
    return dict(lr=g["lr"], beta1=g["betas"][0], beta2=g["betas"][1], eps=g["eps"], weight_decay=g["weight_decay"])


def ratios_after(opt, params, before, coef=1.0, finite=True):
    """largest (p, m, v) error/bound ratios of the optimizer's state against the oracle from `before`."""
    worst = np.zeros(3)
    for p, (p0, g0, m0, v0, s0) in zip(params, before):
        out = (_np(p), _np(opt.state[p]["exp_avg"]), _np(opt.state[p]["exp_avg_sq"]))
        r = check_against_ref(out, (p0, g0, m0, v0), s0, hp_of(opt, p), coef=coef, finite=finite)
        worst = np.maximum(worst, r)
        assert float(opt.state[p]["step"]) == s0 + (1.0 if finite else 0.0)
    return worst


def clone_problem(params, dev):
    out = []
    for p in params:
        q = torch.nn.Parameter(p.detach().clone())
        q.grad = p.grad.detach().clone()
        out.append(q)
    return out


def regroup(params, groups, new_params):
    idx = {id(p): i for i, p in enumerate(params)}
    return [dict(g, params=[new_params[idx[id(p)]] for p in g["params"]]) for g in groups]


@pytest.mark.gpu
def test_one_step_within_bound_and_torch_fused_too(cuda_device):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    params, groups, state = build_problem(dev)
    opt = FusedAdamW(groups)
    load_state(opt, params, state, dev)
    before = snapshot(opt, params)
    opt.step()
    ours = ratios_after(opt, params, before)
    tparams = clone_problem(params, dev)
    for q, (p0, g0, *_), in zip(tparams, before):
        q.data.copy_(_t(p0, dev))
        q.grad = _t(g0, dev)
    topt = torch.optim.AdamW(regroup(params, groups, tparams), fused=True)
    load_state(topt, tparams, state, dev)
    topt.step()
    theirs = ratios_after(topt, tparams, before)
    print(f"\none step: max error/bound FusedAdamW p {ours[0]:.3f} m {ours[1]:.3f} v {ours[2]:.3f}; "
          f"torch fused p {theirs[0]:.3f} m {theirs[1]:.3f} v {theirs[2]:.3f}")
    assert ours.max() <= 1.0 and theirs.max() <= 1.0
    # the checker sees each planted fault on these very inputs
    big = next(i for i, b in enumerate(before) if b[0].size == 1 << 20)
    p0, g0, m0, v0, s0 = before[big]
    hp = hp_of(opt, params[big])
    for fault in FAULTS:
        r = check_against_ref(planted((p0, g0, m0, v0), s0, hp, COEF, fault), (p0, g0, m0, v0), s0, hp, coef=COEF)
        print(f"planted fault {fault}: error/bound p {r[0]:.3g} m {r[1]:.3g} v {r[2]:.3g}")
        assert max(r) > 1.0, fault


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["step", "clip_and_step"])
def test_twenty_step_trajectory_with_cosine_schedule(cuda_device, mode):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    params, groups, state = build_problem(dev, seed=1)
    opt = FusedAdamW(groups)
    load_state(opt, params, state, dev)
    K = 20
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda k: 0.5 * (1 + math.cos(math.pi * k / K)))
    gen = torch.Generator(device=dev).manual_seed(7)
    worst = np.zeros(3)
    with warnings.catch_warnings():
        warnings.simplefilter("error")  # "lr_scheduler.step() before optimizer.step()" would raise here
        for k in range(K):
            for p in params:
                p.grad.copy_(torch.randn(p.shape, generator=gen, device=dev) * 0.1)
            before = snapshot(opt, params)
            if mode == "step":
                opt.step()
                coef = 1.0
            else:
                norm = math.sqrt(sum(float((b[1].astype(np.float64) ** 2).sum()) for b in before))
                total, finite = opt.clip_and_step(0.5 * norm)
                coef = float(np.float32(min(1.0, np.float32(0.5 * norm) / (np.float32(total.item()) + np.float32(1e-6)))))
                assert bool(finite)
            worst = np.maximum(worst, ratios_after(opt, params, before, coef=coef))
            sched.step()
    print(f"\n{K} steps ({mode}), cosine LR: max error/bound p {worst[0]:.3f} m {worst[1]:.3f} v {worst[2]:.3f}")
    assert worst.max() <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.5, 2.0])
def test_clip_fold_is_exact(cuda_device, scale):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW, functional as F
    dev = cuda_device
    params, groups, state = build_problem(dev, seed=2)
    a_params, b_params = clone_problem(params, dev), clone_problem(params, dev)
    a, b = FusedAdamW(regroup(params, groups, a_params)), FusedAdamW(regroup(params, groups, b_params))
    load_state(a, a_params, state, dev)
    load_state(b, b_params, state, dev)
    norm = float(torch.sqrt(sum((p.grad.double() ** 2).sum() for p in params)))
    max_norm = scale * norm  # 0.5: clips; 2.0: does not
    grads_before = [p.grad.clone() for p in a_params]
    total, finite = a.clip_and_step(max_norm)
    F.grad_norm_clip([p.grad for p in b_params], max_norm, clip=True)
    b.step()
    assert bool(finite) and abs(float(total) - norm) <= 1e-5 * norm
    for pa, pb, g0 in zip(a_params, b_params, grads_before):
        assert torch.equal(pa, pb)
        for key in ("exp_avg", "exp_avg_sq", "step"):
            assert torch.equal(a.state[pa][key], b.state[pb][key])
        assert torch.equal(pa.grad, g0)  # clip_and_step leaves the gradients unclipped


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
def test_non_finite_gradient_skips_the_step(cuda_device, bad):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    params, groups, state = build_problem(dev, seed=3)
    opt = FusedAdamW(groups)
    load_state(opt, params, state, dev)
    victim = params[4]
    good = victim.grad[123].item()
    victim.grad[123] = bad
    before = [(p.detach().clone(), {k: t.clone() for k, t in opt.state[p].items()}) for p in params]
    total, finite = opt.clip_and_step(1.0)
    assert not bool(finite) and not math.isfinite(float(total))
    for p, (p0, s0) in zip(params, before):
        assert torch.equal(p, p0)
        for key in s0:
            assert torch.equal(opt.state[p][key], s0[key])
    # the next finite step applies the bias corrections of the step count that was NOT advanced
    victim.grad[123] = good
    snap = snapshot(opt, params)
    norm = math.sqrt(sum(float((b[1].astype(np.float64) ** 2).sum()) for b in snap))
    total, finite = opt.clip_and_step(0.5 * norm)
    assert bool(finite)
    coef = float(np.float32(min(1.0, np.float32(0.5 * norm) / (np.float32(total.item()) + np.float32(1e-6)))))
    worst = ratios_after(opt, params, snap, coef=coef)
    print(f"\nafter a skipped step ({bad}): max error/bound p {worst[0]:.3f} m {worst[1]:.3f} v {worst[2]:.3f}")
    assert worst.max() <= 1.0


@pytest.mark.gpu
def test_no_host_synchronisation(cuda_device):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    params, groups, state = build_problem(dev, seed=4)
    opt = FusedAdamW(groups)
    opt.step()  # warm-up: lazy state, library load
    opt.clip_and_step(1.0)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        opt.step()
        total, finite = opt.clip_and_step(1.0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert bool(finite)


@pytest.mark.gpu
def test_step_moves_version_for_cached_bf16(cuda_device):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW, ops
    dev = cuda_device
    w = torch.nn.Parameter(torch.randn(512, 256, device=dev))
    w.grad = torch.randn_like(w)
    first = ops.cached_bf16(w)
    assert torch.equal(first, w.detach().to(torch.bfloat16))
    v0 = w._version
    FusedAdamW([w], lr=0.1).step()
    assert w._version > v0
    assert torch.equal(ops.cached_bf16(w), w.detach().to(torch.bfloat16))
    assert not torch.equal(ops.cached_bf16(w), first)


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["fused_to_torch", "torch_to_fused"])
def test_checkpoints_move_both_ways(cuda_device, direction):
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    params, groups, _ = build_problem(dev, seed=5)
    src_cls, dst_cls = (FusedAdamW, torch.optim.AdamW) if direction == "fused_to_torch" else \
        (torch.optim.AdamW, FusedAdamW)
    src = src_cls(groups)
    gen = torch.Generator(device=dev).manual_seed(11)
    new_grads = lambda: [torch.randn(p.shape, generator=gen, device=dev) * 0.1 for p in params]
    for _ in range(2):
        for p, g in zip(params, new_grads()):
            p.grad.copy_(g)
        src.step()
    buf = io.BytesIO()  # a checkpoint round trip: the loaded state must not alias the source optimizer's tensors
    torch.save(src.state_dict(), buf)
    buf.seek(0)
    sd = torch.load(buf, weights_only=True)
    if direction == "torch_to_fused":
        assert all(s["step"].device.type == "cpu" for s in sd["state"].values())
    dst_params = clone_problem(params, dev)
    dst = dst_cls(regroup(params, groups, dst_params))
    dst.load_state_dict(sd)
    for p, q in zip(params, dst_params):
        for key in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(src.state[p][key], dst.state[q][key].to(src.state[p][key].device))
    # continue 3 steps in both, with the same gradients; each step of each optimizer against the oracle from its own
    # state before the step
    worst = np.zeros(3)
    for _ in range(3):
        gs = new_grads()
        for ps, opt in ((params, src), (dst_params, dst)):
            for p, g in zip(ps, gs):
                p.grad.copy_(g)
            before = snapshot(opt, ps)
            opt.step()
            worst = np.maximum(worst, ratios_after(opt, ps, before))
    for p, q in zip(params, dst_params):
        assert float(src.state[p]["step"]) == float(dst.state[q]["step"]) == 5.0
        if dst_cls is FusedAdamW:
            assert dst.state[q]["step"].device == q.device  # the CPU step counter was moved once
    print(f"\ncheckpoint {direction}, 3 more steps: max error/bound p {worst[0]:.3f} m {worst[1]:.3f} v {worst[2]:.3f}")
    assert worst.max() <= 1.0


@pytest.mark.gpu
def test_full_gpt2_medium_size_against_torch_fused(cuda_device):
    """355 M fp32 elements in the 290 tensor shapes of the GPT-2-Medium decoder, one step with nonzero moments, checked
    element by element against the fp64 step.  torch's AdamW(fused=True) takes the same step beside it and its ratio is
    printed, but not asserted: at this size it exceeds the bound (measured on a B200: 28 for p and 55 for v), although it
    stays within the bound on the 1.1 M elements of test_one_step_within_bound_and_torch_fused_too."""
    from preference_guided_image_captioning_alignment_b200 import FusedAdamW
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(12)
    params = []
    for s in GPT2_MEDIUM_SHAPES:
        p = torch.nn.Parameter(torch.randn(*s, generator=gen, device=dev))
        p.grad = torch.randn(*s, generator=gen, device=dev) * 0.1
        params.append(p)
    assert len(params) == 290 and sum(p.numel() for p in params) == 354_821_120
    state = {i: dict(step=10.0, exp_avg=torch.randn(p.shape, generator=gen, device=dev) * 0.05,
                     exp_avg_sq=(torch.randn(p.shape, generator=gen, device=dev) * 0.1) ** 2)
             for i, p in enumerate(params)}
    p0 = [p.detach().clone() for p in params]
    tparams = clone_problem(params, dev)
    hp = dict(lr=HP["lr"], betas=(HP["beta1"], HP["beta2"]), eps=HP["eps"], weight_decay=HP["weight_decay"])
    opt, topt = FusedAdamW(params, **hp), torch.optim.AdamW(tparams, fused=True, **hp)
    load_state(opt, params, state, dev)
    load_state(topt, tparams, state, dev)
    opt.step()
    topt.step()
    torch.cuda.synchronize()
    worst, tworst = np.zeros(3), np.zeros(3)
    for i, (p, q) in enumerate(zip(params, tparams)):
        inp = (_np(p0[i]).ravel(), _np(p.grad).ravel(), _np(state[i]["exp_avg"]).ravel(),
               _np(state[i]["exp_avg_sq"]).ravel())
        ref = adamw_ref(*inp, 10.0, **HP)
        for k, (mine, theirs) in enumerate(((p, q), (opt.state[p]["exp_avg"], topt.state[q]["exp_avg"]),
                                            (opt.state[p]["exp_avg_sq"], topt.state[q]["exp_avg_sq"]))):
            key = "pmv"[k]
            worst[k] = max(worst[k], bound_ratio(_np(mine).ravel(), ref[key], ref["S_" + key]))
            tworst[k] = max(tworst[k], bound_ratio(_np(theirs).ravel(), ref[key], ref["S_" + key]))
        assert float(opt.state[p]["step"]) == 11.0
    print(f"\n290 tensors, {sum(p.numel() for p in params)} elements: max error/bound FusedAdamW p {worst[0]:.3f} "
          f"m {worst[1]:.3f} v {worst[2]:.3f}; torch fused p {tworst[0]:.3f} m {tworst[1]:.3f} v {tworst[2]:.3f}")
    assert worst.max() <= 1.0
