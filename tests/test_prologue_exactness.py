"""Element-level exactness of the two fused LayerNorm kernels of xattn.cu, and of their Python wiring (prologue.py).

* `xattn_ln_fwd` / `xattn_ln_bwd`: the decoder's one-key cross-attention plus `attention_norm`,
      y = LayerNorm(pre),  pre = x + b_o + sum_h w[b, t, h] U[b, h]
  one CTA of 256 threads per row in the forward (each thread holds up to four float4 groups of the row), one CTA per
  sequence in the backward (du[b], and per-sequence partials of dgamma / dbeta / db_o that the caller sums over b).
* `ln_l2norm_fwd` / `ln_l2norm_bwd`: the LayerNorm + F.normalize tail of the projection heads, one warp per row,
  n = e / max(||e||, eps_norm); the backward's dgamma / dbeta partials per block of 8 rows.

A global relative norm of 1e-5 cannot tell eps added outside the rsqrt (1e-5 relative at unit variance) from rounding,
nor a wrong float4 group, nor the normalisation gradient of a row below eps_norm.  The checks here:

1. Exact inputs, compared bit for bit (`torch.equal`) with a closed form (`xattn_exact`, `ln_exact`): pre = c + s sigma
   with sigma in {+-1}^E balanced, c dyadic, s a power of two, eps_ln = 0, so the mean is c, the biased variance s^2
   and x-hat = +-1; every operand a small dyadic value, so every partial sum is exact and the kernels' summation order
   cannot matter.  rsqrtf(s^2) is the one statistic that need not be exact: the closed forms take the kernel's own
   rstd (and inv), and the test states whether rsqrtf was exact at those powers of four.
2. Bounded checks against fp64 of the fp32 inputs: per element in the forwards, per row in the gradients, with bounds
   derived from the kernels' operation order (`xattn_fwd_tol`, `xattn_bwd_tol`, `ln_fwd_tol`, `ln_bwd_tol`).
3. Planted faults (`XF_FAULTS`, `XB_FAULTS`, `LN_FAULTS`) are applied to the fp64 reference; every check a fault
   targets must reject it in some case of the test, and the ratio by which it is seen is printed.
4. The wiring: `prologue.collapsed_cross_attention_ln` against nn.MultiheadAttention + nn.LayerNorm in fp64,
   `prologue.ln_l2norm` against layer_norm -> F.normalize autograd in fp64, and the unit-norm promise of the twin.

The helpers are plain torch; the tests not marked `gpu` check the builders and the checkers against fp32 emulations,
and the argument checks of the wrappers.
"""
import math
import types

import numpy as np
import pytest
import torch

from test_kernel_exactness import card, report, rows_within
from test_ntxent_composed_exactness import FaultTally

F32 = np.float32
f64 = torch.float64
U = 2.0 ** -24                      # fp32 unit roundoff
RSQRT = 2.0 ** -22                  # rsqrtf: 2 ulp (CUDA C++ Programming Guide, single-precision functions)
EPS_LN = 1e-5
EPS_NORM = 1e-12
XF_FAULTS = ("head_dropped", "w_neighbour", "u_prev_seq", "bo_dropped", "unbiased_var", "eps_outside",
             "group_dropped")
XB_FAULTS = ("du_missing_last", "du_head_shift", "m2_dropped", "dgamma_from_dy", "dbo_from_dy")
LN_FAULTS = ("projection_below_eps", "projection_omitted", "de_ignored", "inv_once", "partial_missing_row",
             "rows_past_end")


def representable(t):
    """Every entry of the fp64 tensor is an fp32 value."""
    return torch.equal(t.float().double(), t)


def groups(E):
    """float4 groups each thread of the 256-thread xattn CTA holds."""
    return -(-(E // 4) // 256)


def block_depth(E):
    """Roundings on the way of one summand into block_sum: 4 per float4 group (`s += a.x + a.y + a.z + a.w`), five
    butterfly levels in the warp and five more over the 8 warp totals."""
    return 4 * groups(E) + 10


def warp_depth(D):
    """Roundings of one summand in a one-warp row sum: D / 32 serial adds per lane and five butterfly levels."""
    return -(-D // 32) + 5


# ================================================================================================ xattn: fp64 model
def xattn_model(x, u, w, bo, g, b, eps, dy=None, stats=None, fault=None):
    """fp64 forward (and, with dy, backward) of the kernel pair.  stats: (mean, rstd) to use in place of the fp64
    statistics (the kernel's own).  fault: one of XF_FAULTS / XB_FAULTS.
    -> dict(pre, mean, rstd, xh, y[, dx, du, dg, db, dp]) with the per-sequence partials dg, db, dp of shape (B, E)."""
    X, UU = x.double(), u.double()
    B, T, E = X.shape
    H = UU.shape[1]
    W = torch.ones(B, T, H, dtype=f64, device=X.device) if w is None else w.double()
    Wf, Uf = W, UU
    if fault == "w_neighbour":
        Wf = torch.roll(W, -1, dims=1)
    elif fault == "u_prev_seq":
        Uf = torch.roll(UU, 1, dims=0)
    elif fault == "head_dropped":
        Wf = W.clone()
        Wf[:, :, H // 2] = 0
    pre = X + torch.einsum("bth,bhe->bte", Wf, Uf)
    if bo is not None and fault != "bo_dropped":
        pre = pre + bo.double()
    p = pre
    if fault == "group_dropped":          # the highest float4 group of every thread left out of the statistics
        p = pre[..., :1024 * (groups(E) - 1)] if groups(E) > 1 else pre[..., :E - 4]
    mu = p.mean(-1, keepdim=True)
    var = ((p - mu) ** 2).sum(-1, keepdim=True) / (p.shape[-1] - (fault == "unbiased_var"))
    rs = 1.0 / (var.sqrt() + eps) if fault == "eps_outside" else 1.0 / (var + eps).sqrt()
    if stats is not None:
        mu, rs = stats[0].double().view(B, T, 1), stats[1].double().view(B, T, 1)
    xh = (pre - mu) * rs
    out = dict(pre=pre, mean=mu.view(-1), rstd=rs.view(-1), xh=xh, y=xh * g.double() + b.double(), var=var)
    if dy is None:
        return out
    DY = dy.double()
    gg = DY * g.double()
    m1 = gg.mean(-1, keepdim=True)
    m2 = (gg * xh).mean(-1, keepdim=True)
    dp = rs * (gg - m1 - (0 if fault == "m2_dropped" else xh * m2))
    tt = T - 1 if fault == "du_missing_last" else T
    du = torch.einsum("bth,bte->bhe", W[:, :tt], dp[:, :tt])
    if fault == "du_head_shift":
        du = torch.roll(du, 1, dims=1)
    out.update(dx=dp, du=du, dg=(DY * (1.0 if fault == "dgamma_from_dy" else xh)).sum(1), db=DY.sum(1),
               dp=(DY if fault == "dbo_from_dy" else dp).sum(1))
    return out


def xattn_abs_pre(x, u, w, bo):
    """|x| + |b_o| + sum_h |w U|: the magnitude every partial sum of pre is bounded by."""
    B, T, E = x.shape
    H = u.shape[1]
    W = torch.ones(B, T, H, dtype=f64, device=x.device) if w is None else w.double()
    a = x.double().abs() + torch.einsum("bth,bhe->bte", W.abs(), u.double().abs())
    return a + (bo.double().abs() if bo is not None else 0)


def xattn_fwd_tol(ref, x, u, w, bo, g, eps, dpre_extra=0.0):
    """Per-element bounds of the forward (first order in u = 2^-24, every sum bounded by depth u sum |terms|):
        pre      (H + 1) u A,  A = |x| + |b_o| + sum_h |w U|           (the add of b_o, H fmaf)  [+ dpre_extra]
        mean     (block_depth u sum |pre| + sum dpre) / E + u |mean|
        var      the terms fl(a - mean~)^2: 2 d eta + eta^2 + u (d + eta)^2 with d = |pre - mean|, eta = dpre + dmean +
                 u (d + dmean); their block sum (block_depth u), the division and the add of eps (u each)
        rstd     rsqrtf: 2 ulp (2^-22) plus half the relative error of var + eps
        y        |gamma| (eta rstd + d drstd + u |xh|) + u |y|       (x-hat rounded, then one fmaf with beta)
    -> dict(mean, rstd, y, dpre, dmean, drs) of absolute bounds."""
    B, T, E = x.shape
    H = u.shape[1]
    A = xattn_abs_pre(x, u, w, bo)
    pre, mu, var = ref["pre"], ref["mean"].view(B, T, 1), ref["var"]
    rs = ref["rstd"].view(B, T, 1)
    k = block_depth(E)
    dpre = (H + 1) * U * A + dpre_extra
    dmu = (k * U * pre.abs().sum(-1, keepdim=True) + dpre.sum(-1, keepdim=True)) / E + U * mu.abs()
    d = (pre - mu).abs()
    eta = dpre + dmu + U * (d + dmu)
    t = 2 * d * eta + eta ** 2 + U * (d + eta) ** 2
    dvar = (t.sum(-1, keepdim=True) + k * U * (d + eta).pow(2).sum(-1, keepdim=True)) / E + U * var + U * (var + eps)
    r = dvar / (var + eps)
    drs = rs * (0.5 * r + r * r + RSQRT)
    xh = d * rs
    dy = g.double().abs() * (eta * rs + d * drs + U * xh) + U * ref["y"].abs()
    return dict(mean=dmu.view(-1), rstd=drs.view(-1), y=dy * (1 + 1e-3), dpre=dpre, dmean=dmu, drs=drs)


def xattn_bwd_tol(ref, x, u, w, bo, g, dy, dmu, drs, dpre_extra=0.0):
    """Per-row bounds (L2 of per-element bounds) of the backward given the forward's statistics, off from fp64 by
    dmu, drs (measured, per row), with zeta the error of the recomputed x-hat:
        zeta     (dpre + dmu + u (d + dmu)) (rstd + drs) + d drs + 2 u |xh|
        m1       ((block_depth + 1) u sum |gg|) / E + u |m1|           gg = dy gamma, rounded once
        m2       (sum |gg| zeta + (block_depth + 2) u sum |gg xh|) / E + u |m2|
        dx       rstd (u |gg| + dm1 + |xh| dm2 + |m2| zeta + 3 u (|gg| + |m1| + |xh m2|)) + drs |dx| / rstd + u |dx|
        du       sum_t |w| ddx + T u sum_t |w dx|        dgamma: sum_t |dy| zeta + (T + 1) u sum_t |dy xh|
        dbeta    T u sum_t |dy|                          db_o:   sum_t ddx + T u sum_t |dx|
    -> dict(dx, du, dg, db, dp) of per-row bounds."""
    B, T, E = x.shape
    H = u.shape[1]
    k = block_depth(E)
    A = xattn_abs_pre(x, u, w, bo)
    rs, mu = ref["rstd"].view(B, T, 1), ref["mean"].view(B, T, 1)
    dmu, drs = dmu.view(B, T, 1), drs.view(B, T, 1)
    d = (ref["pre"] - mu).abs()
    xh = ref["xh"].abs()
    dpre = (H + 1) * U * A + dpre_extra
    zeta = (dpre + dmu + U * (d + dmu)) * (rs + drs) + d * drs + 2 * U * xh
    DY = dy.double()
    gg = (DY * g.double()).abs()
    m1 = (DY * g.double()).mean(-1, keepdim=True).abs()
    m2 = (DY * g.double() * ref["xh"]).mean(-1, keepdim=True).abs()
    dm1 = (k + 1) * U * gg.sum(-1, keepdim=True) / E + U * m1
    dm2 = ((gg * zeta).sum(-1, keepdim=True) + (k + 2) * U * (gg * xh).sum(-1, keepdim=True)) / E + U * m2
    dxa = ref["dx"].abs()
    ddx = rs * (U * gg + dm1 + xh * dm2 + m2 * zeta + 3 * U * (gg + m1 + xh * m2)) + drs * dxa / rs + U * dxa
    ddx = ddx * (1 + 1e-3)
    W = torch.ones(B, T, H, dtype=f64, device=x.device) if w is None else w.double().abs()
    du = torch.einsum("bth,bte->bhe", W, ddx) + T * U * torch.einsum("bth,bte->bhe", W, dxa)
    dg = (DY.abs() * zeta).sum(1) + (T + 1) * U * (DY * ref["xh"]).abs().sum(1)
    db = T * U * DY.abs().sum(1)
    dp = ddx.sum(1) + T * U * dxa.sum(1)
    l2 = lambda t: t.norm(dim=-1)  # noqa: E731
    return dict(dx=l2(ddx).view(-1), du=l2(du).view(-1), dg=l2(dg), db=l2(db), dp=l2(dp)), \
        dict(dx=ddx, du=du, dg=dg, db=db, dp=dp)


def xattn_ratios(out, ref, tol, keys):
    """Largest error / bound of each output: per element for mean / rstd / y, per row for the gradients."""
    r = {}
    for k in keys:
        o, e = out[k].double(), ref[k]
        if k in ("mean", "rstd", "y"):
            r[k] = float(((o - e.reshape(o.shape)).abs() / tol[k].reshape(o.shape).clamp_min(1e-300)).max())
        else:
            r[k] = rows_within(o.reshape(tol[k].numel(), -1), e.reshape(tol[k].numel(), -1), tol[k].reshape(-1))[1]
    return r


# ================================================================================================ xattn: inputs
def sigma_rows(n, E, gen):
    """(n, E) signs, constant on each column pair (2j, 2j + 1), E / 4 pairs of each sign in a random order."""
    half = torch.tensor([1.0, -1.0]).repeat_interleave(E // 4)
    idx = torch.argsort(torch.rand(n, E // 2, generator=gen), dim=1)
    return half[idx].repeat_interleave(2, dim=1)


def xattn_exact(B, T, E, H, seed, with_bo=True, with_w=True):
    """Exact inputs: pre = c + s sigma (c in Z / 4, s in {1/2, 1, 2}, `sigma_rows`), U[b, h] integers offset by a
    code distinct per (b, h), w[b, t, h] in {0, 1/4, .., 2}, b_o in Z / 2, gamma = +-2^{-1, 0, 1}, beta in Z / 8, and
    x = pre - b_o - sum_h w U.  dy = gg / gamma with gg = p + alpha + beta_r sigma: p = (q, -q) on each column pair,
    alpha, beta_r in {-2, 0, 2} per row, so m1 = alpha, m2 = beta_r and dx = rstd p exactly.
    -> dict(x, u, w, bo, g, b, dy, c, s)"""
    gen = torch.Generator().manual_seed(seed)
    sig = sigma_rows(B * T, E, gen).view(B, T, E)
    s = 2.0 ** torch.randint(-1, 2, (B, T, 1), generator=gen).double()
    c = torch.randint(-16, 17, (B, T, 1), generator=gen).double() / 4
    pre = c + s * sig
    code = torch.arange(1, B * H + 1, dtype=f64).view(B, H, 1)
    u = torch.randint(-3, 4, (B, H, E), generator=gen).double() + code
    w = torch.randint(0, 9, (B, T, H), generator=gen).double() / 4 if with_w else None
    bo = torch.randint(-4, 5, (E,), generator=gen).double() / 2 if with_bo else None
    g = 2.0 ** torch.randint(-1, 2, (E,), generator=gen).double() * (1 - 2 * torch.randint(0, 2, (E,), generator=gen))
    b = torch.randint(-8, 9, (E,), generator=gen).double() / 8
    W = torch.ones(B, T, H, dtype=f64) if w is None else w
    x = pre - torch.einsum("bth,bhe->bte", W, u) - (bo if bo is not None else 0)
    q = torch.randint(-3, 4, (B, T, E // 2), generator=gen).double()
    p = torch.stack([q, -q], -1).view(B, T, E)
    alpha = 2.0 * torch.randint(-1, 2, (B, T, 1), generator=gen)
    beta_r = 2.0 * torch.randint(-1, 2, (B, T, 1), generator=gen)
    dy = (p + alpha + beta_r * sig) / g
    out = dict(x=x, u=u, w=w, bo=bo, g=g, b=b, dy=dy, c=c, s=s, p=p)
    for k, v in out.items():
        assert v is None or representable(v), k
    return {k: (v.float() if v is not None and k not in ("c", "s", "p") else v) for k, v in out.items()}


def xattn_family(name, B, T, E, H, gen, with_bo=True, with_w=True, p_drop=0.1):
    """Bounded-check inputs of one family: fp32 (x, u, w, bo, g, b, dy).  pre is x plus sum_h w U with U ~ N(0, 1/H):
      model     x ~ N(0, 1), gamma ~ U[0.5, 1.5], beta ~ N(0, 0.2)
      offset    x = 1e3 + N(0, 1): the mean's rounding dominates
      flat      x = c + 1e-4 N(0, 1), U ~ 1e-4 N(0, 1): variance far below eps_ln
      outlier   model with one element per row times 100
    w: dropout keep-weights in {0, 1 / (1 - p)}, with whole heads of some sequences zeroed."""
    x = torch.randn(B, T, E, generator=gen)
    u = torch.randn(B, H, E, generator=gen) / math.sqrt(H)
    if name == "offset":
        x = x + 1e3
    elif name == "flat":
        x = torch.randn(B, T, 1, generator=gen) + 1e-4 * x
        u = 1e-4 * u
    elif name == "outlier":
        j = torch.randint(0, E, (B * T,), generator=gen)
        x.view(B * T, E)[torch.arange(B * T), j] *= 100
    w = None
    if with_w:
        w = (torch.rand(B, T, H, generator=gen) >= p_drop).float() / (1 - p_drop)
        w[0, :, 0] = 0                               # a whole head of sequence 0 dropped
    bo = 0.1 * torch.randn(E, generator=gen) if with_bo else None
    g = 0.5 + torch.rand(E, generator=gen)
    b = 0.2 * torch.randn(E, generator=gen)
    dy = torch.randn(B, T, E, generator=gen)
    return x, u, w, bo, g, b, dy


def emulate_xattn(x, u, w, bo, g, b, eps, dy):
    """The kernels' arithmetic in fp32 torch (CPU): pre, mean, biased variance, rsqrt, y; the backward from the
    stored statistics, du / partials summed over t."""
    B, T, E = x.shape
    W = torch.ones(B, T, u.shape[1]) if w is None else w
    pre = x + (bo if bo is not None else 0) + torch.einsum("bth,bhe->bte", W, u)
    mu = pre.sum(-1, keepdim=True) / E
    rs = torch.rsqrt(((pre - mu) ** 2).sum(-1, keepdim=True) / E + eps)
    xh = (pre - mu) * rs
    y = xh * g + b
    gg = dy * g
    m1 = gg.sum(-1, keepdim=True) / E
    m2 = (gg * xh).sum(-1, keepdim=True) / E
    dp = rs * (gg - m1 - xh * m2)
    return dict(mean=mu.view(-1), rstd=rs.view(-1), y=y, dx=dp, du=torch.einsum("bth,bte->bhe", W, dp),
                dg=(dy * xh).sum(1), db=dy.sum(1), dp=dp.sum(1))


def check_xattn(out, x, u, w, bo, g, b, eps, dy, what, log=print, dpre_extra=0.0):
    """Forward per element and backward per row against fp64 (the backward given the kernel's statistics, whose error
    against fp64 is measured); -> {fault: ratio by which the check that targets it sees it}."""
    ref = xattn_model(x, u, w, bo, g, b, eps, dy)
    ft = xattn_fwd_tol(ref, x, u, w, bo, g, eps, dpre_extra)
    worst = xattn_ratios(out, ref, ft, ("mean", "rstd", "y"))
    dmu = (out["mean"].double() - ref["mean"]).abs()
    drs = (out["rstd"].double() - ref["rstd"]).abs()
    bt, _ = xattn_bwd_tol(ref, x, u, w, bo, g, dy, dmu, drs, dpre_extra)
    worst.update(xattn_ratios(out, ref, bt, ("dx", "du", "dg", "db", "dp")))
    log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, (what, worst)
    seen = {}
    for f in XF_FAULTS:
        seen[f] = xattn_ratios(out, xattn_model(x, u, w, bo, g, b, eps, fault=f), ft, ("y",))["y"]
    for f in XB_FAULTS:
        seen[f] = max(xattn_ratios(out, xattn_model(x, u, w, bo, g, b, eps, dy, fault=f), bt,
                                   ("dx", "du", "dg", "db", "dp")).values())
    return worst, seen


# ================================================================================================ ln_l2norm: model
def ln_model(z, g, b, eps_ln, eps_norm, de=None, dn=None, stats=None, fault=None, rows=None):
    """fp64 LayerNorm -> normalize, forward and backward with F.normalize's semantics: a row with ||e|| < eps_norm
    (fp32 eps, as the kernel gets it) is divided by eps and its gradient is dn / eps, no projection.  stats: (rows, 3)
    (mean, rstd, inv) to use in place of the fp64 ones.  dgamma / dbeta as the kernel's partials per block of 8 rows.
    rows: the rows the kernel is given when z, de, dn carry padding rows after them (`rows_past_end`)."""
    Z, G, Bt = z.double(), g.double(), b.double()
    n_all, D = Z.shape
    rows = n_all if rows is None else rows
    mu = Z.mean(-1, keepdim=True)
    rs = 1.0 / (((Z - mu) ** 2).mean(-1, keepdim=True) + eps_ln).sqrt()
    xh = (Z - mu) * rs
    e = xh * G + Bt
    nrm = e.norm(dim=-1, keepdim=True)
    epsn = float(F32(eps_norm))
    below = nrm < epsn
    inv = 1.0 / nrm.clamp_min(epsn)
    if stats is not None:
        st = stats.double()
        mu, rs, inv = st[:, 0:1], st[:, 1:2], st[:, 2:3]
        xh = (Z[:rows] - mu) * rs
        e = xh * G + Bt
    n = e * inv
    out = dict(mean=mu.view(-1)[:rows], rstd=rs.view(-1)[:rows], inv=inv.view(-1)[:rows], e=e[:rows], n=n[:rows],
               norm=nrm.view(-1)[:rows], below=below.view(-1)[:rows])
    if de is None and dn is None:
        return out
    gr = torch.zeros_like(e) if de is None or (fault == "de_ignored" and dn is not None) else de.double()[:e.shape[0]]
    if dn is not None:
        DN = dn.double()[:e.shape[0]]
        dot = (n * DN).sum(-1, keepdim=True)
        proj = below.logical_not()[:e.shape[0]]
        if fault == "projection_below_eps":
            proj = torch.ones_like(proj)
        elif fault == "projection_omitted":
            proj = torch.zeros_like(proj)
        t = DN - n * torch.where(proj, dot, torch.zeros_like(dot))
        gr = gr + (t if fault == "inv_once" else t * inv)
    gq = gr * G
    m1 = gq.mean(-1, keepdim=True)
    m2 = (gq * xh).mean(-1, keepdim=True)
    dz = rs * (gq - m1 - xh * m2)
    nb = -(-rows // 8)
    pg, pb = gr * xh, gr
    keep = torch.arange(pg.shape[0], device=pg.device) < (nb * 8 if fault == "rows_past_end" else rows)
    if fault == "partial_missing_row":
        keep = keep & (torch.arange(pg.shape[0], device=pg.device) % 8 != 7)
    pad = nb * 8 - pg.shape[0]
    part = lambda t: torch.nn.functional.pad(t * keep[:, None], (0, 0, 0, max(pad, 0)))[:nb * 8].view(nb, 8, D).sum(1)  # noqa: E731
    out.update(dz=dz[:rows], dg=part(pg), db=part(pb), g=gr[:rows])
    return out


def ln_fwd_tol(ref, z, g, eps_ln, eps_norm):
    """Per-element bounds of the forward (one warp per row, `warp_depth` roundings per summand):
        mean     warp_depth u sum |z| / D + u |mean|
        var      as in `xattn_fwd_tol` with eta = dmean + u (d + dmean); rstd: 2^-22 + half the relative error
        e        |gamma| (eta rstd + d drstd + u |xh|) + u |e|
        inv      ss = sum fmaf(e, e): sum (2 |e| de + de^2) + warp_depth u ||e||^2; sqrtf and the division rounded
                 (u each); a row at the clamp: inv = fp32(1 / eps), u inv
        n        de inv + |e| dinv + u |n|
    -> dict(mean, rstd, e, inv, n, dmean, drs)."""
    Z = z.double()
    D = Z.shape[1]
    k = warp_depth(D)
    mu, rs = ref["mean"][:, None], ref["rstd"][:, None]
    dmu = k * U * Z.abs().sum(-1, keepdim=True) / D + U * mu.abs()
    d = (Z - mu).abs()
    eta = dmu + U * (d + dmu)
    var = (d * d).mean(-1, keepdim=True)
    t = 2 * d * eta + eta ** 2 + U * (d + eta) ** 2
    dvar = (t.sum(-1, keepdim=True) + k * U * ((d + eta) ** 2).sum(-1, keepdim=True)) / D + U * var + U * (var + eps_ln)
    r = dvar / (var + eps_ln)
    drs = rs * (0.5 * r + r * r + RSQRT)
    xh = d * rs
    de = (g.double().abs() * (eta * rs + d * drs + U * xh) + U * ref["e"].abs()) * (1 + 1e-3)
    ea = ref["e"].abs()
    nrm = ref["norm"][:, None]
    dss = (2 * ea * de + de * de).sum(-1, keepdim=True) + k * U * (ea + de).pow(2).sum(-1, keepdim=True)
    rel = 0.5 * dss / (nrm * nrm).clamp_min(1e-300) + 2 * U
    inv = ref["inv"][:, None]
    dinv = torch.where(ref["below"][:, None], U * inv, inv * (rel + rel * rel) + U * inv)
    dn = de * inv + ea * dinv + U * ref["n"].abs()
    return dict(mean=dmu.view(-1), rstd=drs.view(-1), e=de, inv=dinv.view(-1), n=dn * (1 + 1e-3), dmean=dmu, drs=drs)


def ln_bwd_tol(ref, z, g, de, dn, dmu, drs, dinv):
    """Per-row bounds of the backward given the forward's stats (errors dmu, drs, dinv measured per row):
        zeta     (dmu + u (d + dmu)) (rstd + drs) + d drs + 2 u |xh|    (x-hat recomputed)
        nh       |gamma| zeta inv + |e| dinv + 2 u |nh|                 (e recomputed, times inv)
        dot      sum |dnh| |dn| + warp_depth u sum |nh dn|
        g        de + (dn - nh dot) inv: inv (|dnh dot| + |nh| ddot + 2 u |nh dot| + u |dn - nh dot|)
                 + |dn - nh dot| (dinv + u inv) + u |g|;  below eps: |dn| (dinv + u inv) + u |g|
        dz       the LayerNorm backward of `xattn_bwd_tol` with gg = g gamma (one rounding) and warp_depth
        partials sum over the block's 8 rows of the elements' bounds plus 8 u sum |terms|
    -> dict(dz, dg, db) of per-row bounds."""
    Z, G = z.double()[:ref["e"].shape[0]], g.double()
    rows, D = Z.shape
    k = warp_depth(D)
    rs, mu, inv = ref["rstd"][:, None], ref["mean"][:, None], ref["inv"][:, None]
    dmu, drs, dinv = dmu[:, None], drs[:, None], dinv[:, None]
    d = (Z - mu).abs()
    xh = d * rs
    zeta = (dmu + U * (d + dmu)) * (rs + drs) + d * drs + 2 * U * xh
    ea, ga = ref["e"].abs(), ref["g"].abs()
    nh = ea * inv
    dnh = G.abs() * zeta * inv + ea * dinv + 2 * U * nh
    dg = torch.zeros_like(ea)
    if dn is not None:
        DN = dn.double()[:rows]
        dot = (ref["n"] * DN).sum(-1, keepdim=True).abs()
        ddot = (dnh * DN.abs()).sum(-1, keepdim=True) + k * U * (nh * DN.abs()).sum(-1, keepdim=True)
        t = (DN.abs() + nh * dot)
        above = inv * (dnh * dot + nh * ddot + 2 * U * nh * dot + U * t) + t * (dinv + U * inv)
        below = DN.abs() * (dinv + U * inv)
        dg = torch.where(ref["below"][:, None], below, above)
    dg = (dg + U * ga) * (1 + 1e-3)
    gq = ga * G.abs()
    dgq = G.abs() * dg + U * gq
    m1 = (ref["g"] * G).mean(-1, keepdim=True).abs()
    m2 = (ref["g"] * G * (Z - mu) * rs).mean(-1, keepdim=True).abs()
    dm1 = (dgq.sum(-1, keepdim=True) + k * U * gq.sum(-1, keepdim=True)) / D + U * m1
    dm2 = ((dgq * xh + gq * zeta).sum(-1, keepdim=True) + (k + 1) * U * (gq * xh).sum(-1, keepdim=True)) / D + U * m2
    dza = ref["dz"].abs()
    ddz = rs * (dgq + dm1 + xh * dm2 + m2 * zeta + 3 * U * (gq + m1 + xh * m2)) + drs * dza / rs + U * dza
    nb = -(-rows // 8)
    blk = lambda t: torch.nn.functional.pad(t, (0, 0, 0, nb * 8 - rows)).view(nb, 8, D).sum(1)  # noqa: E731
    dpg = blk(dg * xh + ga * zeta + U * ga * xh) + 8 * U * blk(ga * xh)
    dpb = blk(dg) + 8 * U * blk(ga)
    return dict(dz=(ddz * (1 + 1e-3)).norm(dim=1), dg=dpg.norm(dim=1), db=dpb.norm(dim=1))


def emulate_ln(z, g, b, eps_ln, eps_norm, de, dn):
    """The kernels' arithmetic in fp32 torch (CPU), the clamped rows done right."""
    D = z.shape[1]
    mu = z.sum(-1, keepdim=True) / D
    rs = torch.rsqrt(((z - mu) ** 2).sum(-1, keepdim=True) / D + eps_ln)
    xh = (z - mu) * rs
    e = xh * g + b
    nrm = e.norm(dim=-1, keepdim=True)
    inv = 1.0 / torch.clamp_min(nrm, float(F32(eps_norm)))
    n = e * inv
    gr = torch.zeros_like(z) if de is None else de.clone()
    if dn is not None:
        dot = torch.where(nrm < float(F32(eps_norm)), torch.zeros_like(nrm), (n * dn).sum(-1, keepdim=True))
        gr = gr + (dn - n * dot) * inv
    gq = gr * g
    dz = rs * (gq - gq.sum(-1, keepdim=True) / D - xh * (gq * xh).sum(-1, keepdim=True) / D)
    rows = z.shape[0]
    nb = -(-rows // 8)
    blk = lambda t: torch.nn.functional.pad(t, (0, 0, 0, nb * 8 - rows)).view(nb, 8, D).sum(1)  # noqa: E731
    stats = torch.cat([mu, rs, inv], 1)
    return dict(e=e, n=n, stats=stats, mean=mu.view(-1), rstd=rs.view(-1), inv=inv.view(-1), dz=dz, dg=blk(gr * xh),
                db=blk(gr))


def check_ln(out, z, g, b, eps_ln, eps_norm, de, dn, what, rows=None, log=print):
    """e, n, mean, rstd, inv per element and dz, the dgamma / dbeta partials per row against fp64; the backward given
    the kernel's statistics (errors measured).  z, de, dn may carry padding rows past `rows`.
    -> (worst ratios, {fault: ratio by which the targeted check sees it})"""
    rows = z.shape[0] if rows is None else rows
    ref = ln_model(z, g, b, eps_ln, eps_norm, de, dn, rows=rows)
    ft = ln_fwd_tol(ref, z[:rows], g, eps_ln, eps_norm)
    worst = {}
    for k in ("mean", "rstd", "inv", "e", "n"):
        o = out[k].double().reshape(ref[k].shape)
        worst[k] = float(((o - ref[k]).abs() / ft[k].reshape(o.shape).clamp_min(1e-300)).max())
    if de is None and dn is None:
        log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        assert max(worst.values()) <= 1.0, (what, worst)
        return worst, {}
    dmu = (out["mean"].double() - ref["mean"]).abs()
    drs = (out["rstd"].double() - ref["rstd"]).abs()
    dinv = (out["inv"].double() - ref["inv"]).abs()
    bt = ln_bwd_tol(ref, z, g, de, dn, dmu, drs, dinv)
    for k in ("dz", "dg", "db"):
        worst[k] = rows_within(out[k], ref[k], bt[k])[1]
    log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, (what, worst)
    seen = {}
    for f in LN_FAULTS:
        bad = ln_model(z, g, b, eps_ln, eps_norm, de, dn, fault=f, rows=rows)
        seen[f] = max(rows_within(out[k], bad[k], bt[k])[1] for k in ("dz", "dg", "db"))
    return worst, seen


# ================================================================================================ ln_l2norm: inputs
def ln_exact(rows, D, P, seed, eps_norm):
    """Exact inputs around eps_norm.  Columns: S (P = 4^k columns, gamma = 2^-50, beta = 0), T (P columns,
    gamma = beta = 2^-20), the rest gamma = beta = 0.  z = c + s sigma with sigma balanced per row; even rows have
    sigma = -1 on T (e = 0 there: ||e|| = 2^-50 sqrt(P), below 2^-40), odd rows +1 (e = 2^-19 on T; ||e|| = 2^-19 sqrt(P)
    up to 2^-62 relative from S, which fp32 drops: inv = 2^19 / sqrt(P) exactly).  Upstream gradients are small
    integers (dn divided by the row's inv, so that every row's g is O(1)), with the entries that would put terms 2^30
    apart into one sum cancelled by de: g vanishes on T in the even rows and on S in the odd rows.
    -> dict(z, g, b, de, dn)"""
    assert 2 * P + P <= D and (D - 3 * P) % 2 == 0
    gen = torch.Generator().manual_seed(seed)
    S, T = torch.arange(P), torch.arange(P, 2 * P)
    R = torch.arange(2 * P, D)
    g = torch.zeros(D, dtype=f64)
    b = torch.zeros(D, dtype=f64)
    g[S] = 2.0 ** -50
    g[T] = b[T] = 2.0 ** -20
    sig = torch.empty(rows, D, dtype=f64)
    for r in range(rows):
        st = 1.0 if r % 2 else -1.0
        sig[r, S] = torch.tensor([1.0, -1.0], dtype=f64).repeat(P // 2)[torch.randperm(P, generator=gen)]
        sig[r, T] = st
        nr = len(R)
        rest = torch.cat([torch.full(((nr - P) // 2 + (P if st < 0 else 0),), 1.0, dtype=f64),
                          torch.full(((nr - P) // 2 + (P if st > 0 else 0),), -1.0, dtype=f64)])
        sig[r, R] = rest[torch.randperm(nr, generator=gen)]
    s = 2.0 ** torch.randint(-1, 2, (rows, 1), generator=gen).double()
    c = torch.randint(-16, 17, (rows, 1), generator=gen).double() / 4
    z = c + s * sig
    ref = ln_model(z, g, b, 0.0, eps_norm)
    inv = ref["inv"][:, None]
    de = torch.randint(-3, 4, (rows, D), generator=gen).double()
    dn = torch.randint(-3, 4, (rows, D), generator=gen).double() / inv
    on_s, on_t = torch.zeros(D, dtype=torch.bool), torch.zeros(D, dtype=torch.bool)
    on_s[S], on_t[T] = True, True
    even = (torch.arange(rows) % 2 == 0)[:, None]
    de = torch.where(even & on_t, -dn * inv, de)                 # even rows (e on S): g = 0 on T
    dn = torch.where(~even & on_s, torch.zeros_like(dn), dn)     # odd rows (e on T): g = 0 on S
    dot = (ref["n"] * dn).sum(-1, keepdim=True)
    de = torch.where(~even & on_s, ref["n"] * dot * inv, de)
    out = dict(z=z, g=g, b=b, de=de, dn=dn)
    for k, v in out.items():
        assert representable(v), k
    return {k: v.float() for k, v in out.items()}


def ln_family(name, rows, D, gen, pad=0):
    """Bounded-check inputs (rows + pad rows; the pad rows sit past the end the kernel is given):
      model     z ~ N(0, 1), gamma ~ U[0.5, 1.5], beta ~ N(0, 0.2)
      offset    z = 1e3 + N(0, 1)
      flat      z = c + 1e-4 N(0, 1) (variance far below eps_ln)
      outlier   one element per row times 100
      eps       gamma, beta scaled so that ||e|| of the rows cycles through 0.999, 1.001 and 1e3 times eps_norm
    -> (z, g, b, de, dn)"""
    n = rows + pad
    z = torch.randn(n, D, generator=gen)
    if name == "offset":
        z = z + 1e3
    elif name == "flat":
        z = torch.randn(n, 1, generator=gen) + 1e-4 * z
    elif name == "outlier":
        j = torch.randint(0, D, (n,), generator=gen)
        z[torch.arange(n), j] *= 100
    g = 0.5 + torch.rand(D, generator=gen)
    b = 0.2 * torch.randn(D, generator=gen)
    de, dn = torch.randn(n, D, generator=gen), torch.randn(n, D, generator=gen)
    if name == "eps":            # ||e|| = ||zz gamma|| sqrt(var / (var + eps_ln)): the row's spread sets its norm
        b = torch.zeros(D)
        zz = torch.nn.functional.layer_norm(torch.randn(n, D, generator=gen, dtype=f64), (D,), eps=0.0)
        epsn = float(F32(EPS_NORM))
        g = (g.double() * (2e3 * epsn / float((zz * g.double()).norm(dim=1).min()))).float()
        base = (zz * g.double()).norm(dim=1)
        f = torch.tensor([0.999, 1.001, 1e3], dtype=f64)[torch.arange(n) % 3] * epsn / base
        z = (zz * (f ** 2 * EPS_LN / (1 - f ** 2)).sqrt()[:, None]).float()
    return z, g, b, de, dn


def xattn_exact_outputs(d, stats=None, fault=None):
    """The closed form of the exact inputs: fp64 model (given the kernel's statistics), y rounded once to fp32."""
    r = xattn_model(d["x"], d["u"], d["w"], d["bo"], d["g"], d["b"], 0.0, d["dy"], stats=stats, fault=fault)
    r["y"] = r["y"].float().double()
    return r


def exact_mismatch(out, ref, keys):
    return [k for k in keys if not torch.equal(out[k].double().reshape(ref[k].shape), ref[k])]


XATTN_EXACT_SHAPES = [(2, 3, 4, 1, True, True), (3, 2, 12, 2, True, True), (1, 5, 1020, 31, True, True),
                      (3, 2, 1028, 32, False, True), (3, 4, 1028, 4, True, False), (2, 3, 4096, 2, True, True),
                      (8, 16, 1024, 8, True, True), (2, 1, 1024, 1, True, False)]
LN_EXACT_SHAPES = [(9, 256, 64), (17, 512, 64), (8, 1024, 256), (33, 2048, 256)]


def exact_eps(P):
    """eps_norm above the even rows' norm (those rows clamped), equal to it (not clamped), below every norm."""
    return 2.0 ** -40, 2.0 ** (-50 + int(round(math.log2(P))) // 2), 2.0 ** -60


def ln_exact_outputs(d, eps_norm, stats=None, fault=None):
    r = ln_model(d["z"], d["g"], d["b"], 0.0, eps_norm, d["de"], d["dn"], stats=stats, fault=fault)
    for k in ("e", "n"):
        r[k] = r[k].float().double()
    return r


# ================================================================================================ CPU tests
@pytest.mark.parametrize("B,T,E,H,bo,w", XATTN_EXACT_SHAPES)
def test_xattn_exact_builder(B, T, E, H, bo, w):
    """The exact inputs give mean = c, biased variance = s^2, x-hat = +-1, m1 = alpha, m2 = beta_r, dx = p / s; every
    output of the closed form is an fp32 value, and each planted fault changes some output."""
    d = xattn_exact(B, T, E, H, B * T + E + H, bo, w)
    r = xattn_exact_outputs(d)
    assert torch.equal(r["mean"].view(B, T, 1), d["c"]) and torch.equal(r["var"], d["s"] ** 2)
    assert torch.equal(r["xh"].abs(), torch.ones_like(r["xh"]))
    assert torch.equal(r["dx"], d["p"] / d["s"])
    for k in ("y", "dx", "du", "dg", "db", "dp"):
        assert representable(r[k]), k
    changed = {f for f in XF_FAULTS if exact_mismatch(r, xattn_exact_outputs(d, fault=f), ("y",))}
    changed |= {f for f in XB_FAULTS if exact_mismatch(r, xattn_exact_outputs(d, fault=f), ("dx", "du", "dg", "dp"))}
    expect = set(XF_FAULTS + XB_FAULTS) - {"eps_outside"}          # eps_ln = 0 here
    expect -= {"w_neighbour", "du_missing_last"} if T == 1 else set()
    expect -= {"u_prev_seq"} if B == 1 else set()
    expect -= {"du_head_shift"} if H == 1 else set()
    expect -= {"bo_dropped"} if not bo else set()
    expect -= {"w_neighbour", "du_head_shift"} if not w else set()      # every head weighs 1
    expect -= {"group_dropped"} if groups(E) == 1 else set()              # aimed at E = 1028 and 4096
    assert changed >= expect, expect - changed


@pytest.mark.parametrize("rows,D,P", LN_EXACT_SHAPES)
def test_ln_exact_builder(rows, D, P):
    """Exact ln_l2norm inputs: mean = c, variance = s^2, ||e|| = 2^-50 sqrt(P) on even rows and 2^-19 sqrt(P) on odd
    rows (fp32 of the fp64 norm), inv a power of two; every closed-form output is an fp32 value; which rows are
    clamped follows eps_norm; each planted fault changes some output."""
    for eps_norm in exact_eps(P):
        d = ln_exact(rows, D, P, rows + D, eps_norm)
        r = ln_exact_outputs(d, eps_norm)
        k = int(round(math.log2(P))) // 2
        even = torch.arange(rows) % 2 == 0
        assert torch.equal(r["norm"][even], torch.full((int(even.sum()),), 2.0 ** (-50 + k), dtype=f64))
        assert bool((r["norm"][~even].float() == 2.0 ** (-19 + k)).all())
        assert torch.equal(r["below"], torch.tensor([(2.0 ** (-50 + k) if i % 2 == 0 else 2.0 ** (-19 + k)) < eps_norm
                                                     for i in range(rows)]))
        for key in ("e", "n", "dz", "dg", "db"):
            assert representable(r[key]), (key, eps_norm)
        stats = torch.stack([r["mean"], r["rstd"], r["inv"].float().double()], 1)
        r = ln_exact_outputs(d, eps_norm, stats)
        changed = {f for f in LN_FAULTS if exact_mismatch(r, ln_exact_outputs(d, eps_norm, stats, f), ("dz", "dg", "db"))}
        expect = set(LN_FAULTS) - {"rows_past_end"} - ({"partial_missing_row"} if rows < 8 else set())
        if not bool(r["below"].any()):
            expect.discard("projection_below_eps")
        assert changed >= expect, (eps_norm, expect - changed)


def xattn_cases():
    """(family, B, T, E, H, bo, w) of the CPU checker test: small, every layout the kernel takes."""
    return [("model", 2, 3, 1028, 4, True, True), ("model", 1, 4, 4096, 2, True, True), ("offset", 3, 2, 12, 2, True, True),
            ("flat", 2, 3, 64, 3, False, True), ("outlier", 2, 2, 256, 1, True, False), ("model", 2, 5, 1024, 8, True, True)]


def test_xattn_checker_accepts_emulation_and_rejects_faults():
    """check_xattn accepts an fp32 emulation of both kernels and rejects every planted fault in some case."""
    tally = FaultTally()
    for fam, B, T, E, H, bo, w in xattn_cases():
        gen = torch.Generator().manual_seed(B * T * E + H)
        x, u, ww, bb, g, b, dy = xattn_family(fam, B, T, E, H, gen, bo, w)
        out = emulate_xattn(x, u, ww, bb, g, b, EPS_LN, dy)
        _, seen = check_xattn(out, x, u, ww, bb, g, b, EPS_LN, dy, f"emulation {fam}", log=lambda *a: None)
        tally.add(seen)
    tally.report("xattn emulation")


def test_ln_checker_accepts_emulation_and_rejects_faults():
    """check_ln accepts an fp32 emulation of both kernels (clamped rows without the projection) and rejects every
    planted fault in some case; rows_past_end through padding rows after the last one."""
    tally = FaultTally()
    for fam, rows, D in (("model", 9, 64), ("eps", 12, 128), ("offset", 7, 33), ("outlier", 17, 512), ("flat", 9, 31),
                         ("model", 3, 1)):
        for mode in ("de", "dn", "both"):
            gen = torch.Generator().manual_seed(rows * D + len(mode))
            pad = (-rows) % 8
            z, g, b, de, dn = ln_family(fam, rows, D, gen, pad)
            de_, dn_ = (de if mode != "dn" else None), (dn if mode != "de" else None)
            out = emulate_ln(z[:rows], g, b, EPS_LN, EPS_NORM, None if de_ is None else de_[:rows],
                             None if dn_ is None else dn_[:rows])
            _, seen = check_ln(out, z, g, b, EPS_LN, EPS_NORM, de_, dn_, f"emulation {fam} {mode}", rows=rows,
                               log=lambda *a: None)
            tally.add(seen)
    tally.report("ln_l2norm emulation")


@pytest.mark.parametrize("fn", ["xattn_ln_fwd", "xattn_ln_bwd", "ln_l2norm_fwd", "ln_l2norm_bwd"])
def test_wrappers_reject_wrong_dtype_shape_layout(fn):
    """functional.xattn_ln_* / ln_l2norm_* check dtype, shape and contiguity of every buffer before anything else
    (the kernels read them as contiguous fp32 of the given shape), so the error names the argument, on any device."""
    from preference_guided_image_captioning_alignment_b200 import _lib, functional as F
    B, T, E, H, rows, D = 2, 3, 8, 2, 5, 8
    x, u, w = torch.zeros(B, T, E), torch.zeros(B, H, E), torch.ones(B, T, H)
    g, b, m = torch.ones(E), torch.zeros(E), torch.zeros(B * T)
    z, st = torch.zeros(rows, D), torch.zeros(rows, 3)
    calls = {
        "xattn_ln_fwd": lambda **k: F.xattn_ln_fwd(k.get("x", x), k.get("u", u), k.get("w", w), k.get("bo", b),
                                                   k.get("g", g), k.get("b", b), 1e-5),
        "xattn_ln_bwd": lambda **k: F.xattn_ln_bwd(k.get("x", x), x, u, k.get("w", w), k.get("bo", b), k.get("g", g),
                                                   k.get("m", m), m),
        "ln_l2norm_fwd": lambda **k: F.ln_l2norm_fwd(z, k.get("g", g), k.get("b", b), 1e-5, 1e-12),
        "ln_l2norm_bwd": lambda **k: F.ln_l2norm_bwd(z, k.get("g", g), b, k.get("st", st), z, k.get("dn", z)),
    }
    bad = [dict(g=g.half()), dict(g=g.double()), dict(g=torch.ones(E + 4)), dict(g=torch.ones(2 * E)[::2])]
    if fn.startswith("xattn"):
        bad += [dict(w=w.bool()), dict(w=w.half()), dict(w=w.double()), dict(w=torch.ones(B, T, H + 1)),
                dict(bo=b.bfloat16())]
    if fn == "xattn_ln_bwd":
        bad += [dict(m=m.double())]
    if fn == "ln_l2norm_bwd":
        bad += [dict(st=torch.zeros(rows, 2)), dict(dn=torch.zeros(D, rows).t())]
    if fn == "ln_l2norm_fwd":
        bad += [dict(b=b.bfloat16())]
    for kw in bad:
        with pytest.raises(_lib.PgicaError, match="contiguous float32"):
            calls[fn](**kw)
    with pytest.raises(_lib.PgicaError, match="no CPU fallback"):          # well-formed: only the device is wrong
        calls[fn]()


def test_keep_weights_reach_the_kernel_as_fp32(monkeypatch):
    """collapsed_cross_attention_ln hands keep-weights given as bool, fp16 or fp64 to the kernel as fp32 values."""
    from preference_guided_image_captioning_alignment_b200 import prologue
    seen = []

    def fake_fwd(x, u, w, out_bias, gamma, beta, eps):
        seen.append(w)
        return torch.zeros_like(x), torch.zeros(x.shape[0] * x.shape[1]), torch.ones(x.shape[0] * x.shape[1])

    monkeypatch.setattr(prologue.F, "xattn_ln_fwd", fake_fwd)
    B, T, E, H = 2, 3, 8, 2
    mha, norm = torch.nn.MultiheadAttention(E, H, batch_first=True), torch.nn.LayerNorm(E)
    keep = torch.rand(B, T, H, generator=torch.Generator().manual_seed(0)) >= 0.5
    for k in (keep, keep.half() * 2, keep.double() * 2):
        prologue.collapsed_cross_attention_ln(torch.randn(B, T, E), torch.randn(B, 1, E), mha, norm, keep_weights=k)
        assert seen[-1].dtype == torch.float32 and torch.equal(seen[-1], k.float())


def test_ln_l2norm_rejects_rows_its_backward_cannot_take():
    """prologue.ln_l2norm raises at the call for D > 2048 (the forward takes 8192, the backward 2048), before any
    forward work, instead of failing in the backward."""
    from preference_guided_image_captioning_alignment_b200 import prologue
    with pytest.raises(ValueError, match="2048"):
        prologue.ln_l2norm(torch.randn(4, 4096), torch.nn.LayerNorm(4096))


def test_normalized_carrier_returns_the_twin_only_for_its_own_call():
    """F.normalize on the carrier gives the precomputed twin for p = 2, dim = -1 and eps = 1e-12 (positional or by
    keyword), and computes afresh for another eps passed either way and whenever out= is given."""
    from preference_guided_image_captioning_alignment_b200 import prologue
    fn = torch.nn.functional.normalize
    base = torch.randn(4, 8, generator=torch.Generator().manual_seed(1))
    t = base.as_subclass(prologue.NormalizedCarrier)
    twin = torch.full((4, 8), 7.0)
    t._pgica_normalized = twin
    assert fn(t, 2.0, -1) is twin and fn(t, p=2, dim=-1, eps=1e-12) is twin and fn(t, 2.0, 1, 1e-12) is twin
    for got in (fn(t, 2.0, -1, 10.0), fn(t, p=2.0, dim=-1, eps=10.0)):
        assert got is not twin and torch.equal(got, fn(base, 2.0, -1, 10.0))
    out = torch.empty(4, 8)
    got = fn(t, 2.0, -1, 1e-12, out)
    assert got is not twin and torch.equal(out, fn(base, dim=-1))
    out2 = torch.empty(4, 8)
    fn(t, dim=-1, out=out2)
    assert torch.equal(out2, fn(base, dim=-1))


# ================================================================================================ GPU tests
@pytest.fixture(scope="module")
def F(cuda_device):
    from preference_guided_image_captioning_alignment_b200 import _lib, functional
    lib = _lib.load()
    assert lib.pgica_device_check() == 0, lib.pgica_last_error()
    return functional


def run_xattn(F, dev, x, u, w, bo, g, b, eps, dy):
    put = lambda t: None if t is None else t.to(dev)  # noqa: E731
    x, u, w, bo, g, b, dy = map(put, (x, u, w, bo, g, b, dy))
    y, mean, rstd = F.xattn_ln_fwd(x, u, w, bo, g, b, eps)
    dx, du, dg, db, dp = F.xattn_ln_bwd(dy, x, u, w, bo, g, mean, rstd)
    return dict(y=y, mean=mean, rstd=rstd, dx=dx, du=du, dg=dg, db=db, dp=dp), (x, u, w, bo, g, b, dy)



# ------------------------------------------------------------------------------------------------ 1. exact
@pytest.mark.gpu
@pytest.mark.parametrize("B,T,E,H,bo,w", XATTN_EXACT_SHAPES)
def test_xattn_exact(F, cuda_device, B, T, E, H, bo, w):
    """Exact inputs (`xattn_exact`): mean == c, y == the closed form given the kernel's rstd (one rounding), dx, du
    and the dgamma / dbeta / db_o partials == the closed form bit for bit; rstd within 2 ulp of 1 / s (whether it is
    exact is printed); each planted fault the inputs can show is rejected."""
    d = xattn_exact(B, T, E, H, B * T + E + H, bo, w)
    out, _ = run_xattn(F, cuda_device, d["x"], d["u"], d["w"], d["bo"], d["g"], d["b"], 0.0, d["dy"])
    out = {k: v.cpu() for k, v in out.items()}
    rs_exact = 1.0 / d["s"].view(-1)
    assert torch.equal(out["mean"].double(), d["c"].view(-1))
    assert bool(((out["rstd"].double() - rs_exact).abs() <= RSQRT * rs_exact).all())
    exact = torch.equal(out["rstd"].double(), rs_exact)
    ref = xattn_exact_outputs(d, stats=(out["mean"], out["rstd"]))
    bad = exact_mismatch(out, ref, ("y", "dx", "du", "dg", "db", "dp"))
    assert bad == [], (bad, {k: float((out[k].double().reshape(ref[k].shape) - ref[k]).abs().max()) for k in bad})
    rejected = [f for f in XF_FAULTS if exact_mismatch(out, xattn_exact_outputs(d, fault=f), ("y",))]
    rejected += [f for f in XB_FAULTS if exact_mismatch(out, xattn_exact_outputs(d, (out["mean"], out["rstd"]), f),
                                                         ("dx", "du", "dg", "dp"))]
    print(f"[exact] xattn B={B} T={T} E={E} H={H} bo={bo} w={w}: bit-exact; rsqrtf exact at powers of four: {exact}; "
          f"faults rejected: {', '.join(rejected)} ({card()})")
    for f in ("head_dropped", "bo_dropped" if bo else None, "group_dropped" if groups(E) > 1 else None,
              "m2_dropped", "dgamma_from_dy", "dbo_from_dy"):
        assert f is None or f in rejected, f


@pytest.mark.gpu
@pytest.mark.parametrize("rows,D,P", LN_EXACT_SHAPES)
def test_ln_l2norm_exact(F, cuda_device, rows, D, P):
    """Exact inputs around eps_norm (`ln_exact`), eps_norm above / at / below the even rows' norm: mean == c; inv ==
    the fp32 power of two; e, n, dz and the dgamma / dbeta partials == the closed form bit for bit given the kernel's
    rstd; a clamped row gets de + dn inv, no projection, and the rows above (and at) eps keep it."""
    for eps_norm in exact_eps(P):
        d = ln_exact(rows, D, P, rows + D, eps_norm)
        z, g, b, de, dn = (d[k].to(cuda_device) for k in ("z", "g", "b", "de", "dn"))
        e, n, st = F.ln_l2norm_fwd(z, g, b, 0.0, eps_norm)
        dz, dg, db = F.ln_l2norm_bwd(z, g, b, st, de, dn)
        out = dict(e=e.cpu(), n=n.cpu(), dz=dz.cpu(), dg=dg.cpu(), db=db.cpu())
        st = st.cpu()
        r0 = ln_exact_outputs(d, eps_norm)
        assert torch.equal(st[:, 0].double(), r0["mean"])
        assert bool(((st[:, 1].double() - r0["rstd"]).abs() <= RSQRT * r0["rstd"]).all())
        exact = torch.equal(st[:, 1].double(), r0["rstd"])
        if exact:
            assert torch.equal(st[:, 2].double(), r0["inv"].float().double())
        ref = ln_exact_outputs(d, eps_norm, st)
        bad = exact_mismatch(out, ref, ("e", "n", "dz", "dg", "db"))
        assert bad == [], (eps_norm, bad)
        rejected = [f for f in LN_FAULTS if exact_mismatch(out, ln_exact_outputs(d, eps_norm, st, f), ("dz", "dg", "db"))]
        print(f"[exact] ln_l2norm rows={rows} D={D} eps_norm=2^{int(math.log2(eps_norm))} clamped rows "
              f"{int(ref['below'].sum())}: bit-exact; rsqrtf exact: {exact}; faults rejected: {', '.join(rejected)}")
        if bool(ref["below"].any()):
            assert "projection_below_eps" in rejected
        assert "projection_omitted" in rejected and "inv_once" in rejected and "de_ignored" in rejected


# ------------------------------------------------------------------------------------------------ 2. bounded
XATTN_MODEL = [(8, 128, 1024, 1, True, False), (8, 128, 1024, 8, True, True), (16, 128, 1024, 16, True, True)]
XATTN_EDGES = [(1, 1, 4, 1, False, False), (3, 2, 12, 2, True, True), (3, 127, 1020, 31, True, True),
               (1, 2, 1028, 32, False, True), (3, 2, 1028, 2, True, False), (1, 127, 4096, 1, True, False),
               (3, 2, 4096, 32, True, True), (3, 1, 12, 2, True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["model", "offset", "flat", "outlier"])
def test_xattn_bounded_fp64(F, cuda_device, fam):
    """Both kernels against fp64 at the model's shapes (B in {8, 16}, T = 128, E = 1024, H in {1 (eval), 8, 16}) and
    at the edges (E in {4, 12, 1020, 1028, 4096}, T in {1, 2, 127}, H in {1, 2, 31, 32}, B in {1, 3}, with and without
    b_o and w; dropout keep-weights with a whole head zeroed): y, mean, rstd per element, the gradients per row
    (`check_xattn`); every planted fault rejected in some case."""
    worst, tally = 0.0, FaultTally()
    for i, (B, T, E, H, bo, w) in enumerate(XATTN_MODEL + XATTN_EDGES):
        gen = torch.Generator().manual_seed(1000 * i + len(fam))
        inp = xattn_family(fam, B, T, E, H, gen, bo, w)
        out, dev_inp = run_xattn(F, cuda_device, *inp[:6], EPS_LN, inp[6])
        r, seen = check_xattn(out, *dev_inp[:6], EPS_LN, dev_inp[6], f"xattn {fam} B={B} T={T} E={E} H={H} bo={bo} w={w}")
        worst = max(worst, max(r.values()))
        tally.add(seen)
    report(f"xattn {fam} all shapes", worst)
    tally.report(f"xattn {fam}", optional=() if fam == "model" else ("eps_outside", "unbiased_var", "group_dropped"))


LN_MODEL = [(8, 512), (64, 512), (4096, 512)]
LN_EDGES = [(1, 1), (7, 31), (9, 33), (8, 1024), (297, 2048), (9, 2048), (7, 1024), (1, 33)]


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["model", "offset", "flat", "outlier", "eps"])
def test_ln_l2norm_bounded_fp64(F, cuda_device, fam):
    """ln_l2norm at the model's shape (D = 512, rows in {8, 64, 4096}) and the edges (D in {1, 31, 33, 1024, 2048},
    rows in {1, 7, 8, 9, 8k + 1}; D = 8192 forward only), with de only, dn only and both, padding rows after the last
    row: e, n, mean, rstd, inv per element, dz and the partials per row (`check_ln`); every planted fault rejected."""
    worst, tally = 0.0, FaultTally()
    for i, (rows, D) in enumerate(LN_MODEL + LN_EDGES + [(9, 8192)]):
        if fam == "eps" and D < 8:
            continue
        for mode in (("de", "dn", "both") if D <= 2048 else ("fwd",)):
            gen = torch.Generator().manual_seed(100 * i + len(mode) + len(fam))
            pad = (-rows) % 8 or 8
            z, g, b, de, dn = (t.to(cuda_device) for t in ln_family(fam, rows, D, gen, pad))
            de_ = de if mode in ("de", "both") else None
            dn_ = dn if mode in ("dn", "both") else None
            e, n, st = F.ln_l2norm_fwd(z[:rows], g, b, EPS_LN, EPS_NORM)
            out = dict(e=e, n=n, mean=st[:, 0], rstd=st[:, 1], inv=st[:, 2])
            if mode != "fwd":
                out["dz"], out["dg"], out["db"] = F.ln_l2norm_bwd(z[:rows], g, b, st, None if de_ is None else de_[:rows],
                                                                  None if dn_ is None else dn_[:rows])
            r, seen = check_ln(out, z, g, b, EPS_LN, EPS_NORM, de_, dn_, f"ln_l2norm {fam} rows={rows} D={D} {mode}",
                               rows=rows)
            worst = max(worst, max(r.values()))
            tally.add(seen)
    report(f"ln_l2norm {fam} all shapes", worst)
    # eps: dn inv is 1e12 times de there, so dropping de is below fp32 resolution
    tally.report(f"ln_l2norm {fam}", optional=("de_ignored",) if fam == "eps" else ("projection_below_eps",))


# ------------------------------------------------------------------------------------------------ 4. the wiring
def gemm_err(a, b, k):
    """Bound on |fl(A B) - A B| for an fp32 GEMM with k products per entry: k u |A| |B|."""
    return k * U * (a.abs() @ b.abs())


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,E,H", [(8, 128, 1024, 8), (3, 17, 256, 4)])
def test_collapsed_cross_attention_fp64(F, cuda_device, B, T, E, H):
    """prologue.collapsed_cross_attention_ln against nn.MultiheadAttention + nn.LayerNorm run in fp64, in eval mode
    and in train mode with given keep-weights (a bool mask as well): y per element, and per row the gradients of
    text, vision, the v third of in_proj_weight / in_proj_bias, out_proj weight and bias, gamma and beta (bounds:
    the kernels' plus the torch fp32 GEMMs around them, k u |A| |B| each); the q / k gradients are exact zeros."""
    import copy
    from preference_guided_image_captioning_alignment_b200 import prologue
    torch.manual_seed(B * T + H)
    dev = cuda_device
    mha = torch.nn.MultiheadAttention(E, H, dropout=0.1, batch_first=True).to(dev)
    norm = torch.nn.LayerNorm(E).to(dev)
    with torch.no_grad():
        norm.weight.uniform_(0.5, 1.5)
        norm.bias.normal_(0, 0.2)
        mha.out_proj.bias.normal_(0, 0.1)
        mha.in_proj_bias.normal_(0, 0.1)
    mha64, norm64 = copy.deepcopy(mha).double(), copy.deepcopy(norm).double()
    text, vis, up = torch.randn(B, T, E, device=dev), torch.randn(B, 1, E, device=dev), torch.randn(B, T, E, device=dev)
    hd = E // H
    worst = 0.0
    for mode in ("eval", "train"):
        keep = None
        if mode == "train":
            keep = torch.rand(B, T, H, device=dev) >= 0.1
            keep[0, :, 0] = False
        kw = None if keep is None else keep.float() / 0.9
        mha.train(mode == "train")
        mha64.eval()
        t32, v32 = text.clone().requires_grad_(True), vis.clone().requires_grad_(True)
        for p in list(mha.parameters()) + list(norm.parameters()) + list(mha64.parameters()) + list(norm64.parameters()):
            p.grad = None
        y = prologue.collapsed_cross_attention_ln(t32, v32, mha, norm, keep_weights=kw)
        (y * up).sum().backward()
        # fp64 reference: the stock modules; dropout as the keep-mask on the (all-ones) attention weights per head
        t64, v64 = text.double().requires_grad_(True), vis.double().requires_grad_(True)
        if keep is None:
            att = mha64(t64, v64, v64, need_weights=False)[0]
        else:
            wv, bv = mha64.in_proj_weight[2 * E:], mha64.in_proj_bias[2 * E:]
            v = (v64.reshape(B, E) @ wv.t() + bv).view(B, 1, H, hd) * kw.double().unsqueeze(-1)
            att = v.reshape(B, T, E) @ mha64.out_proj.weight.t() + mha64.out_proj.bias
        y64 = norm64(t64 + att)
        (y64 * up.double()).sum().backward()
        # the kernel's inputs in fp64 and the error the torch GEMMs put into U
        with torch.no_grad():
            wv, bv, wo = (p.double() for p in (mha.in_proj_weight[2 * E:], mha.in_proj_bias[2 * E:], mha.out_proj.weight))
            vb = vis.double().reshape(B, E)
            v = vb @ wv.t() + bv
            dv_ = gemm_err(vb, wv.t(), E + 1)
            if keep is None:
                u = (v @ wo.t()).unsqueeze(1)
                du_ = (dv_ @ wo.t().abs() + gemm_err(v, wo.t(), E)).unsqueeze(1)
                w = None
            else:
                u = torch.einsum("bhd,ehd->bhe", v.view(B, H, hd), wo.view(E, H, hd))
                du_ = torch.einsum("bhd,ehd->bhe", dv_.view(B, H, hd), wo.abs().view(E, H, hd)) + \
                    hd * U * torch.einsum("bhd,ehd->bhe", v.abs().view(B, H, hd), wo.abs().view(E, H, hd))
                w = kw
            Wt = torch.ones(B, T, u.shape[1], device=dev, dtype=f64) if w is None else w.double()
            extra = torch.einsum("bth,bhe->bte", Wt, du_) + U * u.abs().sum(1, keepdim=True)
            x, g, b, bo = text, norm.weight.detach(), norm.bias.detach(), mha.out_proj.bias.detach()
            ref = xattn_model(x, u, w, bo, g, b, norm.eps, up)
            ft = xattn_fwd_tol(ref, x, u, w, bo, g, norm.eps, extra)
            r = {"y": xattn_ratios(dict(y=y.detach()), dict(y=y64.detach()), ft, ("y",))["y"]}
            rows_b, el = xattn_bwd_tol(ref, x, u, w, bo, g, up, ft["dmean"], ft["drs"], extra)
            r["text"] = rows_within(t32.grad.view(B * T, E), t64.grad.view(B * T, E), rows_b["dx"])[1]
            # every downstream gradient is linear in (du, db_o, dgamma, dbeta): propagate the element bounds through
            # |coefficients| and add the fp32 GEMMs' k u |A| |B|
            du64 = torch.einsum("bth,bte->bhe", Wt, ref["dx"])
            dua, due = du64.abs(), el["du"]
            if keep is None:
                dv_g, dv_e = du64[:, 0] @ wo, due[:, 0] @ wo.abs() + gemm_err(dua[:, 0], wo, E)
                dwo_e = due[:, 0].t() @ v.abs() + dua[:, 0].t() @ dv_ + gemm_err(dua[:, 0].t(), v, B)
            else:
                dv_e = (torch.einsum("bhe,ehd->bhd", due, wo.abs().view(E, H, hd)) + E * U *
                        torch.einsum("bhe,ehd->bhd", dua, wo.abs().view(E, H, hd))).reshape(B, E)
                dv_g = torch.einsum("bhe,ehd->bhd", du64, wo.view(E, H, hd)).reshape(B, E)
                dwo_e = (torch.einsum("bhe,bhd->ehd", due, v.abs().view(B, H, hd)) +
                         torch.einsum("bhe,bhd->ehd", dua, dv_.view(B, H, hd)) + B * U *
                         torch.einsum("bhe,bhd->ehd", dua, v.abs().view(B, H, hd))).reshape(E, E)
            dvis_e = dv_e @ wv.abs() + gemm_err(dv_g, wv, E)
            dwv_e = dv_e.t() @ vb.abs() + gemm_err(dv_g.t(), vb, B)
            dbv_e = dv_e.sum(0) + B * U * dv_g.abs().sum(0)
            col = lambda t: t.reshape(-1, 1)  # noqa: E731
            sums = lambda p, pe: (pe.sum(0) + B * U * p.abs().sum(0))  # noqa: E731
            checks = [("vision", v32.grad.view(B, E), v64.grad.view(B, E), dvis_e.norm(dim=1)),
                      ("in_proj_weight v", mha.in_proj_weight.grad[2 * E:], mha64.in_proj_weight.grad[2 * E:],
                       dwv_e.norm(dim=1)),
                      ("in_proj_bias v", col(mha.in_proj_bias.grad[2 * E:]), col(mha64.in_proj_bias.grad[2 * E:]), dbv_e),
                      ("out_proj weight", mha.out_proj.weight.grad, mha64.out_proj.weight.grad, dwo_e.norm(dim=1)),
                      ("out_proj bias", col(mha.out_proj.bias.grad), col(mha64.out_proj.bias.grad),
                       sums(ref["dp"], el["dp"])),
                      ("gamma", col(norm.weight.grad), col(norm64.weight.grad), sums(ref["dg"], el["dg"])),
                      ("beta", col(norm.bias.grad), col(norm64.bias.grad), sums(ref["db"], el["db"]))]
            for nm, got, want, bound in checks:
                r[nm] = rows_within(got, want, bound * (1 + 1e-3))[1]
            assert float(mha.in_proj_weight.grad[:2 * E].abs().max()) == 0.0
            assert float(mha.in_proj_bias.grad[:2 * E].abs().max()) == 0.0
        print(f"[worst error/bound] collapsed cross-attention {mode} B={B} T={T} E={E} H={H}: " +
              " ".join(f"{k} {v:.3g}" for k, v in r.items()))
        assert max(r.values()) <= 1.0, (mode, r)
        worst = max(worst, max(r.values()))
    report(f"collapsed cross-attention B={B} T={T} E={E} H={H}", worst)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,D", [(64, 512), (9, 2048), (4096, 512)])
def test_ln_l2norm_wiring_fp64(F, cuda_device, rows, D):
    """prologue.ln_l2norm against fp64 layer_norm -> F.normalize autograd (upstream gradients on both outputs, three
    constant rows): e, n per element, dz, dgamma, dbeta per row; and the promise `_pgica_unit_norm`
    makes to the bounded NT-Xent paths: every row of n above eps has an fp64 norm within (D / 32 + 5) / 2 + 3 units of
    2^-24 of 1."""
    from preference_guided_image_captioning_alignment_b200 import prologue
    gen = torch.Generator().manual_seed(rows + D)
    z, g, b, de, dn = (t.to(cuda_device) for t in ln_family("model", rows, D, gen))
    z[:3] = z[:3] * 0 + z[:3, :1]                    # constant rows: e = beta
    norm = torch.nn.LayerNorm(D).to(cuda_device)
    with torch.no_grad():
        norm.weight.copy_(g)
        norm.bias.copy_(b)
    zz = z.clone().requires_grad_(True)
    e, n = prologue.ln_l2norm(zz, norm)
    ((e * de).sum() + (n * dn).sum()).backward()
    z64 = z.double().requires_grad_(True)
    g64, b64 = g.double().requires_grad_(True), b.double().requires_grad_(True)
    e64 = torch.nn.functional.layer_norm(z64, (D,), g64, b64, EPS_LN)
    n64 = torch.nn.functional.normalize(e64, dim=-1, eps=float(F32(EPS_NORM)))
    ((e64 * de.double()).sum() + (n64 * dn.double()).sum()).backward()
    ref = ln_model(z, g, b, EPS_LN, EPS_NORM, de, dn)
    ft = ln_fwd_tol(ref, z, g, EPS_LN, EPS_NORM)
    r = {"e": float(((e.double() - e64).abs() / ft["e"]).max()), "n": float(((n.double() - n64).abs() / ft["n"]).max())}
    bt = ln_bwd_tol(ref, z, g, de, dn, ft["mean"], ft["rstd"], ft["inv"])
    nb = -(-rows // 8)
    r["dz"] = rows_within(zz.grad, z64.grad, bt["dz"])[1]
    for nm, got, want, part in (("dgamma", norm.weight.grad, g64.grad, ref["dg"]), ("dbeta", norm.bias.grad, b64.grad,
                                                                                   ref["db"])):
        bound = (bt["dg" if nm == "dgamma" else "db"].sum() + (nb * U * part.abs().sum(0)).norm()) * (1 + 1e-3)
        r[nm] = float((got.double() - want).norm() / bound)
    above = ~ref["below"]
    unit = (n.double()[above].norm(dim=1) - 1).abs() / (((D / 32 + 5) / 2 + 3) * U)
    r["unit norm"] = float(unit.max())
    print(f"[worst error/bound] ln_l2norm wiring rows={rows} D={D}: " + " ".join(f"{k} {v:.3g}" for k, v in r.items()))
    assert max(r.values()) <= 1.0, r
    assert prologue.ln_l2norm(z, norm)[1] is not None


@pytest.mark.gpu
def test_patched_forwards_fall_back_outside_the_kernel_limits(F, cuda_device):
    """The instance patches run the stock modules where the kernels cannot: E % 4 != 0, E > 4096, more than 32 heads
    under active dropout, a LayerNorm without weight or bias (cross-attention norm and projection tail); a bool
    keep-mask reaches the kernel as fp32 and gives the fp32 mask's result."""
    from preference_guided_image_captioning_alignment_b200 import prologue
    dev = cuda_device
    rel = lambda a, b: float((a - b).norm() / b.norm())  # noqa: E731
    for E, H, drop, affine in ((6, 2, 0.0, True), (4100, 4, 0.0, True), (64 * 33, 33, 0.1, True), (64, 4, 0.0, False)):
        torch.manual_seed(E)
        mha = torch.nn.MultiheadAttention(E, H, dropout=drop, batch_first=True).to(dev)
        norm = torch.nn.LayerNorm(E, elementwise_affine=affine).to(dev)
        dec = types.SimpleNamespace(cross_attention=mha, attention_norm=norm)
        text, vis = torch.randn(2, 3, E, device=dev), torch.randn(2, 1, E, device=dev)
        mha.train(drop > 0)
        prologue.fuse_cross_attention(dec)
        attended, _ = dec.cross_attention(query=text, key=vis, value=vis)
        out = dec.attention_norm(text + attended)
        prologue.unfuse_cross_attention(dec)
        if drop == 0:
            assert rel(out, norm(text + mha(text, vis, vis)[0])) < 1e-5, (E, H)
        else:
            assert out.shape == text.shape and bool(torch.isfinite(out).all())
    for bias in (False, True):
        norm = torch.nn.LayerNorm(64, bias=bias, elementwise_affine=bias).to(dev)
        enc = types.SimpleNamespace(projection=torch.nn.Sequential(torch.nn.Linear(64, 64), norm).to(dev))
        x = torch.randn(5, 64, device=dev)
        ref = enc.projection(x)
        prologue.fuse_projection_tail(enc)
        assert rel(enc.projection(x), ref) < 1e-5
        prologue.unfuse_projection_tail(enc)
    # a bool keep-mask: the values of the fp32 mask
    mha = torch.nn.MultiheadAttention(64, 4, dropout=0.5, batch_first=True).to(dev).train()
    norm = torch.nn.LayerNorm(64).to(dev)
    text, vis = torch.randn(2, 3, 64, device=dev), torch.randn(2, 1, 64, device=dev)
    keep = torch.rand(2, 3, 4, device=dev) >= 0.5
    a = prologue.collapsed_cross_attention_ln(text, vis, mha, norm, keep_weights=keep)
    b = prologue.collapsed_cross_attention_ln(text, vis, mha, norm, keep_weights=keep.float())
    assert torch.equal(a, b)
