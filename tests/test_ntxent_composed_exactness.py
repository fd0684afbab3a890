"""Element-level exactness of the NT-Xent paths that run outside the one-CTA kernel: several launches composed in Python.

* fp32 embeddings beyond 128 rows (`ops.ntxent` / `ops.ntxent_bwd`, reached through `losses.ContrastiveLoss`): the
  forward runs on the two-term bf16 split [hi|lo|hi] . [hi|hi|lo] (`split3`), the backward returns
  g3[:, :D] + g3[:, 2D:] of two softmax-gradient launches, i.e. bf16(G) (b_hi + b_lo) and bf16(G)^T (a_hi + a_lo).
* the components flavour (`components.ContrastiveLoss` -> `ops.ntxent_cosine`): `rownorm_fwd(split=True)`, the bounded
  forward on the split, two backward launches and `rownorm_bwd` with g_second = 2 D, which adds the hi and lo blocks.
* global negatives (`distributed._GlobalNTXent` with `CudaCompute`), W ranks emulated on one device through the
  `CudaCompute` methods, composed as `_GlobalNTXent` composes them (the collectives are covered by the gloo test).

The lo half of the split is at most 2^-9 of an element, so a global 1e-2 norm cannot tell whether the split path delivers
the accuracy it exists for.  The checks here:

1. Exact inputs (`gadget`): row i of a owns the coordinates (2i, 2i + 1) with a = (1 + 2^-8, -1), row pi(i) of b has
   (257, 257) there.  The split gives a_hi = (1, -1), a_lo = (2^-8, 0), b_hi = (256, 256), b_lo = (1, 1), so the split
   logit a_hi.b_hi + a_lo.b_hi + a_hi.b_lo = 0 + 1 + 0 is exactly [j == pi(i)]: it exists only through the lo parts
   (the fp64 product of the fp32 values is 1 + 2^-8, the a_lo.b_lo term the split drops by definition).  With
   inv_tau = fp32(0.6931472) the kernels' log2 scale is 1; n = 2^m - 1 rows make every log2-sum-exp m.  Each element
   of dA and dB is one product of a bf16(G) entry and one operand entry, so the whole step is exact and must equal
   `gadget_closed_form` (the kernels' fp32 roundings of G, the lse and the loss reduction emulated) bit for bit.
2. Realistic inputs against fp64 at every element (`SplitCheck`): lse_row, lse_col and the loss against fp64 of the
   fp32 values with `split_dz` as the logit error; dA and dB per row against the contract bf16(G) (b_hi + b_lo),
   bf16(G)^T (a_hi + a_lo) (bf16 rounding of G kept, flips bounded as in `row_bound`), then with a looser bound
   against the true fp64 gradient.  Against the true gradient, bf16(G) noise and a dropped lo block are the same size;
   against the contract the dropped block stands out.  `rownorm_fwd` (split outputs bit-exact given the kernel's own
   inv_norm) and `rownorm_bwd` (per row against fp64) separately; the cosine flavour end to end; the global-negatives
   composition and `lse_combine` per element.
3. Planted faults (`SPLIT_FAULTS`, `ROWNORM_FAULTS`, `GLOBAL_FAULTS`, `COMBINE_FAULTS`) are applied to the reference and
   must be rejected; the ratio by which each is seen is printed.  A fault whose effect is below what the fp32 bound
   resolves in one case (a dropped lo block where G itself is below the fp32 resolution of the exponentials, at a small
   tau) is reported there, and each fault must be rejected in some case of every test.

`CudaCompute.to_operand` rounds fp32 inputs to bf16 (unlike the single-GPU fp32 path): the global checks bound the
kernels against fp64 of the bf16-rounded values, which is that path's contract.

The helpers are plain torch; the tests not marked `gpu` check the builders and the checkers against fp32 emulations.
"""
import math

import numpy as np
import pytest
import torch

from test_kernel_exactness import (LN2, TILE, Reference, bf16_flips, card, dot_err, report, row_bound, rows_within,
                                   ulps)
from test_ntxent_small_exactness import (EXACT_INV_TAU, FAMILIES, KLN2, OUTS, TAUS, exact_mismatch, family,
                                         fp64_model, permutation, split3_torch, split_dz, ulp_diff)

F32 = np.float32
EPS = 1e-12                                   # F.normalize / components.ContrastiveLoss
GADGET_CASES = [(255, 512), (511, 1024)]      # n = 2^m - 1 rows, both above the 128-row dispatch
SPLIT_FAULTS = ("lo_dropped_da", "db_wrong_block", "forward_bf16")
ROWNORM_FAULTS = ("g_second_ignored", "xhat_from_bf16", "projection_below_eps")
GLOBAL_FAULTS = ("combine_rank_missing", "owned_cols_shifted", "db_partial_dropped")
COMBINE_FAULTS = ("combine_rank_missing",)


def parts(x):
    """(hi, lo) of the two-term bf16 split as fp32 tensors: hi = bf16(x), lo = bf16(x - hi)."""
    l3, _ = split3_torch(x)
    d = x.shape[1]
    return l3[:, :d].float(), l3[:, d:2 * d].float()


# ================================================================================================ 1. exact inputs
def gadget(n, D, seed):
    """fp32 (a, b, pi) whose split logits are exactly [j == pi(i)] (see the module docstring); pi a derangement with
    pi != pi^-1, so the positive (i, i) has logit 0 and G is not symmetric."""
    assert 2 * n <= D
    gen = torch.Generator().manual_seed(seed)
    pi = permutation(n, "random", gen)
    a, b = torch.zeros(n, D), torch.zeros(n, D)
    r = torch.arange(n)
    a[r, 2 * r] = 1.0 + 2.0 ** -8
    a[r, 2 * r + 1] = -1.0
    b[pi, 2 * r] = 257.0
    b[pi, 2 * r + 1] = 257.0
    return a, b, pi


def split_logits(a, b):
    """a_hi.b_hi + a_lo.b_hi + a_hi.b_lo in fp64: the product the split kernels compute (a_lo.b_lo dropped)."""
    ha, la = (t.double() for t in parts(a))
    hb, lb = (t.double() for t in parts(b))
    return ha @ hb.T + la @ hb.T + ha @ lb.T


def loss_kernel_sum(lr, lc, diag, inv_denom):
    """ntxent_loss_kernel in fp32: 1024 threads, thread t sums i = t, t + 1024, ... of (lr - d) + (lc - d); a butterfly
    warp_sum, then one over the 32 warp sums; loss = (0.5 v) inv_denom."""
    lr, lc, diag = (np.asarray(v, F32) for v in (lr, lc, diag))
    acc = np.zeros(1024, F32)
    for i in range(lr.size):
        acc[i % 1024] = F32(acc[i % 1024] + F32(F32(lr[i] - diag[i]) + F32(lc[i] - diag[i])))

    def butterfly(v):                                   # v: (..., 32)
        lane = np.arange(32)
        for o in (16, 8, 4, 2, 1):
            v = (v + v[..., lane ^ o]).astype(F32)
        return v[..., 0]

    total = butterfly(butterfly(acc.reshape(32, 32)))
    return F32(F32(F32(0.5) * total) * F32(inv_denom))


def gadget_closed_form(a, b, pi, mean, fault=None):
    """The outputs of the unbounded fp32 path on a gadget, from its structure: every log2-sum-exp m = log2(n + 1);
    lse = fp32(m fp32(ln 2)); diag = 0; loss from `loss_kernel_sum`; coef = fp32(fp32(mult) inv_tau) as
    ntxent_bwd_impl forms it; G in fp32 in g_chunk's order (coef 2^(z - m) + coef 2^(z - m), then - coef for the column
    one-hot and - coef for the row one-hot), rounded to bf16; dA = bf16(G) (b_hi + b_lo), dB = bf16(G)^T (a_hi + a_lo),
    exact.  fault: one of SPLIT_FAULTS planted.  -> (loss, lse_row, lse_col, da, db)"""
    n = a.shape[0]
    m = int(round(math.log2(n + 1)))
    it = F32(EXACT_INV_TAU)
    if fault == "forward_bf16":       # the forward on bf16(x): a_hi . b_hi = 0, every lse log n
        L = F32(math.log(n))
    else:
        L = F32(F32(m) * KLN2)
    lse = np.full(n, L, F32)
    loss = loss_kernel_sum(lse, lse, np.zeros(n, F32), (1.0 / n) if mean else 1.0)
    coef = torch.tensor(F32(F32((1.0 / (2 * n)) if mean else 0.5) * it))
    z = torch.zeros(n, n)
    z[torch.arange(n), pi] = 1.0
    e = torch.exp2(z - m)
    g = coef * e
    g = g + coef * e
    eye = torch.eye(n, dtype=torch.bool)
    g = torch.where(eye, (g - coef) - coef, g)
    gb = g.bfloat16().double()
    ha, la = (t.double() for t in parts(a))
    hb, lb = (t.double() for t in parts(b))
    da = gb @ (hb if fault == "lo_dropped_da" else hb + lb)
    db = gb.T @ (2 * ha if fault == "db_wrong_block" else ha + la)
    return (torch.tensor(float(loss)), torch.from_numpy(lse.copy()), torch.from_numpy(lse.copy()), da.float(),
            db.float())


# ================================================================================================ 2. bounded checks
def family32(name, n, D, gen, unit=False):
    """fp32 inputs of one family of the small-kernel tests: its bf16 rows times (1 + u), |u| <= 2^-9 per element, so
    every element has a lo part; equal rows get the same u (the ties of `duplicates` stay ties).  unit: rows
    normalised in fp32 (what `assume_normalized` promises)."""
    out = []
    for x in family(name, n, D, gen):
        _, inv = torch.unique(x.float(), dim=0, return_inverse=True)
        u = (torch.rand(n, D, generator=gen) - 0.5) * 2.0 ** -8
        x = x.float() * (1 + u[inv])
        out.append(torch.nn.functional.normalize(x, dim=-1) if unit else x)
    return out


def exp_eps(inv_tau, tmax, lmax, dz, lse_err):
    """Relative error of one exponential of the backward kernels, P~ = P (1 + d): three ex2.approx (2^-22 each) and
    the fp32 coefficient formed with two roundings (2^-22); the fp32 arguments z c - lse log2 e (or the shared form
    z c - c, c - lse log2 e), each rounded relative to magnitudes <= 2 (tmax + lmax) (2^-21 (tmax + lmax) in natural
    units); the logit error dz (natural units) and the error of the lse the backward is handed (measured)."""
    return 2.0 ** -20 + 2.0 ** -21 * (tmax + lmax) + dz + lse_err


class SplitCheck:
    """Bounds of a split-path result out = (loss, lse_row, lse_col, dA, dB) against fp64 (`fp64_model`).

    x, y: the values whose product the logits approximate (fp32 embeddings, or the unit rows of the cosine flavour);
    (hx, lx), (hy, ly): the split parts the kernels use; dz: bound on the logit error in natural units.
        lse       ulps(lse, 16) + dz + 2^-22 tmax    (c = fp32(inv_tau log2 e) rounded)
        loss      loss_mult (sum of the lse bounds + 2 n dz + 32 2^-24 sum |terms|) + 4 2^-24 |loss|
        dA, dB    row_bound with K = max(n, 128) products and `exp_eps`, against the contract bf16(G) (b_hi + b_lo),
                  plus 2^-23 sum_j |G_ij| ||b_j|| for the fp32 sum of the two column blocks."""

    def __init__(self, out, x, y, hx, lx, hy, ly, inv_tau, mean, dz):
        self.out = tuple(o.double() for o in out)
        self.x, self.y, self.inv_tau, self.mean = x, y, inv_tau, mean
        self.hx, self.lx, self.hy, self.ly = (t.double() for t in (hx, lx, hy, ly))
        self.ref = ref = self.model()
        n = x.shape[0]
        tmax = float(ref["t"].abs().max()) * LN2
        lmax = float(torch.cat([ref["lse_row"], ref["lse_col"]]).abs().max())
        tr = ulps(ref["lse_row"], 16) + dz + 2.0 ** -22 * tmax
        tc = ulps(ref["lse_col"], 16) + dz + 2.0 ** -22 * tmax
        diag = ref["t"].diagonal().abs() * LN2
        mag = (ref["lse_row"].abs() + ref["lse_col"].abs() + 2 * diag).sum()
        self.tol = {"lse_row": tr, "lse_col": tc,
                    "loss": (ref["lm_exact"] * (tr.sum() + tc.sum() + 2 * n * dz + 32 * 2.0 ** -24 * mag)
                             + 4 * 2.0 ** -24 * ref["loss"].abs()).reshape(())}
        lse_err = float(torch.cat([self.out[1] - ref["lse_row"], self.out[2] - ref["lse_col"]]).abs().max())
        self.eps_p = eps_p = exp_eps(inv_tau, tmax, lmax, dz, lse_err)
        e = ref["w"] * (ref["pr"] + ref["pc"])
        self.ga = ga = ref["g"].abs()
        _, flip = bf16_flips(ref["g"], eps_p * e + 2.0 ** -22 * ga)
        An = self.hx.norm(dim=1) + self.lx.norm(dim=1)
        Bn = self.hy.norm(dim=1) + self.ly.norm(dim=1)
        k = max(n, TILE)
        self.tol["da"] = row_bound(ga @ Bn, flip @ Bn, e @ Bn, k, eps_p) + 2.0 ** -23 * (ga @ Bn)
        self.tol["db"] = row_bound(ga.T @ An, flip.T @ An, e.T @ An, k, eps_p) + 2.0 ** -23 * (ga.T @ An)

    def model(self, fault=None):
        if fault == "forward_bf16":
            return fp64_model(self.hx, self.hy, self.inv_tau, self.mean)
        ref = fp64_model(self.x, self.y, self.inv_tau, self.mean, grad_ops=(self.hx + self.lx, self.hy + self.ly))
        if fault == "lo_dropped_da":
            ref["da"] = ref["gb"] @ self.hy
        elif fault == "db_wrong_block":
            ref["db"] = ref["gb"].T @ (2 * self.hx)
        return ref

    def ratios(self, ref, out=None):
        out = self.out if out is None else out
        r = {}
        for nm, o in zip(OUTS, out):
            if nm in ("da", "db"):
                r[nm] = rows_within(o, ref[nm], self.tol[nm])[1]
            else:
                r[nm] = float(((o - ref[nm]).abs() / self.tol[nm]).max())
        return r

    def run(self, what, log=print):
        """Assert every output within its bound; -> {fault: largest error / bound against the faulty reference}."""
        worst = self.ratios(self.ref)
        log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        assert max(worst.values()) <= 1.0, (what, worst)
        return {f: max(self.ratios(self.model(f)).values()) for f in SPLIT_FAULTS}

    def true_gradient(self, what, log=print):
        """dA, dB against the true fp64 gradient of (x, y) (G unrounded, the fp32 values): the contract bound plus the
        two roundings the contract makes, bf16(G) and the split (2^-9 + 2^-17 relative), as 2^-7 sum_j |G_ij| ||y_j||."""
        tm = fp64_model(self.x, self.y, self.inv_tau, self.mean, round_g=False)
        xn, yn = self.x.double().norm(dim=1), self.y.double().norm(dim=1)
        ga = tm["g"].abs()
        worst = {"da": rows_within(self.out[3], tm["da"], self.tol["da"] + 2.0 ** -7 * (ga @ yn))[1],
                 "db": rows_within(self.out[4], tm["db"], self.tol["db"] + 2.0 ** -7 * (ga.T @ xn))[1]}
        log(f"[worst error/bound] {what} true gradient: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        assert max(worst.values()) <= 1.0, (what, worst)
        return tm


class FaultTally:
    """The smallest and largest ratio by which each planted fault is seen over the cases of one test."""

    def __init__(self):
        self.seen = {}

    def add(self, seen):
        for f, v in seen.items():
            lo, hi, cnt, tot = self.seen.get(f, (math.inf, 0.0, 0, 0))
            self.seen[f] = (min(lo, v), max(hi, v), cnt + (v > 1.0), tot + 1)

    def report(self, what, optional=()):
        for f, (lo, hi, cnt, tot) in sorted(self.seen.items()):
            print(f"[fault error/bound] {what} {f}: rejected in {cnt} of {tot} cases, seen by {lo:.3g} .. {hi:.3g}")
            assert cnt > 0 or f in optional, (what, f, "planted fault never rejected")


def split_optional(tau):
    """The split faults a test at this tau need not reject: below tau = 0.5 a pair's softmax is peaked, G cancels to
    (1 - p) of the exponentials it is formed from, and a dropped lo block (2^-9 of G's row) falls below the allowance
    for the logit error (split_dz inv_tau times those exponentials); at tau = 0.03 aligned pairs leave a gradient of
    about e^-26 of those exponentials, below what fp32 resolves for a wrong dB block as well.  The exact gadget tests
    reject both bit for bit."""
    if tau >= 0.5:
        return ()
    return ("lo_dropped_da",) if tau >= 0.07 else ("lo_dropped_da", "db_wrong_block")


def emulate_split(x, y, inv_tau, mean, gen=None):
    """The split path's arithmetic in fp32 torch (CPU): logits from the fp32 product of the split operands times
    fp32(inv_tau log2 e), lse in log2 units with the fp32 sums, loss, G = coef (2^(t - lr) + 2^(t - lc)) - 2 coef I
    rounded to bf16, dA = bf16(G) b_hi + bf16(G) b_lo.  With gen, every exponential carries a relative error up to
    2^-23."""
    n, d = x.shape
    l3, _ = split3_torch(x)
    _, r3 = split3_torch(y)
    it = F32(inv_tau)
    c = float(F32(it * F32(1.4426950408889634)))
    t = (l3.float() @ r3.float().T) * c

    def ex2(v):
        out = torch.exp2(v)
        if gen is not None:
            out = (out.double() * (1 + (torch.rand(v.shape, generator=gen, dtype=torch.float64) - 0.5) * 2.0 ** -22)).float()
        return out

    m = t.amax(1, keepdim=True)
    lr = (m + torch.log2(ex2(t - m).sum(1, keepdim=True))).squeeze(1)
    m = t.amax(0, keepdim=True)
    lc = (m + torch.log2(ex2(t - m).sum(0, keepdim=True))).squeeze(0)
    lse_r, lse_c = lr * float(KLN2), lc * float(KLN2)
    diag = t.diagonal() / c * float(it)
    loss = torch.tensor(float(loss_kernel_sum(lse_r.numpy(), lse_c.numpy(), diag.numpy(), 1.0 / n if mean else 1.0)))
    coef = float(F32(F32((1.0 / (2 * n)) if mean else 0.5) * it))
    g = coef * ex2(t - lr[:, None]) + coef * ex2(t - lc[None, :])
    g = torch.where(torch.eye(n, dtype=torch.bool), (g - coef) - coef, g)      # g_chunk's order
    gb = g.bfloat16().float()
    hx, lx = parts(x)
    hy, ly = parts(y)
    return loss, lse_r, lse_c, gb @ hy + gb @ ly, gb.T @ hx + gb.T @ lx


# ------------------------------------------------------------------------------------------------ row normalisation
def rownorm_inv_tol(x, inv_ref):
    """|inv~ - inv| for inv = 1 / max(||x||, eps): the fp32 sum of squares over D / 32 fmaf per lane and a 5-level
    butterfly ((D / 32 + 5) 2^-24 relative), halved by the square root, then sqrtf and the division rounded."""
    D = x.shape[1]
    return 2.0 ** -24 * ((D / 32 + 5) / 2 + 2) * inv_ref


def rownorm_bwd_reference(x, g, eps=EPS, fault=None):
    """F.normalize's gradient in fp64 (torch semantics: a row with ||x|| < eps gets g / eps, no projection).
    fault: `xhat_from_bf16` projects on bf16(x / ||x||); `projection_below_eps` projects clamped rows as well."""
    x, g = x.double(), g.double()
    nrm = x.norm(dim=1, keepdim=True)
    inv = 1.0 / nrm.clamp_min(eps)
    u = x * inv
    if fault == "xhat_from_bf16":
        u = u.float().bfloat16().double()
    proj = (u * g).sum(1, keepdim=True)
    if fault != "projection_below_eps":
        proj = torch.where(nrm < eps, torch.zeros_like(proj), proj)
    return (g - u * proj) * inv


def rownorm_bwd_tol(x, g, inv_rel):
    """Per-row bound on ||dx~ - dx||: dx = (g - xh <xh, g>) inv with xh = fp32(x inv~).  The dot product (D / 32 fmaf
    per lane, 5 butterfly levels, xh rounded) is off by (D / 32 + 7) 2^-24 ||g|| plus inv_rel ||g||; each element is
    formed with 4 roundings and carries inv_rel twice (in xh and in the factor); the sum of the two column blocks of g
    one rounding: (D / 32 + 16) 2^-24 + 3 inv_rel, relative to inv ||g||."""
    D = x.shape[1]
    inv = 1.0 / x.double().norm(dim=1).clamp_min(EPS)
    return inv * g.double().norm(dim=1) * ((D / 32 + 16) * 2.0 ** -24 + 3 * inv_rel)


def varied_rows(n, D, gen, clamped=0):
    """fp32 rows with norms 10^U(-3, 3); the last `clamped` rows get norm 0 < ||x|| < eps, and one of them 0."""
    x = torch.randn(n, D, generator=gen)
    x = torch.nn.functional.normalize(x, dim=-1) * torch.pow(10.0, torch.rand(n, 1, generator=gen) * 6 - 3)
    if clamped:
        x[n - clamped:] = torch.nn.functional.normalize(x[n - clamped:], dim=-1) * 3e-13
        x[n - 1] = 0.0
    return x


# ------------------------------------------------------------------------------------------------ global negatives
class TorchCompute:
    """fp32 torch stand-in for `CudaCompute` (CPU tests of the global checker): the same operands (bf16), lse in
    fp32, G rounded to bf16."""

    def to_operand(self, x):
        return x.bfloat16()

    def ntxent_fwd(self, a, b_all, inv_tau, off):
        t = (a.float() @ b_all.float().T) * float(F32(inv_tau))
        i = torch.arange(a.shape[0])
        return torch.logsumexp(t, 1), t[i, i + off], torch.logsumexp(t, 0)

    def lse_combine(self, parts_):
        return torch.logsumexp(parts_, 0)

    def ntxent_loss(self, lse_row, diag, lse_col_owned, inv_denom):
        return 0.5 * ((lse_row - diag) + (lse_col_owned - diag)).sum() * float(F32(inv_denom))

    def ntxent_bwd(self, a, b_all, inv_tau, off, lse_row, lse_col, grad_loss, mult):
        it = float(F32(inv_tau))
        t = (a.float() @ b_all.float().T) * it
        coef = float(grad_loss) * float(F32(F32(mult) * F32(inv_tau)))
        g = coef * (torch.exp(t - lse_row[:, None]) + torch.exp(t - lse_col[None, :]))
        i = torch.arange(a.shape[0])
        g[i, i + off] -= 2 * coef
        gb = g.bfloat16().float()
        return gb @ b_all.float(), gb.T @ a.float()


def run_ranks(compute, a, b, world, inv_tau, mean=True):
    """`_GlobalNTXent` forward and backward for `world` ranks on one device: rank r owns rows [r nb, (r + 1) nb) of a
    and b; the all-gathers are concatenations, the all-reduce of the loss and the reduce-scatter of dB are sums."""
    B = a.shape[0]
    nb = B // world
    a_ops = [compute.to_operand(a[r * nb:(r + 1) * nb]) for r in range(world)]
    b_all = torch.cat([compute.to_operand(b[r * nb:(r + 1) * nb]) for r in range(world)])
    fw = [compute.ntxent_fwd(a_ops[r], b_all, inv_tau, r * nb) for r in range(world)]
    parts_ = torch.stack([f[2].reshape(B) for f in fw])
    lse_col = compute.lse_combine(parts_)
    inv_denom = (1.0 / B) if mean else 1.0
    losses = [compute.ntxent_loss(fw[r][0], fw[r][1], lse_col[r * nb:(r + 1) * nb].contiguous(), inv_denom)
              for r in range(world)]
    loss = sum(losses)
    grad = torch.ones((), device=a.device)
    mult = (1.0 / (2.0 * B)) if mean else 0.5
    bw = [compute.ntxent_bwd(a_ops[r], b_all, inv_tau, r * nb, fw[r][0], lse_col, grad, mult) for r in range(world)]
    db = bw[0][1].clone()
    for r in range(1, world):
        db += bw[r][1]
    return dict(a=torch.cat(a_ops), b=b_all, parts=parts_, lse_row=torch.cat([f[0] for f in fw]), lse_col=lse_col,
                loss=loss, losses=losses, da=torch.cat([w[0] for w in bw]), db=db, db_parts=[w[1] for w in bw], nb=nb)


def combine_tol(parts_, ref):
    """|lse_combine~ - lse| per element: the max is exact; each term ex2((p - m) kLog2e) with the difference and the
    product rounded (2^-23 |p - m| in log2 units, weighted by the term's share) and ex2.approx (2^-22); the serial
    fp32 sum (W 2^-24); log2f (2^-21 for a result below 32) and m + log2f(s) kLn2 rounded twice (2^-23 |lse|)."""
    p = parts_.double()
    m = p.amax(0)
    share = torch.exp(p - ref[None, :])
    return (2.0 ** -22 + p.shape[0] * 2.0 ** -24 + 2.0 ** -23 * (share * (p - m).abs()).sum(0) + 2.0 ** -21
            + 2.0 ** -23 * ref.abs())


def check_global(res, inv_tau, world, what, mean=True, log=print):
    """The composed global step against fp64 of the bf16 operands, element by element: lse_col (after the merge) per
    column, lse_row per row, the summed loss, dA per rank per row and dB per row after the partials are summed
    (`Reference`: G of the fp64 statistics, bf16 rounding kept).  -> {fault: ratio it is seen by}"""
    a, b = res["a"], res["b"]
    B, D = a.shape
    nb = res["nb"]
    an, bn = a.double().norm(dim=1), b.double().norm(dim=1)
    dz = dot_err(D, float(F32(inv_tau)), float(an.max()), float(bn.max()))
    it = float(F32(inv_tau))
    lr = torch.empty(B, dtype=torch.float64, device=a.device)
    lc_parts = []
    for r0 in range(0, B, 4096):
        z = it * (a[r0:r0 + 4096].double() @ b.double().T)
        lr[r0:r0 + 4096] = torch.logsumexp(z, 1)
        lc_parts.append(torch.logsumexp(z, 0))
        del z
    lc = torch.logsumexp(torch.stack(lc_parts), 0)
    diag = it * (a.double() * b.double()).sum(1)
    tmax = it * float(an.max() * bn.max())
    worst, tol = {}, {}
    for nm, got, ref in (("lse_row", res["lse_row"], lr), ("lse_col", res["lse_col"], lc)):
        tol[nm] = ulps(ref, 16) + dz + 2.0 ** -22 * tmax + (combine_tol(res["parts"], ref) if nm == "lse_col" else 0)
        worst[nm] = float(((got.double() - ref).abs() / tol[nm]).max())
    lm = (0.5 / B) if mean else 0.5
    loss_ref = lm * ((lr - diag) + (lc - diag)).sum()
    mag = (lr.abs() + lc.abs() + 2 * diag.abs()).sum()
    ltol = lm * (tol["lse_row"].sum() + tol["lse_col"].sum() + 2 * B * dz + 32 * 2.0 ** -24 * mag) \
        + (4 + world) * 2.0 ** -24 * loss_ref.abs()
    worst["loss"] = float((res["loss"].double() - loss_ref).abs() / ltol)
    # each rank's term before the all-reduce
    terms = lm * ((lr - diag) + (lc - diag))
    tterm = lm * (tol["lse_row"] + tol["lse_col"] + 2 * dz + 32 * 2.0 ** -24 * (lr.abs() + lc.abs() + 2 * diag.abs()))

    def rank_ratio(r, ref_terms):
        sl = slice(r * nb, (r + 1) * nb)
        ref_r = ref_terms[sl].sum()
        return float((res["losses"][r].double() - ref_r).abs() / (tterm[sl].sum() + 4 * 2.0 ** -24 * ref_r.abs()))

    worst["loss per rank"] = max(rank_ratio(r, terms) for r in range(world))
    lse_err = float(torch.cat([res["lse_row"].double() - lr, res["lse_col"].double() - lc]).abs().max())
    lmax = float(torch.cat([lr, lc]).abs().max())
    eps_p = exp_eps(inv_tau, tmax, lmax, dz, lse_err)
    coef = float(F32(F32((1.0 / (2 * B)) if mean else 0.5) * F32(inv_tau)))
    idx = torch.arange(B, device=a.device)
    row = (lr, torch.full((B,), coef, dtype=torch.float64, device=a.device), idx.int())
    col = (lc, row[1], idx.int())
    ref = Reference(a, b, it, row, col, eps_p)
    tda, tdb = ref.bounds
    worst["da"] = rows_within(res["da"], ref.out_x, tda)[1]
    worst["db"] = rows_within(res["db"], ref.out_y, tdb)[1]
    log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert max(worst.values()) <= 1.0, (what, worst)
    # planted faults, each on the rank whose change is largest
    seen = {}
    p = res["parts"].double()
    drop = max(range(world), key=lambda r: float(torch.exp(p[r] - lc).max()))
    keep = [r for r in range(world) if r != drop]
    missing = torch.logsumexp(p[keep], 0)
    seen["combine_rank_missing"] = float(((res["lse_col"].double() - missing).abs() / tol["lse_col"]).max())
    shifted = lm * ((lr - diag) + (torch.roll(lc, -nb) - diag))    # a rank sums the columns of the next rank
    seen["owned_cols_shifted"] = max(rank_ratio(r, shifted) for r in range(world))
    seen["db_partial_dropped"] = max(rows_within(res["db"], ref.out_y - res["db_parts"][r].double(), tdb)[1]
                                     for r in range(world))
    return seen


# ================================================================================================ CPU tests
@pytest.mark.parametrize("n,D", GADGET_CASES + [(7, 16), (31, 64)])
def test_gadget_logits(n, D):
    """The gadget's split logits are exactly the permutation matrix, in fp64 and in an fp32 product of the split
    operands; the fp64 product of the fp32 values is 1 + 2^-8 there (the a_lo.b_lo term the split drops); the 1
    needs the lo parts (a_hi . b_hi == 0); pi has no fixed point and pi != pi^-1."""
    a, b, pi = gadget(n, D, n + D)
    P = torch.zeros(n, n, dtype=torch.float64)
    P[torch.arange(n), pi] = 1.0
    assert torch.equal(split_logits(a, b), P)
    l3, _ = split3_torch(a)
    _, r3 = split3_torch(b)
    assert torch.equal((l3.float() @ r3.float().T).double(), P)
    assert torch.equal(a.double() @ b.double().T, P * (1 + 2.0 ** -8))
    ha, la = parts(a)
    hb, lb = parts(b)
    assert float((ha @ hb.T).abs().max()) == 0.0 and float(la.abs().max()) == 2.0 ** -8 and float(lb.abs().max()) == 1
    r = torch.arange(n)
    assert bool((pi != r).all()) and not torch.equal(pi[pi], r)
    assert 2 ** int(round(math.log2(n + 1))) == n + 1


def test_exact_inv_tau_through_the_module():
    """losses.ContrastiveLoss(temperature = 1 / inv_tau) hands the kernels exactly fp32(0.6931472)."""
    assert F32(1.0 / float(1.0 / float(EXACT_INV_TAU))) == EXACT_INV_TAU


@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("n,D", [(7, 16), (31, 64), (255, 512)])
def test_gadget_closed_form_equals_emulation(n, D, mean):
    """The closed form equals an fp32 emulation of the split path (exact exponentials), and each planted fault changes
    some output bit-exactly."""
    a, b, pi = gadget(n, D, n + D)
    ref = gadget_closed_form(a, b, pi, mean)
    emu = emulate_split(a, b, float(EXACT_INV_TAU), mean)
    assert exact_mismatch(emu, ref) == [], {nm: ulp_diff(o, r) for nm, o, r in zip(OUTS, emu, ref)}
    for f in SPLIT_FAULTS:
        assert exact_mismatch(ref, gadget_closed_form(a, b, pi, mean, f)) != [], f


@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_split_check_accepts_emulation_and_rejects_faults(fam, tau):
    """SplitCheck (contract and true gradient) accepts an fp32 emulation of the split path with approximate
    exponentials, and rejects each planted fault in some case."""
    inv_tau = float(F32(1.0 / tau))
    tally = FaultTally()
    for n, D, mean in ((129, 128, True), (200, 256, False)):
        gen = torch.Generator().manual_seed(n + D + int(100 * tau))
        x, y = family32(fam, n, D, gen)
        l3, _ = split3_torch(x)
        _, r3 = split3_torch(y)
        out = emulate_split(x, y, inv_tau, mean, gen=gen)
        chk = SplitCheck(out, x, y, *parts(x), *parts(y), inv_tau, mean, inv_tau * split_dz(x, y, l3, r3))
        tally.add(chk.run("emulation", log=lambda *s: None))
        chk.true_gradient("emulation", log=lambda *s: None)
    tally.report(f"emulation {fam} tau={tau}", split_optional(tau))


def test_rownorm_checks_accept_emulation_and_reject_faults():
    """The rownorm_bwd bound accepts an fp32 emulation of the kernel (with the clamped rows done right) and rejects
    each planted fault."""
    gen = torch.Generator().manual_seed(5)
    n, D = 64, 512
    x = varied_rows(n, D, gen, clamped=3)
    g0, g1 = torch.randn(n, D, generator=gen), torch.randn(n, D, generator=gen) * 2.0 ** -9
    inv = 1.0 / torch.clamp_min(x.norm(dim=1), EPS)
    ge = g0 + g1
    xh = x * inv[:, None]
    dot = (xh * ge).sum(1)
    dot = torch.where(x.double().norm(dim=1) < EPS, torch.zeros_like(dot), dot)
    dx = (ge - xh * dot[:, None]) * inv[:, None]
    tol = rownorm_bwd_tol(x, ge, 2.0 ** -21)
    ref = rownorm_bwd_reference(x, g0.double() + g1.double())
    assert rows_within(dx, ref, tol)[0]
    for f in ROWNORM_FAULTS:
        bad = rownorm_bwd_reference(x, g0.double() if f == "g_second_ignored" else g0.double() + g1.double(),
                                    fault=None if f == "g_second_ignored" else f)
        assert not rows_within(dx, bad, tol)[0], f


def test_global_check_accepts_emulation_and_rejects_faults():
    """check_global accepts the rank composition run on the fp32 torch stand-in (W = 3 x 100) and rejects each planted
    fault."""
    x, y = rank_pairs(3, 100, 128, 3)
    for inv_tau in (2.0, float(F32(1 / 0.07))):
        res = run_ranks(TorchCompute(), x, y, 3, inv_tau)
        seen = check_global(res, inv_tau, 3, "emulation", log=lambda *s: None)
        assert min(seen.values()) > 1.0, seen


def test_lse_combine_check_rejects_missing_partial():
    """combine_tol accepts an fp32 merge and rejects a partial dropped, with partials 100+ nats apart."""
    gen = torch.Generator().manual_seed(9)
    p = combine_inputs(8, 1000, gen)
    ref = torch.logsumexp(p.double(), 0)
    got = torch.logsumexp(p, 0)
    tol = combine_tol(p, ref)
    assert bool(((got.double() - ref).abs() <= tol).all())
    miss = torch.logsumexp(p.double()[1:], 0)
    assert bool(((got.double() - miss).abs() > tol).any())


def combine_inputs(world, n, gen):
    """fp32 column partials (world, n): ordinary spreads, columns whose partials differ by more than 100 nats, and
    columns where rank 0 dominates."""
    p = torch.randn(world, n, generator=gen) * 3 + 8
    p[:, : n // 4] += torch.linspace(0, 140, world)[:, None]           # > 100 nats apart
    p[0, n // 4: n // 2] += 30.0                                        # rank 0 dominates
    p[:, n // 2: n // 2 + 8] = 5.0                                      # ties
    return p


def test_l2_normalize_bwd_matches_torch_below_eps():
    """oracle.closed_form: l2_normalize_bwd and ntxent(normalize=True) equal torch autograd of F.normalize in fp64 for
    rows with 0 < ||x|| < eps (g / eps, no projection), ||x|| = 0, ||x|| just above eps and ordinary rows."""
    from oracle import closed_form as cf
    x = below_eps_rows(np.random.default_rng(1), 16)
    g = np.random.default_rng(2).standard_normal(x.shape)
    xt = torch.tensor(x, requires_grad=True)
    torch.nn.functional.normalize(xt, dim=-1, eps=EPS).backward(torch.tensor(g))
    np.testing.assert_allclose(cf.l2_normalize_bwd(x, g), xt.grad.numpy(), rtol=1e-12, atol=0)
    # the issue's example row: (3e-13, 4e-13, 0), g = (1, 2, 3) -> g / eps
    np.testing.assert_allclose(cf.l2_normalize_bwd(np.array([[3e-13, 4e-13, 0.0]]), np.array([[1.0, 2.0, 3.0]])),
                               [[1e12, 2e12, 3e12]], rtol=1e-12)
    y = rng_rows(np.random.default_rng(3), 16, 8)
    x = below_eps_rows(np.random.default_rng(1), 16, along=y)
    xt, yt = torch.tensor(x, requires_grad=True), torch.tensor(y, requires_grad=True)
    loss = torch_cosine_ntxent(xt, yt, 0.5, "mean")
    loss.backward()
    o = cf.ntxent(x, y, 0.5, normalize=True, clamp_tau=True)
    assert o["loss"] == pytest.approx(float(loss.detach()), rel=1e-12)
    np.testing.assert_allclose(o["dx"], xt.grad.numpy(), rtol=1e-10, atol=0)
    np.testing.assert_allclose(o["dy"], yt.grad.numpy(), rtol=1e-10, atol=0)


def below_eps_rows(rng, n, D=8, along=None):
    """Rows of norm 3e-13, 7e-13, 0 (below eps), 1.01e-12 and 2e-12 (just above eps), then ordinary rows.  along: take
    the directions of those rows (plus a little noise) from it, so that the upstream gradient has a large radial part
    and the projection a clamped row must not get would change it by O(1)."""
    x = rng.standard_normal((n, D))
    if along is not None:
        x = np.asarray(along, np.float64) + 0.3 * x / math.sqrt(D)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    for i, s in enumerate((3e-13, 7e-13, 0.0, 1.01e-12, 2e-12)):
        x[i] *= s
    return x


def rng_rows(rng, n, D):
    y = rng.standard_normal((n, D))
    return y / np.linalg.norm(y, axis=1, keepdims=True)


def torch_cosine_ntxent(x, y, tau, reduction):
    """components.ContrastiveLoss in torch (the reference's arithmetic): F.normalize, clamp tau to [0.1, 2], symmetric
    cross-entropy, halved."""
    t = min(max(tau, 0.1), 2.0)
    s = torch.nn.functional.normalize(x, dim=-1) @ torch.nn.functional.normalize(y, dim=-1).T / t
    lab = torch.arange(x.shape[0], device=x.device)
    ce = torch.nn.functional.cross_entropy
    return 0.5 * (ce(s, lab, reduction=reduction) + ce(s.T, lab, reduction=reduction))


# ================================================================================================ GPU tests
@pytest.fixture(scope="module")
def pg(cuda_device):
    import preference_guided_image_captioning_alignment_b200 as pkg
    from preference_guided_image_captioning_alignment_b200 import _lib
    lib = _lib.load()
    assert lib.pgica_device_check() == 0, lib.pgica_last_error()
    return pkg


# ------------------------------------------------------------------------------------------------ 1. exact
@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("n,D", GADGET_CASES)
def test_split_path_exact_gadget(pg, cuda_device, n, D, mean):
    """The unbounded fp32 path (`ops.ntxent` with autograd, and `losses.ContrastiveLoss` for the mean) on the gadget:
    loss, lse_row, lse_col, dA and dB equal the closed form bit for bit; each planted fault is rejected."""
    from preference_guided_image_captioning_alignment_b200 import losses, ops
    a0, b0, pi = gadget(n, D, n + D)
    ref = gadget_closed_form(a0, b0, pi, mean)
    a, b = a0.to(cuda_device).requires_grad_(True), b0.to(cuda_device).requires_grad_(True)
    loss, lse_row, lse_col = ops.ntxent(a, b, float(EXACT_INV_TAU), mean)
    loss.backward()
    out = (loss.detach(), lse_row, lse_col, a.grad, b.grad)
    bad = exact_mismatch(out, ref)
    assert bad == [], (n, D, mean, {nm: ulp_diff(o, r) for nm, o, r in zip(OUTS, out, ref) if nm in bad})
    for f in SPLIT_FAULTS:
        assert exact_mismatch(out, gadget_closed_form(a0, b0, pi, mean, f)) != [], (f, "planted fault not rejected")
    if mean:
        a2, b2 = a0.to(cuda_device).requires_grad_(True), b0.to(cuda_device).requires_grad_(True)
        mod = losses.ContrastiveLoss(temperature=1.0 / float(EXACT_INV_TAU))
        l2 = mod(a2, b2)
        l2.backward()
        assert exact_mismatch((l2.detach(), lse_row, lse_col, a2.grad, b2.grad), ref) == []
    print(f"[exact] split gadget n={n} D={D} mean={mean}: bit-exact, {len(SPLIT_FAULTS)} faults rejected ({card()})")


# ------------------------------------------------------------------------------------------------ 2. fp32 trainer
@pytest.mark.gpu
@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_split_path_bounded_fp64(pg, cuda_device, fam, tau):
    """fp32 embeddings, B in {129, 300, 1024, 4096}, D = 512, assume_normalized off (general rows) and on (rows
    normalised in fp32; the one-pass forward and the shared-exponential backward), through `ops.ntxent` with
    autograd (mean and sum; `losses.ContrastiveLoss` once per B): every output against fp64 of the fp32 values, the
    gradients against the contract and the true gradient."""
    from preference_guided_image_captioning_alignment_b200 import losses, ops
    inv_tau = float(F32(1.0 / tau))
    D = 512
    worst, tally = 0.0, FaultTally()
    for B in (129, 300, 1024, 4096):
        for unit in (False, True):
            gen = torch.Generator().manual_seed(B + 7 * unit + int(100 * tau))
            x, y = (t.to(cuda_device) for t in family32(fam, B, D, gen, unit=unit))
            l3, _ = split3_torch(x)
            _, r3 = split3_torch(y)
            dz = inv_tau * split_dz(x, y, l3, r3)
            for mean in (True, False):
                a, b = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
                loss, lse_row, lse_col = ops.ntxent(a, b, inv_tau, mean, unit)
                loss.backward()
                out = (loss.detach(), lse_row, lse_col, a.grad, b.grad)
                what = f"split {fam} tau={tau} B={B} unit={unit} mean={mean}"
                chk = SplitCheck(out, x, y, *parts(x), *parts(y), inv_tau, mean, dz)
                tally.add(chk.run(what))
                chk.true_gradient(what)
                worst = max(worst, max(chk.ratios(chk.ref).values()))
                if mean:                  # the module's call: within the same bounds (dA is add-reduced)
                    mod = losses.ContrastiveLoss(temperature=1.0 / inv_tau)
                    mod.assume_normalized = unit
                    a2, b2 = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
                    l2 = mod(a2, b2)
                    l2.backward()
                    r2 = chk.ratios(chk.ref, (l2.detach().double(), chk.out[1], chk.out[2], a2.grad.double(),
                                              b2.grad.double()))
                    assert max(r2.values()) <= 1.0, (what, "ContrastiveLoss", r2)
                del chk
    report(f"split {fam} tau={tau} all cases", worst)
    tally.report(f"split {fam} tau={tau}", split_optional(tau))


# ------------------------------------------------------------------------------------------------ 2. cosine flavour
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_rownorm_fwd_split_bit_exact(pg, cuda_device, dtype):
    """rownorm_fwd(split=True): y, [hi|lo|hi], [hi|hi|lo] bit for bit from v = fp32(x inv) with the kernel's own
    inv_norm; inv_norm within `rownorm_inv_tol` (a few ulps) of fp64 1 / max(||x||, eps); rows of norm 1e-3 .. 1e3,
    clamped rows and a zero row, D = 512 and a D that is not a multiple of 32."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    worst = 0.0
    for n, D in ((64, 512), (300, 512), (1024, 512), (300, 200)):
        x = varied_rows(n, D, torch.Generator().manual_seed(n + D), clamped=3).to(dtype).to(cuda_device)
        y, inv, _, l3, r3 = F.rownorm_fwd(x, EPS, split=True)
        inv_ref = 1.0 / x.double().norm(dim=1).clamp_min(float(F32(EPS)))
        ratio = float(((inv.double() - inv_ref).abs() / rownorm_inv_tol(x, inv_ref)).max())
        worst = max(worst, ratio)
        assert ratio <= 1.0, (n, D, ratio)
        v = x.float() * inv[:, None]
        hi = v.bfloat16()
        lo = (v - hi.float()).bfloat16()
        bits = lambda t: t.view(torch.int16)  # noqa: E731
        assert torch.equal(bits(y), bits(hi))
        assert torch.equal(bits(l3), bits(torch.cat([hi, lo, hi], 1)))
        assert torch.equal(bits(r3), bits(torch.cat([hi, hi, lo], 1)))
        assert bool((lo != 0).any()) or dtype == torch.bfloat16
    report(f"rownorm_fwd inv_norm {dtype}", worst)


@pytest.mark.gpu
def test_rownorm_bwd_fp64(pg, cuda_device):
    """rownorm_bwd per row against fp64 given the same g, for fp32 / bf16 x and g, a pitch larger than D, g_second
    >= 0 (the split layout [g_hi | . | g_lo] and an arbitrary offset) and < 0; clamped rows included.  Each planted
    fault is rejected."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    n, D = 300, 512
    worst, tally = 0.0, FaultTally()
    for xdt in (torch.float32, torch.bfloat16):
        for gdt in (torch.float32, torch.bfloat16):
            for pitch, second in ((D, -1), (3 * D, 2 * D), (3 * D, -1), (2 * D + 40, D + 17)):
                gen = torch.Generator().manual_seed(pitch + second + 3 * (xdt == torch.bfloat16) + (gdt == torch.bfloat16))
                x = varied_rows(n, D, gen, clamped=3).to(xdt).to(cuda_device)
                g = (torch.randn(n, pitch, generator=gen) * torch.pow(10.0, torch.rand(n, 1, generator=gen) * 4 - 2))
                g = g.to(gdt).to(cuda_device)
                _, inv, _ = F.rownorm_fwd(x, EPS)
                dx = F.rownorm_bwd(x, inv, g, second=second)
                g0 = g[:, :D].double()
                ge = g0 + (g[:, second:second + D].double() if second >= 0 else 0)
                inv_ref = 1.0 / x.double().norm(dim=1).clamp_min(float(F32(EPS)))
                inv_rel = float(((inv.double() - inv_ref).abs() / inv_ref).max())
                tol = rownorm_bwd_tol(x, ge, inv_rel)
                ok, r = rows_within(dx, rownorm_bwd_reference(x, ge, float(F32(EPS))), tol)
                worst = max(worst, r)
                assert ok, (xdt, gdt, pitch, second, r)
                seen = {f: rows_within(dx, rownorm_bwd_reference(x, ge, float(F32(EPS)), fault=f), tol)[1]
                        for f in ROWNORM_FAULTS if f != "g_second_ignored"}
                if second >= 0:
                    seen["g_second_ignored"] = rows_within(dx, rownorm_bwd_reference(x, g0, float(F32(EPS))), tol)[1]
                tally.add(seen)
    report("rownorm_bwd all layouts", worst)
    tally.report("rownorm_bwd")


@pytest.mark.gpu
@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("tau", [0.5, 0.07])
def test_cosine_flavour_fp64(pg, cuda_device, tau, reduction):
    """components.ContrastiveLoss (tau 0.07 clamps to 0.1) at B in {64, 300, 1024} on rows of norm 1e-3 .. 1e3, fp32
    and bf16 inputs: lse and the loss against fp64 of F.normalize + NT-Xent; dx, dy per row against the contract
    (rownorm backward in fp64 of bf16(G) (y^_hi + y^_lo), the split of the kernel's own unit rows) and against the
    true fp64 gradient.  The planted faults of the split and of rownorm_bwd are rejected."""
    from preference_guided_image_captioning_alignment_b200 import components, functional as F, ops
    D = 512
    tau_eff = min(max(tau, 0.1), 2.0)
    inv_tau = float(F32(1.0 / tau_eff))
    mean = reduction == "mean"
    worst, tally = 0.0, FaultTally()
    for B in (64, 300, 1024):
        for dtype in (torch.float32, torch.bfloat16):
            gen = torch.Generator().manual_seed(B + int(100 * tau) + mean)
            u, v = family32("aligned", B, D, gen)
            scale = lambda: torch.pow(10.0, torch.rand(B, 1, generator=gen) * 6 - 3)  # noqa: E731
            x, y = (u * scale()).to(dtype).to(cuda_device), (v * scale()).to(dtype).to(cuda_device)
            with torch.no_grad():
                out = ops.ntxent_cosine(x, y, inv_tau, mean, EPS)
            mod = components.ContrastiveLoss(temperature=tau, reduction=reduction)
            a, b = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
            loss = mod(a, b)
            loss.backward()
            _, inv_x, _, xl, _ = F.rownorm_fwd(x, EPS, split=True)
            _, inv_y, _, _, yr = F.rownorm_fwd(y, EPS, split=True)
            hx, lx = xl[:, :D].float(), xl[:, D:2 * D].float()
            hy, ly = yr[:, :D].float(), yr[:, 2 * D:].float()
            xu = torch.nn.functional.normalize(x.double(), dim=-1)
            yu = torch.nn.functional.normalize(y.double(), dim=-1)
            inv_rel = max(float(((i.double() * t.double().norm(dim=1) - 1).abs()).max()) for i, t in
                          ((inv_x, x), (inv_y, y)))
            # logit error: the split of fp32(x inv~) against x / ||x||: split_dz plus 2 (inv_rel + 2^-24)
            dz = inv_tau * (split_dz(xu, yu, xl, yr) + 2 * (inv_rel + 2.0 ** -24))
            what = f"cosine tau={tau} {reduction} B={B} {dtype}"
            chk = SplitCheck((loss.detach(), out[1], out[2], a.grad, b.grad), xu, yu, hx, lx, hy, ly, inv_tau, mean,
                             dz)
            ref = chk.ref
            r = {nm: float(((chk.out[i] - ref[nm]).abs() / chk.tol[nm]).max())
                 for i, nm in ((0, "loss"), (1, "lse_row"), (2, "lse_col"))}
            # the gradients: rownorm backward of the contract / of the true gradient w.r.t. the unit rows
            tm = fp64_model(xu, yu, inv_tau, mean, round_g=False)
            ga = tm["g"].abs()
            faults = {}
            for nm, side, t, inv, base_tol, G in (("dx", 3, x, inv_x, chk.tol["da"], ga),
                                                  ("dy", 4, y, inv_y, chk.tol["db"], ga.T)):
                key = "da" if nm == "dx" else "db"
                nrm = 1.0 / t.double().norm(dim=1).clamp_min(EPS)
                other = yu if nm == "dx" else xu
                contract = rownorm_bwd_reference(t, ref[key])
                tol = nrm * base_tol + rownorm_bwd_tol(t, ref[key], inv_rel)
                if dtype == torch.bfloat16:       # the op hands the gradient back in the input's dtype
                    tol = tol + 2.0 ** -8 * contract.norm(dim=1)
                r[nm] = rows_within(chk.out[side], contract, tol)[1]
                true = rownorm_bwd_reference(t, tm[key])
                r[nm + " true"] = rows_within(chk.out[side], true, tol + nrm * 2.0 ** -7 * (G @ other.norm(dim=1)))[1]
                for f in SPLIT_FAULTS:
                    bad = chk.model(f)
                    faults[f] = max(faults.get(f, 0.0), rows_within(chk.out[side], rownorm_bwd_reference(t, bad[key]),
                                                                    tol)[1])
                block0 = ref["gb"] @ hy.double() if nm == "dx" else ref["gb"].T @ hx.double()
                faults["g_second_ignored"] = max(faults.get("g_second_ignored", 0.0),
                                                 rows_within(chk.out[side], rownorm_bwd_reference(t, block0), tol)[1])
                faults["xhat_from_bf16"] = max(faults.get("xhat_from_bf16", 0.0), rows_within(
                    chk.out[side], rownorm_bwd_reference(t, ref[key], fault="xhat_from_bf16"), tol)[1])
            print(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in r.items()))
            assert max(r.values()) <= 1.0, (what, r)
            worst = max(worst, max(r.values()))
            tally.add(faults)
    report(f"cosine tau={tau} {reduction} all cases", worst)
    optional = () if tau_eff >= 0.5 else split_optional(tau_eff) + ("g_second_ignored", "xhat_from_bf16")
    tally.report(f"cosine tau={tau} {reduction}", optional)


# ------------------------------------------------------------------------------------------------ 2. global negatives
@pytest.mark.gpu
@pytest.mark.parametrize("world,nb", [(8, 4096), (3, 300)])
@pytest.mark.parametrize("unit", [False, True])
def test_global_negatives_ranks_fp64(pg, cuda_device, world, nb, unit):
    """_GlobalNTXent's composition through CudaCompute, W ranks on one GPU (the 8-GPU bench shape 8 x 4096 and a
    ragged 3 x 300, D = 512, tau = 0.07 and 0.5), assume_normalized off and on: lse_col after the merge, the summed
    loss, dA per rank per row and dB per row after the partials are summed, against fp64 of the bf16 operands."""
    from preference_guided_image_captioning_alignment_b200.distributed import CudaCompute
    D = 512
    tally = FaultTally()
    for tau in (0.07, 0.5):
        inv_tau = float(F32(1.0 / tau))
        x, y = (t.to(cuda_device) for t in rank_pairs(world, nb, D, world * nb + int(100 * tau)))
        res = run_ranks(CudaCompute(unit), x, y, world, inv_tau)
        tally.add(check_global(res, inv_tau, world, f"global W={world}x{nb} unit={unit} tau={tau}"))
        del res
    tally.report(f"global W={world}x{nb} unit={unit}")


def rank_pairs(world, nb, D, seed):
    """fp32 unit pairs whose alignment differs by rank (noise 0.5 + 0.25 r), so that the ranks' column log-sum-exps
    differ and a rank summing another rank's columns changes its loss term."""
    gen = torch.Generator().manual_seed(seed)
    b = torch.nn.functional.normalize(torch.randn(world * nb, D, generator=gen), dim=-1)
    sigma = (0.5 + 0.25 * torch.arange(world)).repeat_interleave(nb)[:, None]
    a = torch.nn.functional.normalize(b + sigma / math.sqrt(D) * torch.randn(world * nb, D, generator=gen), dim=-1)
    return a, b


@pytest.mark.gpu
def test_global_operand_contract_bf16(pg, cuda_device):
    """CudaCompute.to_operand rounds fp32 rows to bf16: the kernels' loss is that of the bf16-rounded rows (checked
    above); this states the size of that rounding against fp64 of the fp32 rows at tau = 0.07, B = 4096 unit pairs,
    and requires it below 1e-4 relative."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    x, y = (t.to(cuda_device) for t in family32("aligned", 4096, 512, torch.Generator().manual_seed(1), unit=True))
    inv_tau = float(F32(1 / 0.07))
    ref32 = fp64_model(x, y, inv_tau, True)["loss"]
    ref16 = fp64_model(F.as_bf16(x), F.as_bf16(y), inv_tau, True)["loss"]
    rel = float(((ref16 - ref32) / ref32).abs())
    print(f"[bf16 operands] loss relative change {rel:.3g} at tau=0.07, B=4096")
    assert rel < 1e-4


@pytest.mark.gpu
def test_lse_combine_fp64(pg, cuda_device):
    """pgica_lse_combine per element against fp64 within `combine_tol` (a few ulps), W in {1, 2, 3, 8, 15}, partials
    100+ nats apart and one rank dominating; a dropped partial is rejected."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    worst, tally = 0.0, FaultTally()
    for world in (1, 2, 3, 8, 15):
        p = combine_inputs(world, 5000, torch.Generator().manual_seed(world)).to(cuda_device)
        got = F.lse_combine(p)
        ref = torch.logsumexp(p.double(), 0)
        tol = combine_tol(p, ref)
        ok, r = rows_within(got[:, None], ref[:, None], tol)
        worst = max(worst, r)
        assert ok, (world, r)
        if world > 1:
            tally.add({"combine_rank_missing": float(((got.double() - torch.logsumexp(p.double()[1:], 0)).abs()
                                                      / tol).max())})
    report("lse_combine", worst)
    tally.report("lse_combine")


# ------------------------------------------------------------------------------------------------ 4. below eps
@pytest.mark.gpu
def test_normalize_gradient_below_eps(pg, cuda_device):
    """ops.l2_normalize and components.ContrastiveLoss on rows with 0 < ||x|| < eps, ||x|| = 0, ||x|| just above eps and
    ordinary rows, against torch autograd of F.normalize in fp64: a clamped row gets g / eps, no projection."""
    from preference_guided_image_captioning_alignment_b200 import components, ops
    n, D = 16, 512
    y0 = torch.tensor(rng_rows(np.random.default_rng(5), n, D), dtype=torch.float32)
    x0 = torch.tensor(below_eps_rows(np.random.default_rng(4), n, D, along=y0.numpy()), dtype=torch.float32)
    g0 = torch.randn(n, D, generator=torch.Generator().manual_seed(4)).bfloat16()
    x = x0.to(cuda_device).requires_grad_(True)
    yb, _ = ops.l2_normalize(x, EPS)
    yb.backward(g0.to(cuda_device))
    xr = x0.double().requires_grad_(True)
    torch.nn.functional.normalize(xr, dim=-1, eps=float(F32(EPS))).backward(g0.double())
    tol = rownorm_bwd_tol(x0, g0, 2.0 ** -20)
    ok, r = rows_within(x.grad.cpu(), xr.grad, tol)
    report("l2_normalize gradient below / at / above eps", r)
    assert ok, r
    assert not rows_within(x.grad.cpu(), rownorm_bwd_reference(x0, g0, float(F32(EPS)), "projection_below_eps"),
                           tol)[0]
    a, b = x0.to(cuda_device).requires_grad_(True), y0.to(cuda_device).requires_grad_(True)
    components.ContrastiveLoss(temperature=0.5)(a, b).backward()
    ar, br = x0.double().requires_grad_(True), y0.double().requires_grad_(True)
    torch_cosine_ntxent(ar, br, 0.5, "mean").backward()
    # bf16 G and the split: 2^-7 of each row's gradient, times 1 / max(||x||, eps)
    for got, ref in ((a.grad.cpu(), ar.grad), (b.grad.cpu(), br.grad)):
        ok, r = rows_within(got, ref, 2.0 ** -7 * ref.norm(dim=1) + 1e-30)
        report("components.ContrastiveLoss gradient below / at / above eps", r)
        assert ok, r
    # the rows below eps with the projection applied (the old gradient) are outside that bound
    dxhat = ar.grad * ar.detach().norm(dim=1, keepdim=True).clamp_min(float(F32(EPS)))  # exact for clamped rows
    wrong = rownorm_bwd_reference(x0, dxhat, float(F32(EPS)), "projection_below_eps")
    assert not rows_within(a.grad.cpu()[:2], wrong[:2], 2.0 ** -7 * ar.grad[:2].norm(dim=1))[0]
