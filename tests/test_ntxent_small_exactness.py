"""Element-level exactness of the one-launch small-batch NT-Xent (`ntxent_small_kernel`, csrc/ntxent_small.cu).

The kernel serves every NT-Xent step with at most 128 rows per side and D in {128, 256, 384, 512}: the trainer's batch
of 8 fp32 unit vectors (through the two-term bf16 split, similarity depth 3 D) and BASELINE config 1's batch of 64.  One
CTA forms Z = A B^T, both log-sum-exps and the loss, then G = w (softmax_row + softmax_col - 2 I) as a bf16 tile, then
dA = G B and dB = G^T A (the same G tile read MN-major) in 2 D / 128 double-buffered output passes.  A global-norm
comparison does not see a transposed G when G is nearly symmetric, one pass landing in the other buffer's columns, a
padding row counted in a sum at tau = 0.07 or one 32-column chunk of G lost; the checks here look at every element.

1. Exact inputs.  inv_tau = fp32(0.6931472) makes the host's c = fp32(inv_tau * fp32(log2 e)) exactly 1, so the
   kernel's log2-domain logits t equal z.  Integer operands with A B^T = P, a permutation matrix, and n = 2^m - 1
   rows give every row and column the exponent sum 1 + (n - 1) / 2 = 2^(m - 1), so every log2-sum-exp is m exactly.
   G_ij = w 2^(z_ij - m + 1) (minus 2 w on the diagonal, rounded to fp32 as the kernel does, then to bf16) is an
   integer multiple of one power of two, and every partial sum of bf16(G) B and bf16(G)^T A stays below 2^19 of it:
   dA and dB are exact in fp32 in any summation order.  Disjoint supports (z = 0) do the same for n a power of two,
   with every log2-sum-exp log2 n.  The kernel must equal `closed_form` bit for bit.  This rests on ex2.approx.ftz
   returning exact powers of two at the integer arguments -7..0 and on log2f being exact at powers of two.
2. Realistic inputs against fp64 (`fp64_model`), element by element (`Check`): lse_row and lse_col within `lse_tol`,
   the loss within `loss_tol`, dA and dB per row within `row_bound` with a per-element error of the exponentials
   (`exp_err`).  The kernel's G is the exact G of its own logits (one fp32 tile feeds the lse and G), so the logit
   error cancels through the lse by a factor 1 - p: a peaked softmax keeps its small gradient to fp32 resolution,
   and the bounds say so.
3. The fp32 split path: `split3` bit for bit; the forward against fp64 of the fp32 values; the gradients against the
   documented contract bf16(G) B_hi, bf16(G)^T A_hi and, with a looser bound, against the true fp64 gradient.
4. Every comparison is applied to the reference with each planted fault (`FAULTS`) and must reject it.

The helpers are plain torch and run on the CPU; the tests not marked `gpu` check the closed forms against the fp64
model and the checkers against an fp32 emulation of the kernel.
"""
import math

import numpy as np
import pytest
import torch

from test_kernel_exactness import (LN2, LOG2E, TILE, adversarial_pairs, bf16_flips, card, dot_err, report,
                                   row_bound, rows_within, ulps)

KLOG2E = np.float32(1.4426950408889634)   # kLog2e (ptx.cuh)
KLN2 = np.float32(0.6931471805599453)     # kLn2 (ntxent_small.cu)
EXACT_INV_TAU = np.float32(0.6931472)     # fp32(inv_tau * kLog2e) == 1
PERM_ROWS = [1, 3, 7, 15, 31, 63, 127]    # 2^m - 1
ZERO_ROWS = [2, 8, 64, 128]               # powers of two: the trainer, config 1 and the edges
ROWS = [1, 2, 8, 31, 32, 33, 63, 64, 65, 96, 127, 128]
DIMS = [128, 256, 384, 512]
TAUS = [0.5, 0.07, 0.03]
FAMILIES = ["aligned", "adversarial", "duplicates", "peaked", "nonunit"]
OUTS = ("loss", "lse_row", "lse_col", "da", "db")
FAULTS = ("db_untransposed", "g_chunk3_zeroed", "pass_repeated", "padding_counted", "lse_col_ln2", "diag_missing",
          "mean_sum_swapped", "split_lo_in_db")


def host_params(n, inv_tau, mean):
    """(c, w, loss_mult) in fp32, computed in the order ntxent_small_launch computes them."""
    it = np.float32(inv_tau)
    c = it * KLOG2E
    if mean:
        return c, it / (np.float32(2.0) * np.float32(n)), np.float32(0.5) / np.float32(n)
    return c, it * np.float32(0.5), np.float32(0.5)


# ================================================================================================ input builders
def permutation(n, kind, gen):
    """pi with no fixed point and pi != pi^-1, so that G is not symmetric: a cyclic shift by one ("shift") or a random
    such permutation.  n = 1: the identity, the only permutation there is."""
    r = torch.arange(n)
    if n == 1:
        return r
    if kind == "shift":
        return (r + 1) % n
    while True:
        pi = torch.randperm(n, generator=gen)
        if bool((pi != r).all()) and not torch.equal(pi[pi], r):
            return pi


def _fill(x, cols, gen):
    x[:, cols] = torch.randint(-3, 4, (x.shape[0], cols.numel()), generator=gen).float()


def perm_operands(n, D, pi, gen):
    """bf16 integers with A B^T = P, P_ij = [j == pi(i)]: row i of A has its 1 in column i, row j of B in column
    pi^-1(j).  Columns [n, D) alternate between fill in {-3..3} for A and for B, so dA (which sums rows of B) and dB
    (rows of A) are non-zero in every 128-column pass."""
    a, b = torch.zeros(n, D), torch.zeros(n, D)
    r = torch.arange(n)
    a[r, r] = 1.0
    b[pi, r] = 1.0
    rest = torch.arange(n, D)
    _fill(a, rest[0::2], gen)
    _fill(b, rest[1::2], gen)
    return a.bfloat16(), b.bfloat16()


def zero_operands(n, D, gen):
    """bf16 integers on disjoint supports (A on even columns, B on odd ones): z == 0."""
    a, b = torch.zeros(n, D), torch.zeros(n, D)
    cols = torch.arange(D)
    _fill(a, cols[0::2], gen)
    _fill(b, cols[1::2], gen)
    return a.bfloat16(), b.bfloat16()


def exact_cases(D):
    """(name, a, b, pi or None, lse2): the permutation cases (both kinds of pi) and the zero-logit ones."""
    out = []
    for n in PERM_ROWS:
        for kind in ("shift", "random"):
            gen = torch.Generator().manual_seed(1000 * n + D + (kind == "random"))
            pi = permutation(n, kind, gen)
            a, b = perm_operands(n, D, pi, gen)
            out.append((f"perm-{kind} n={n}", a, b, pi, int(round(math.log2(n + 1)))))
    for n in ZERO_ROWS:
        gen = torch.Generator().manual_seed(7 * n + D)
        a, b = zero_operands(n, D, gen)
        out.append((f"zero n={n}", a, b, None, int(round(math.log2(n)))))
    return out


def unit_pairs(n, D, gen):
    """fp32 unit rows b and a = unit(b + noise of norm about 0.75): cosine about 0.8 on the pairs, about 0 off them."""
    b = torch.nn.functional.normalize(torch.randn(n, D, generator=gen), dim=-1)
    a = torch.nn.functional.normalize(b + 0.75 / math.sqrt(D) * torch.randn(n, D, generator=gen), dim=-1)
    return a, b


def family(name, n, D, gen):
    """bf16 (a, b) of one input family:
    aligned      `unit_pairs`: the pairs the trainer produces;
    adversarial  mixed-sign near-equal rows in every 32-row group (`adversarial_pairs`);
    duplicates   aligned, with rows 2k + 1 of a and of b equal to rows 2k: ties in every row and column max;
    peaked       aligned, with row n // 2 of a replaced by 4 b[n // 2]: one row with one dominant logit;
    nonunit      aligned, rows of a and b scaled by norms in [1/4, 4] (the kernel does not normalise)."""
    if name == "adversarial":
        return adversarial_pairs(n, D, gen)
    a, b = unit_pairs(n, D, gen)
    if name == "duplicates":
        src = torch.arange(n) // 2 * 2
        a, b = a[src], b[src]
    elif name == "peaked":
        a[n // 2] = 4.0 * b[n // 2]
    elif name == "nonunit":
        a = a * torch.exp2(torch.rand(n, 1, generator=gen) * 4 - 2)
        b = b * torch.exp2(torch.rand(n, 1, generator=gen) * 4 - 2)
    return a.bfloat16(), b.bfloat16()


def split3_torch(x):
    """The two-term bf16 split in torch: hi = bf16(x), lo = bf16(x - hi); ([hi|lo|hi], [hi|hi|lo])."""
    hi = x.float().bfloat16()
    lo = (x.float() - hi.float()).bfloat16()
    return torch.cat([hi, lo, hi], 1), torch.cat([hi, hi, lo], 1)


# ================================================================================================ references
def closed_form(a, b, pi, lse2, inv_tau, mean):
    """The kernel's outputs for the exact inputs, from their structure alone: logits z_ij = [j == pi(i)] (pi None:
    z = 0), every row and column log2-sum-exp the integer lse2.  -> (loss, lse_row, lse_col, da, db), fp32, exact.

        lse      = fp32(lse2 * fp32(ln 2))
        G        = bf16(fp32(w 2^(z - lse2 + 1) - 2 w I))
        loss     = fp32(fp32(fp32(sum_i 2 (lse2 - z_ii)) * fp32(ln 2)) * loss_mult)
        dA, dB   = G B, G^T A   (exact)"""
    n = a.shape[0]
    c, w, lm = host_params(n, inv_tau, mean)
    assert c == np.float32(1.0), "inv_tau does not make the kernel's log2 scale exactly 1"
    z = torch.zeros(n, n, dtype=torch.float64)
    if pi is not None:
        z[torch.arange(n), pi] = 1.0
    wd = float(w)
    g = wd * torch.exp2(z - lse2 + 1) - 2 * wd * torch.eye(n, dtype=torch.float64)
    gb = g.float().bfloat16().double()
    lse = torch.full((n,), float(np.float32(lse2) * KLN2))
    s = np.float32(2 * (lse2 * n - float(z.diagonal().sum())))
    loss = np.float32(s * KLN2) * lm
    return (torch.tensor(float(loss)), lse, lse.clone(), (gb @ b.double()).float(), (gb.T @ a.double()).float())


def fp64_model(a, b, inv_tau, mean, scale2=None, grad_ops=None, fault=None, round_g=True):
    """The step in fp64 from its definition, keeping the roundings that are part of what the kernel defines: the fp32
    host weight w and G rounded to fp32, then to bf16 (round_g).

    a, b: the operands of the similarity (bf16, or the fp32 values of the split path); t = scale2 a b^T in log2 units
    (default fp32(inv_tau) log2 e).  grad_ops: (A, B[, A_lo]) of the gradient products (default a, b; the split
    path's hi parts).  fault: one of FAULTS, planted into the result (a fault in an lse reaches G and the loss as it
    would in the kernel).  The loss uses the exact factor 0.5 / n (mean) or 0.5 (sum).  -> dict"""
    n, D = a.shape[0], (grad_ops[0] if grad_ops is not None else a).shape[1]
    dev = a.device
    scale2 = float(np.float32(inv_tau)) * LOG2E if scale2 is None else scale2
    red = (not mean) if fault == "mean_sum_swapped" else mean
    _, w, lm = host_params(n, inv_tau, red)
    lm_exact = 0.5 / n if red else 0.5
    t = scale2 * (a.double() @ b.double().T)

    def lse2(x, dim):
        m = x.amax(dim, keepdim=True)
        return (m + torch.log2(torch.exp2(x - m).sum(dim, keepdim=True))).squeeze(dim)

    lr, lc = lse2(t, 1), lse2(t, 0)
    if fault == "padding_counted":          # a zero-filled padding column in every row sum: + exp2(0 - lse2)
        lr = lr + torch.log1p(torch.exp2(-lr)) * LOG2E
    elif fault == "lse_col_ln2":            # one column's lse too large by ln 2
        lc = lc.clone()
        lc[n // 2] += 1.0
    wd = float(w)
    pr, pc = torch.exp2(t - lr[:, None]), torch.exp2(t - lc[None, :])
    g = wd * (pr + pc) - 2 * wd * torch.eye(n, dtype=torch.float64, device=dev)
    if fault == "diag_missing":
        g[n // 2, n // 2] += 2 * wd
    gb = g.float().bfloat16().double() if round_g else g.clone()
    if fault == "g_chunk3_zeroed":          # columns 96..127 of G: chunk 3 of store_g_chunk
        gb[:, 96:128] = 0.0
    ops = (a, b) if grad_ops is None else grad_ops
    A, B = ops[0].double(), ops[1].double()
    da = gb @ B
    if fault == "db_untransposed":
        db = gb @ A
    elif fault == "split_lo_in_db":
        db = gb.T @ ops[2].double()
    else:
        db = gb.T @ A
    if fault == "pass_repeated":            # the last output pass holds the one before it
        both = torch.cat([da, db], 1)
        both[:, -128:] = both[:, -256:-128]
        da, db = both[:, :D], both[:, D:]
    diag = t.diagonal()
    sum2 = ((lr - diag) + (lc - diag)).sum()
    return dict(t=t, lse2_row=lr, lse2_col=lc, sum2=sum2, lm=lm, lm_exact=lm_exact, w=wd, pr=pr, pc=pc, g=g, gb=gb,
                da=da, db=db, loss=lm_exact * LN2 * sum2, lse_row=lr * LN2, lse_col=lc * LN2)


def kernel_rounding(m):
    """The fp32 outputs an exact model gives when rounded as the kernel rounds: lse = fp32(fp32(lse2) fp32(ln 2)),
    loss = fp32(fp32(fp32(sum2) fp32(ln 2)) loss_mult), dA and dB to fp32."""
    kl = torch.tensor(float(KLN2))
    loss = np.float32(np.float32(float(m["sum2"])) * KLN2) * m["lm"]
    return (torch.tensor(float(loss)), (m["lse2_row"].float().cpu() * kl), (m["lse2_col"].float().cpu() * kl),
            m["da"].float().cpu(), m["db"].float().cpu())


def applicable_faults(n, split=False, symmetric=False):
    """The planted faults that change the result of an n-row case: the transposition needs an asymmetric G, the mean /
    sum swap, the pass mix-up and the transposition need n >= 2 (at n = 1 G is 0 and both factors agree), chunk 3 of G
    exists for n > 96, the lo operand only on the split path."""
    out = ["lse_col_ln2", "diag_missing", "padding_counted"]
    if n >= 2:
        out += ["mean_sum_swapped", "pass_repeated"] + ([] if symmetric else ["db_untransposed"])
    if n > 96:
        out.append("g_chunk3_zeroed")
    if split:
        out.append("split_lo_in_db")
    return out


def exact_mismatch(out, ref):
    """-> the names of the outputs that differ from ref bit for bit"""
    return [nm for nm, o, r in zip(OUTS, out, ref) if not torch.equal(o.float().cpu(), r.float().cpu())]


def ulp_diff(o, r):
    """Largest difference in fp32 ulps of the reference (for the failure message)."""
    o, r = o.double().cpu(), r.double().cpu()
    _, e = torch.frexp(r.float())
    return float(((o - r).abs() / torch.ldexp(torch.ones_like(r), (e - 24).to(torch.int32))).max())


# ================================================================================================ bounded checks
def lse_tol(lse, n, dzs, tmax):
    """Bound on |lse_kernel - lse_fp64| (natural log) per element.  The kernel takes t = fp32(z~ c), the row max m,
    s = sum_j ex2(t_j - m) as a serial fp32 sum, lr = m + log2f(s) and lse = fp32(lr kLn2).

    * the logits: |z~ - z| <= dz (fp32 accumulation over the depth, `dot_err`; the split path adds its dropped terms),
      c and the product rounded (3 * 2^-24 |t|).  lse is 1-Lipschitz in the max norm of t, so this moves lse2 by at
      most dzs + 3 * 2^-24 tmax, dzs = scale2 dz;
    * s, relatively (the relative error of s is the absolute error of ln s): ex2.approx 2^-22, the serial sum of
      n terms below s (n - 1) 2^-24, each argument t_j - m rounded (|t_j - m| <= 2 tmax: 2^-23 tmax in log2 units);
    * log2f: 2 ulps of a result below 8 (2^-20); m + log2f(s) rounded and the product with fp32(ln 2) rounded
      twice: 2^-22 |lse|.

        tol = ln 2 (dzs + 2^-21 tmax + 2^-20) + 2^-22 + n 2^-24 + 2^-22 |lse|"""
    return LN2 * (dzs + 2.0 ** -21 * tmax + 2.0 ** -20) + 2.0 ** -22 + n * 2.0 ** -24 + 2.0 ** -22 * lse.abs()


def lse_arith(t, p, lse2, dim):
    """Error of the kernel's lse2 (log2 units) beyond its logits, per row (dim = 1) or column (dim = 0): the relative
    error of s = sum_j ex2(t_j - m) (ex2.approx 2^-22, the serial fp32 sum (n - 1) 2^-24, each argument t_j - m
    rounded: ln 2 2^-24 |t_j - m| weighted by its share p_j, doubled for p~ against p), log2f (2 ulps of a result below
    8: 2^-20) and m + log2f(s) rounded (2^-24 |lse2|)."""
    n = t.shape[dim]
    m = t.amax(dim, keepdim=True)
    rel = 2.0 ** -22 + (n - 1) * 2.0 ** -24 + LN2 * 2.0 ** -23 * (p * (t - m).abs()).sum(dim)
    return LOG2E * rel + 2.0 ** -20 + 2.0 ** -24 * lse2.abs()


def loss_tol(ref, dt, ar, ac):
    """Bound on |loss_kernel - loss_fp64|, loss = loss_mult ln 2 sum_i (lr_i - t_ii) + (lc_i - t_ii).

    The kernel's loss is that of its own logits t~ (|t~ - t| <= dt): d loss / d t_ij = loss_mult ln 2
    (P_row + P_col - 2 I)_ij, so the logit error moves it by at most loss_mult ln 2 dt sum_ij |P_row + P_col - 2 I|
    (plus 4 n dt^2 for the softmax at an intermediate point); a peaked softmax, where the loss itself is small, cancels
    it.  Then the lse arithmetic beyond the logits (`lse_arith`, ar / ac) and the fp32 arithmetic of the sum (3
    roundings per row, 7 levels of the 128-value reduction: 16 * 2^-24 of sum_i |s_i|), the products with fp32(ln 2)
    and the fp32 loss_mult (4 * 2^-24 of the loss)."""
    n = ref["t"].shape[0]
    eye = torch.eye(n, dtype=torch.float64, device=ref["t"].device)
    diag = ref["t"].diagonal()
    s = ((ref["lse2_row"] - diag) + (ref["lse2_col"] - diag)).abs().sum()
    grad = (ref["pr"] + ref["pc"] - 2 * eye).abs().sum()
    return (ref["lm_exact"] * LN2 * (dt * (grad + 4 * n * dt) + ar.sum() + ac.sum() + 16 * 2.0 ** -24 * s)
            + 4 * 2.0 ** -24 * ref["loss"].abs())


def exp_err(ref, dt, ar, ac):
    """Bound on |G~_ij - G_ij| before G~ is rounded to bf16, G = w (P_row + P_col) - 2 w I from the fp64 lse.

    The kernel forms P~_ij = ex2(fl(t~_ij - lr~_i)) from its own logits t~ (|t~ - t| <= dt, log2 units) and the lse2
    lr~ it computed from them.  The logit error cancels through the lse: log2 P_ij = t_ij - lse2_i(t) changes by
    (1 - p_ij) d_j - sum_(k != j) p_ik d_k at an intermediate point, at most 2 dt (1 - p_ij + 2 dt).  A peaked row
    (p_ii ~ 1, where G_ii = -2 w (1 - p_ii) is a small difference) therefore keeps its gradient to fp32 resolution.
    Per exponential, relatively: ex2.approx 2^-22; the sum of the two and the product with w rounded, 2^-23; and
    ln 2 times the argument's error in log2 units: the cancelled logit error, the rounding of t - lr (2^-24
    |t - lr|) and the lse arithmetic beyond the logits (`lse_arith`)."""
    t, pr, pc = ref["t"], ref["pr"], ref["pc"]
    er = 2.0 ** -22 + 2.0 ** -23 + LN2 * (2 * dt * (1 - pr + 2 * dt) + 2.0 ** -24 * (t - ref["lse2_row"][:, None]).abs()
                                         + ar[:, None])
    ec = 2.0 ** -22 + 2.0 ** -23 + LN2 * (2 * dt * (1 - pc + 2 * dt) + 2.0 ** -24 * (t - ref["lse2_col"][None, :]).abs()
                                         + ac[None, :])
    return ref["w"] * (er * pr + ec * pc)


class Check:
    """The bounded comparison of one kernel result out = (loss, lse_row, lse_col, da, db) with the fp64 model.

    lse_row, lse_col per element within `lse_tol`; the loss within `loss_tol`; dA, dB per row against bf16(G) B,
    bf16(G)^T A within `row_bound` with the per-element exponential error `exp_err` (K = 128 terms per product: the
    padded tile).  dz: the bound on the logit error before scaling (default: the fp32 accumulation of a b^T,
    `dot_err`; the split path's `split_dz`)."""

    def __init__(self, out, a, b, inv_tau, mean, grad_ops=None, dz=None):
        self.out = tuple(o.double() for o in out)
        self.a, self.b, self.inv_tau, self.mean, self.grad_ops = a, b, inv_tau, mean, grad_ops
        n = a.shape[0]
        an, bn = a.double().norm(dim=1), b.double().norm(dim=1)
        dz = dot_err(a.shape[1], 1.0, float(an.max()), float(bn.max())) if dz is None else dz
        self.ref = ref = self.model()
        t = ref["t"]
        tmax = float(t.abs().max())
        dzs = float(np.float32(inv_tau)) * LOG2E * dz
        dt = dzs + 3 * 2.0 ** -24 * tmax            # t = fp32(z~ c): c and the product rounded
        ar = lse_arith(t, ref["pr"], ref["lse2_row"], 1)
        ac = lse_arith(t, ref["pc"], ref["lse2_col"], 0)
        self.tol = {"lse_row": lse_tol(ref["lse_row"], n, dzs, tmax), "lse_col": lse_tol(ref["lse_col"], n, dzs, tmax),
                    "loss": loss_tol(ref, dt, ar, ac).reshape(())}
        self.err_g = exp_err(ref, dt, ar, ac)
        ops = (a, b) if grad_ops is None else grad_ops
        self.norms = An, Bn = ops[0].double().norm(dim=1), ops[1].double().norm(dim=1)
        ga = ref["g"].abs()
        _, flip = bf16_flips(ref["g"], self.err_g + 2.0 ** -23 * ga)
        self.tol["da"] = row_bound(ga @ Bn, flip @ Bn, self.err_g @ Bn, TILE, 1.0)
        self.tol["db"] = row_bound(ga.T @ An, flip.T @ An, self.err_g.T @ An, TILE, 1.0)

    def model(self, fault=None, round_g=True):
        return fp64_model(self.a, self.b, self.inv_tau, self.mean, grad_ops=self.grad_ops, fault=fault,
                          round_g=round_g)

    def ratios(self, ref):
        """-> {output: largest error / bound} of the kernel result against ref"""
        r = {}
        for nm, o in zip(OUTS, self.out):
            if nm in ("da", "db"):
                r[nm] = rows_within(o, ref[nm], self.tol[nm])[1]
            else:
                r[nm] = float(((o - ref[nm]).abs() / self.tol[nm]).max())
        return r

    def resolvable(self, fault):
        """Whether a planted fault changes some exact output (G unrounded) by more than rounding may move it.

        The floor of an lse is 2^-13 max(1, |lse|); of the loss 2^-13 loss_mult ln 2 sum_i |lr| + |lc| + 2 |t_ii|; of
        a row of dA (dB) 2^-13 w sum_j (P_row + P_col)_ij ||b_j||, the size of the terms that cancel to form it, plus
        sum_j s_ij ||b_j||, s_ij <= 2^-7 |G_ij| the bf16 spacing of G_ij (the most its rounding to bf16 may move the
        row).  The kernel's fp32 arithmetic may be off by (n - 1) 2^-24 ~ 2^-17 of those magnitudes (the serial sum of
        128 exponentials), ex2.approx by 2^-22: a fault beyond 2^-13 is resolvable, a smaller one is not told apart
        from rounding by any fp32 kernel.  At tau = 0.03 with aligned unit rows the whole gradient is about e^-20 w,
        so the faults that scale it are not planted there; the exact tests plant every fault in every case."""
        ref, bad = self.model(round_g=False), self.model(fault, round_g=False)
        e = ref["w"] * (ref["pr"] + ref["pc"])
        ga = ref["g"].abs()
        An, Bn = self.norms
        diag = ref["t"].diagonal().abs()
        floor = {"lse_row": 2.0 ** -13 * ref["lse_row"].abs().clamp_min(1.0),
                 "lse_col": 2.0 ** -13 * ref["lse_col"].abs().clamp_min(1.0),
                 "loss": 2.0 ** -13 * ref["lm_exact"] * LN2 * (ref["lse2_row"].abs() + ref["lse2_col"].abs()
                                                                + 2 * diag).sum(),
                 "da": 2.0 ** -13 * (e @ Bn) + 2.0 ** -7 * (ga @ Bn),
                 "db": 2.0 ** -13 * (e.T @ An) + 2.0 ** -7 * (ga.T @ An)}
        for nm in OUTS:
            d = (bad[nm] - ref[nm]).norm(dim=1) if nm in ("da", "db") else (bad[nm] - ref[nm]).abs()
            if bool((d > floor[nm]).any()):
                return True
        return False

    def run(self, faults, what, log=print):
        """Assert every output within its bound and each planted fault that fp32 can resolve outside;
        -> {fault: ratio it is seen by}"""
        worst = self.ratios(self.ref)
        log(f"[worst error/bound] {what}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        bad = {k: v for k, v in worst.items() if not v <= 1.0}
        assert not bad, (what, bad)
        seen = {}
        for f in faults:
            if self.resolvable(f):
                seen[f] = max(self.ratios(self.model(f)).values())
                assert seen[f] > 1.0, (what, f, "planted fault not rejected", seen[f])
        return seen


def emulate(a, b, inv_tau, mean, grad_ops=None, gen=None):
    """The kernel's arithmetic restated in fp32 torch (CPU): t = fp32(z) c; per row and per column the max, the fp32 sum
    of exp2(t - m), lse2 = m + log2(s); loss = ((sum_i (lr - t_ii) + (lc - t_ii)) kLn2) loss_mult;
    G = w (exp2(t - lr) + exp2(t - lc)) - 2 w I in fp32, rounded to bf16; dA = bf16(G) B, dB = bf16(G)^T A in fp32.
    With gen, every exponential carries a relative error of up to 2^-23 (half of what ex2.approx may have)."""
    n = a.shape[0]
    c, w, lm = host_params(n, inv_tau, mean)

    def ex2(x):
        y = torch.exp2(x)
        if gen is not None:
            noise = (torch.rand(x.shape, generator=gen, dtype=torch.float64) - 0.5) * 2.0 ** -22
            y = (y.double() * (1 + noise)).float()
        return y

    t = (a.float() @ b.float().T) * float(c)
    m = t.amax(1)
    lr = m + torch.log2(ex2(t - m[:, None]).sum(1))
    m = t.amax(0)
    lc = m + torch.log2(ex2(t - m[None, :]).sum(0))
    d = t.diagonal()
    loss = ((((lr - d) + (lc - d)).sum() * float(KLN2)) * float(lm)).reshape(())
    g = float(w) * (ex2(t - lr[:, None]) + ex2(t - lc[None, :]))
    g = g - 2 * float(w) * torch.eye(n)
    gb = g.bfloat16().float()
    A, B = ((a, b) if grad_ops is None else grad_ops)[:2]
    return loss, lr * float(KLN2), lc * float(KLN2), gb @ B.float(), gb.T @ A.float()


def split_dz(x, y, l3, r3):
    """Logit error of the three-term split product [hi|lo|hi] . [hi|hi|lo] against x . y: its fp32 accumulation over
    3 D (`dot_err` with the norms of the split rows) and the terms it drops.  With |lo| <= 2^-9 |x| and
    |x - hi - lo| <= 2^-18 |x|, each product x_k y_k loses lo lo' and the residues:
    <= (2^-18 + 2 * 2^-18 (1 + 2^-8)) |x_k| |y_k| < 2^-16 |x_k| |y_k|; summed, <= 2^-16 ||x|| ||y||."""
    nrm = lambda t: float(t.double().norm(dim=1).max())  # noqa: E731
    return dot_err(l3.shape[1], 1.0, nrm(l3), nrm(r3)) + 2.0 ** -16 * nrm(x) * nrm(y)


# the faults the looser true-gradient check must see as well (a transposed G is left to the contract check: the
# allowance for bf16(G) and B_hi is about as large as G's asymmetric part at tau = 0.5)
TRUE_GRAD_FAULTS = ("diag_missing", "split_lo_in_db", "mean_sum_swapped", "pass_repeated")


def true_grad_check(out, x, y, inv_tau, mean, chk, l3, faults, what, log=print):
    """The split path's gradients against the true fp64 gradient of the fp32 inputs (G unrounded, from fp64 lse,
    times the fp32 operands).  Beyond the contract bound it allows the two roundings the contract makes, bf16(G)
    and B_hi (each 2^-9 relative): 2^-8 sum_j |G_ij| ||y_j|| doubled for margin, 2^-7 in all."""
    D = x.shape[1]
    ops = (x, y, l3[:, D:2 * D])
    tm = fp64_model(x, y, inv_tau, mean, grad_ops=ops, round_g=False)
    xn, yn = x.double().norm(dim=1), y.double().norm(dim=1)
    ga = tm["g"].abs()
    bounds = (chk.tol["da"] + 2.0 ** -7 * (ga @ yn), chk.tol["db"] + 2.0 ** -7 * (ga.T @ xn))
    worst = [rows_within(o.double(), tm[nm], bd)[1] for o, nm, bd in zip(out[3:], ("da", "db"), bounds)]
    log(f"[worst error/bound] {what} true gradient: da {worst[0]:.3g} db {worst[1]:.3g}")
    assert max(worst) <= 1.0, (what, worst)
    seen = {}
    for f in faults:
        fm = fp64_model(x, y, inv_tau, mean, grad_ops=ops, round_g=False, fault=f)
        seen[f] = max(rows_within(o.double(), fm[nm], bd)[1] for o, nm, bd in zip(out[3:], ("da", "db"), bounds))
    return seen


# ================================================================================================ CPU tests
def test_host_scale_is_exactly_one():
    """inv_tau = fp32(0.6931472): the host's c = fp32(inv_tau * fp32(log2 e)) is exactly 1, so t = z."""
    c, _, _ = host_params(1, EXACT_INV_TAU, True)
    assert c == np.float32(1.0)
    assert np.float32(np.float32(0.6931471) * KLOG2E) != np.float32(1.0)     # the neighbour does not: c is not slack


@pytest.mark.parametrize("D", DIMS)
def test_exact_builders(D):
    """A B^T is the permutation (or zero) matrix exactly; pi has no fixed point and pi != pi^-1; fill in {-3..3}
    reaches every 128-column pass of dA and of dB (D >= 256)."""
    for name, a, b, pi, lse2 in exact_cases(D):
        n = a.shape[0]
        z = a.double() @ b.double().T
        if pi is None:
            assert torch.equal(z, torch.zeros(n, n, dtype=torch.float64)), name
            assert 2 ** lse2 == n
        else:
            p = torch.zeros(n, n, dtype=torch.float64)
            p[torch.arange(n), pi] = 1.0
            assert torch.equal(z, p), name
            assert 2 ** lse2 == n + 1
            if n > 1:
                r = torch.arange(n)
                assert bool((pi != r).all()) and not torch.equal(pi[pi], r), name
        for t in (a, b):
            assert torch.equal(t.double(), t.double().round()) and float(t.double().abs().max()) <= 3
        if D >= 256:
            for p0 in range(0, D, 128):
                assert bool((a[:, p0:p0 + 128] != 0).any()) and bool((b[:, p0:p0 + 128] != 0).any()), (name, p0)


@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("D", DIMS)
def test_closed_form_equals_fp64_model(D, mean):
    """The closed forms equal the fp64 model from the definition (every lse2 the integer claimed, G, dA, dB, loss
    bit for bit after the kernel's roundings), and an fp32 emulation of the kernel with exact exponentials; every
    entry of bf16(G) is a multiple of the off-diagonal ulp u and every partial sum of |bf16(G)| |B|, |bf16(G)|^T |A|
    stays below 2^19 u (so any fp32 summation order is exact)."""
    inv_tau = EXACT_INV_TAU
    for name, a, b, pi, lse2 in exact_cases(D):
        n = a.shape[0]
        ref = closed_form(a, b, pi, lse2, inv_tau, mean)
        m = fp64_model(a, b, inv_tau, mean, scale2=1.0)
        assert torch.equal(m["lse2_row"], torch.full((n,), float(lse2), dtype=torch.float64)), name
        assert torch.equal(m["lse2_col"], torch.full((n,), float(lse2), dtype=torch.float64)), name
        assert exact_mismatch(kernel_rounding(m), ref) == [], name
        assert exact_mismatch(emulate(a, b, inv_tau, mean), ref) == [], name
        if n == 1:
            assert float(ref[0]) == 0.0 and float(ref[3].abs().max()) == 0.0
            continue
        _, w, _ = host_params(n, inv_tau, mean)
        _, ew = math.frexp(float(w))
        u = 2.0 ** (ew - 8 + 1 - lse2)                    # ulp of bf16(w 2^(1 - lse2)), the smallest entry
        gb = m["gb"]
        assert torch.equal(gb / u, (gb / u).round()), name
        for prod in (gb.abs() @ b.double().abs(), gb.abs().T @ a.double().abs()):
            assert float(prod.max()) < 2.0 ** 19 * u, name


@pytest.mark.parametrize("D", [128, 384])
def test_exact_checker_rejects_planted_faults(D):
    """Each planted fault changes some output of every exact case it applies to (the bit-exact comparison sees it)."""
    for mean in (True, False):
        for name, a, b, pi, lse2 in exact_cases(D):
            n = a.shape[0]
            ref = closed_form(a, b, pi, lse2, EXACT_INV_TAU, mean)
            for f in applicable_faults(n, symmetric=pi is None):
                bad = kernel_rounding(fp64_model(a, b, EXACT_INV_TAU, mean, scale2=1.0, fault=f))
                assert exact_mismatch(bad, ref) != [], (name, mean, f)


CPU_BOUNDED = [(8, 512, True), (33, 128, False), (127, 384, True), (128, 256, False), (1, 128, True), (65, 512, True)]


@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_bounded_checks_accept_emulation_and_reject_faults(fam, tau):
    """The bounded checks accept an fp32 emulation of the kernel (approximate exponentials, fp32 sums, bf16 G) and
    reject every planted fault that applies, on CPU-sized cases of each family."""
    inv_tau = float(np.float32(1.0 / tau))
    for n, D, mean in CPU_BOUNDED:
        gen = torch.Generator().manual_seed(n * 1000 + D + int(100 * tau))
        a, b = family(fam, n, D, gen)
        out = emulate(a, b, inv_tau, mean, gen=gen)
        chk = Check(out, a, b, inv_tau, mean)
        faults = applicable_faults(n)
        chk.run(faults, f"emulation {fam} tau={tau} n={n} D={D} mean={mean}", log=lambda *x: None)


@pytest.mark.parametrize("n", [8, 64, 128])
def test_split_checks_accept_emulation_and_reject_faults(n):
    """The split path's checks (contract and true gradient) accept an fp32 emulation of the kernel on the split
    operands and reject every planted fault, A_lo in dB included."""
    D, inv_tau = 512, float(np.float32(1 / 0.07))
    gen = torch.Generator().manual_seed(n)
    x, y = unit_pairs(n, D, gen)
    l3, _ = split3_torch(x)
    _, r3 = split3_torch(y)
    ops = (l3[:, :D], r3[:, :D], l3[:, D:2 * D])
    out = emulate(l3, r3, inv_tau, True, grad_ops=ops, gen=gen)
    chk = Check(out, x, y, inv_tau, True, grad_ops=ops, dz=split_dz(x, y, l3, r3))
    faults = applicable_faults(n, split=True)
    chk.run(faults, f"split emulation n={n}", log=lambda *x: None)
    seen = true_grad_check(out, x, y, inv_tau, True, chk, l3, TRUE_GRAD_FAULTS, "split emulation",
                           log=lambda *x: None)
    assert min(seen.values()) > 1.0, seen


def test_split3_torch_reference():
    """split3_torch: hi + lo recovers x to 2^-16 relative, lo = 0 for bf16-exact values."""
    x = torch.randn(16, 64, generator=torch.Generator().manual_seed(3))
    l3, r3 = split3_torch(x)
    hi, lo = l3[:, :64].float(), l3[:, 64:128].float()
    assert bool(((hi + lo - x).abs() <= 2.0 ** -16 * x.abs()).all())
    assert torch.equal(r3[:, 128:], l3[:, 64:128]) and torch.equal(r3[:, :64], l3[:, 128:])
    xb = x.bfloat16().float()
    assert bool((split3_torch(xb)[0][:, 64:128] == 0).all())


def test_support_boundaries():
    """pgica_ntxent_small_supported: 1 <= rows <= 128 and dim in {128, 256, 384, 512}, nothing else."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    for rows in (0, 1, 128, 129):
        for dim in (64, 127, 128, 130, 256, 384, 512, 640):
            want = 1 <= rows <= 128 and dim in (128, 256, 384, 512)
            assert F.ntxent_small_supported(rows, dim) == want, (rows, dim)


# ================================================================================================ GPU tests
@pytest.fixture(scope="module")
def F(cuda_device):
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional
    lib = _lib.load()
    assert lib.pgica_device_check() == 0, lib.pgica_last_error()
    return functional


# ------------------------------------------------------------------------------------------------ 1. exact
@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("D", DIMS)
def test_ntxent_small_exact_permutation_logits(F, cuda_device, D, mean):
    """Permutation logits (n = 2^m - 1, pi a cyclic shift and a random derangement with pi != pi^-1) and zero logits
    (n a power of two): loss, lse_row, lse_col, dA and dB equal the closed form bit for bit; each planted fault that
    applies is rejected by the same comparison."""
    for name, a, b, pi, lse2 in exact_cases(D):
        n = a.shape[0]
        ref = closed_form(a, b, pi, lse2, EXACT_INV_TAU, mean)
        out = F.ntxent_small(a.to(cuda_device), b.to(cuda_device), float(EXACT_INV_TAU), mean)
        torch.cuda.synchronize()
        bad = exact_mismatch(out, ref)
        assert bad == [], (name, D, mean, {nm: ulp_diff(o, r) for nm, o, r in zip(OUTS, out, ref) if nm in bad})
        for f in applicable_faults(n, symmetric=pi is None):
            wrong = kernel_rounding(fp64_model(a, b, EXACT_INV_TAU, mean, scale2=1.0, fault=f))
            assert exact_mismatch(out, wrong) != [], (name, f, "planted fault not rejected")
    print(f"[exact] D={D} mean={mean}: {len(exact_cases(D))} cases bit-exact ({card()})")


# ------------------------------------------------------------------------------------------------ 2. bounded
@pytest.mark.gpu
@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_ntxent_small_bounded_fp64(F, cuda_device, fam, tau):
    """Every n in ROWS (warp and 32-column-chunk edges, the trainer's 8, config 1's 64, 128), every D, mean and sum:
    lse_row, lse_col and loss per element and dA, dB per row within their bounds of fp64; every planted fault that
    applies is rejected (the smallest ratio by which each is seen is printed)."""
    inv_tau = float(np.float32(1.0 / tau))
    worst, seen, planted, cases = 0.0, {}, {}, 0
    for n in ROWS:
        for D in DIMS:
            gen = torch.Generator().manual_seed(n * 1000 + D + int(100 * tau))
            a, b = family(fam, n, D, gen)
            a, b = a.to(cuda_device), b.to(cuda_device)
            for mean in (True, False):
                out = F.ntxent_small(a, b, inv_tau, mean)
                chk = Check(out, a, b, inv_tau, mean)
                for f, v in chk.run(applicable_faults(n), f"{fam} tau={tau} n={n} D={D} mean={mean}").items():
                    seen[f] = min(seen.get(f, math.inf), v)
                    planted[f] = planted.get(f, 0) + 1
                worst = max(worst, max(chk.ratios(chk.ref).values()))
                cases += 1
    report(f"{fam} tau={tau} all {cases} cases", worst)
    for f, v in sorted(seen.items()):
        print(f"[fault error/bound] {fam} tau={tau} {f}: planted in {planted[f]} of {cases} cases, seen by >= {v:.3g}")


# ------------------------------------------------------------------------------------------------ 3. split path
def split_inputs(n, D, seed):
    """fp32 unit pairs as the trainer hands them over (normalised in fp32, not rounded to bf16)."""
    return unit_pairs(n, D, torch.Generator().manual_seed(seed))


@pytest.mark.gpu
def test_split3_bit_exact(F, cuda_device):
    """split3 equals hi = bf16(x), lo = bf16(x - hi) laid out [hi|lo|hi], [hi|hi|lo] bit for bit: ordinary values,
    values already exact in bf16 (lo = 0), fp32 subnormals and normal values whose lo is subnormal."""
    gen = torch.Generator().manual_seed(17)
    x = torch.randn(64, 256, generator=gen)
    x[8:16] = x[8:16].bfloat16().float()                                     # lo = 0
    x[16:24] *= 2.0 ** -130                                                  # subnormal x
    x[24:32] = 2.0 ** -118 * (1 + x[24:32].bfloat16().float().abs()) + 2.0 ** -140 * torch.randint(
        -5, 6, (8, 256), generator=gen).float()                              # normal hi, subnormal lo
    x[32:40] *= 2.0 ** 100
    x[40, :8] = torch.tensor([0.0, -0.0, 2.0 ** -149, -2.0 ** -149, 2.0 ** -126, 3.0 * 2.0 ** -133, 1.0, -1.0])
    assert bool(((x[16:24] != 0) & (x[16:24].abs() < 2.0 ** -126)).any())
    l3, r3 = F.split3(x.to(cuda_device))
    rl, rr = split3_torch(x)
    lo = rl[24:32, 256:512].float()
    assert bool(((lo != 0) & (lo.abs() < 2.0 ** -126)).any())               # the subnormal lo are there
    assert torch.equal(l3.cpu().view(torch.int16), rl.view(torch.int16))
    assert torch.equal(r3.cpu().view(torch.int16), rr.view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 64, 127, 128])
@pytest.mark.parametrize("tau", [0.07, 0.5])
def test_ntxent_small_split_fp64(F, cuda_device, n, tau):
    """The fp32 split path at D = 512 (n = 8: the trainer's call): lse and loss against fp64 of the fp32 values within
    the bounds plus the split product's logit error (`split_dz`); dA, dB against the contract bf16(G) B_hi,
    bf16(G)^T A_hi per row, and against the true fp64 gradient within the looser bound; every planted fault that
    applies (A_lo in dB included) is rejected by each."""
    from preference_guided_image_captioning_alignment_b200.ops import _ntxent_small_impl
    D, inv_tau = 512, float(np.float32(1.0 / tau))
    x, y = split_inputs(n, D, n + int(100 * tau))
    x, y = x.to(cuda_device), y.to(cuda_device)
    l3, _ = F.split3(x)
    _, r3 = F.split3(y)
    for mean in (True, False):
        out = F.ntxent_small_split(l3, r3, D, inv_tau, mean)
        ops = (l3[:, :D], r3[:, :D], l3[:, D:2 * D])
        chk = Check(out, x, y, inv_tau, mean, grad_ops=ops, dz=split_dz(x, y, l3, r3))
        faults = applicable_faults(n, split=True)
        what = f"split tau={tau} n={n} mean={mean}"
        for f, v in chk.run(faults, what).items():
            print(f"[fault error/bound] {what} {f}: {v:.3g}")
        gfaults = [f for f in TRUE_GRAD_FAULTS if f in faults]
        for f, v in true_grad_check(out, x, y, inv_tau, mean, chk, l3, gfaults, what).items():
            print(f"[fault error/bound] {what} true gradient {f}: {v:.3g}")
            assert v > 1.0, (what, f)
        again = _ntxent_small_impl(x, y, inv_tau, mean)           # the op's own call: the same launch
        assert all(torch.equal(o, p) for o, p in zip(out, again))


# ------------------------------------------------------------------------------------------------ 5. dispatch
@pytest.mark.gpu
def test_ntxent_auto_both_sides_of_the_dispatch(F, cuda_device):
    """ntxent_auto at n = 128 (this kernel) and n = 129 (the general kernels) on the same aligned bf16 family, both
    against the same fp64 reference: lse per element (this kernel: lse_tol; the general one: 16 ulps plus the logit
    error), the loss, and the bf16 gradients per row.  The general kernels recompute the logits in the backward, so
    nothing here relies on the logit error cancelling: eps_p = 3 * 2^-22 + 2^-23 + ln 2 (2 dt + 2^-21 (tmax + lmax2))
    plus the measured lse error, the loss within loss_mult (sum of the lse bounds + 2 n ln 2 dt + its arithmetic),
    and the rounding of each gradient row to bf16 (2^-9 of it) on top of row_bound."""
    from preference_guided_image_captioning_alignment_b200 import ops
    D, tau = 512, 0.07
    inv_tau = float(np.float32(1.0 / tau))
    a0, b0 = family("aligned", 129, D, torch.Generator().manual_seed(129))
    for n in (128, 129):
        assert F.ntxent_small_supported(n, D) == (n == 128)
        a = a0[:n].to(cuda_device).requires_grad_(True)
        b = b0[:n].to(cuda_device).requires_grad_(True)
        loss, lse_row, lse_col = ops.ntxent_auto(a, b, inv_tau, True)
        loss.backward()
        ref = fp64_model(a.detach(), b.detach(), inv_tau, True)
        an, bn = a.detach().double().norm(dim=1), b.detach().double().norm(dim=1)
        dzs = inv_tau * LOG2E * dot_err(D, 1.0, float(an.max()), float(bn.max()))
        tmax = float(ref["t"].abs().max())
        dt = dzs + 3 * 2.0 ** -24 * tmax
        worst, tols = {}, {}
        for nm, got in (("lse_row", lse_row), ("lse_col", lse_col)):
            tols[nm] = lse_tol(ref[nm], n, dzs, tmax) if n == 128 else ulps(ref[nm], 16) + dzs * LN2
            worst[nm] = float(((got.double() - ref[nm]).abs() / tols[nm]).max())
        diag = ref["t"].diagonal().abs()
        mag = (ref["lse2_row"].abs() + ref["lse2_col"].abs() + 2 * diag).sum() * LN2
        ltol = (ref["lm_exact"] * (tols["lse_row"].sum() + tols["lse_col"].sum() + 2 * n * LN2 * dt
                                   + 16 * 2.0 ** -24 * mag) + 4 * 2.0 ** -24 * ref["loss"].abs())
        worst["loss"] = float((loss.detach().double() - ref["loss"]).abs() / ltol)
        lse_err = float(torch.cat([lse_row.double() - ref["lse_row"], lse_col.double() - ref["lse_col"]]).abs().max())
        lmax2 = float(torch.cat([ref["lse2_row"], ref["lse2_col"]]).abs().max())
        eps_p = 3 * 2.0 ** -22 + 2.0 ** -23 + LN2 * (2 * dt + 2.0 ** -21 * (tmax + lmax2)) + lse_err
        g = ref["g"]
        e = ref["w"] * (ref["pr"] + ref["pc"])
        ga = g.abs()
        _, flip = bf16_flips(g, eps_p * e + 2.0 ** -23 * ga)
        k = max(n, TILE)
        for nm, grad, bnd in (("da", a.grad, row_bound(ga @ bn, flip @ bn, e @ bn, k, eps_p)),
                              ("db", b.grad, row_bound(ga.T @ an, flip.T @ an, e.T @ an, k, eps_p))):
            assert grad.dtype == torch.bfloat16
            bnd = bnd + 2.0 ** -9 * (ref[nm].norm(dim=1) + bnd)
            worst[nm] = rows_within(grad, ref[nm], bnd)[1]
        print(f"[worst error/bound] ntxent_auto n={n}: " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        assert max(worst.values()) <= 1.0, (n, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_upstream_gradient_scaling_exact(F, cuda_device, dtype):
    """_NTXentSmallEager and the pgica::ntxent_small op hand back da * g_loss and db * g_loss cast to the input dtype,
    bit for bit, for g_loss in {3, -0.25}."""
    from preference_guided_image_captioning_alignment_b200 import ops
    inv_tau = float(np.float32(1 / 0.07))
    for n in (8, 64):
        x, y = split_inputs(n, 512, 5 * n)
        a0, b0 = x.to(cuda_device).to(dtype), y.to(cuda_device).to(dtype)
        _, _, _, da, db = ops._ntxent_small_impl(a0, b0, inv_tau, True)
        for g in (3.0, -0.25):
            for via in ("eager", "op"):
                a, b = a0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
                if via == "eager":
                    loss = ops._NTXentSmallEager.apply(a, b, inv_tau, True)[0]
                else:
                    loss = torch.ops.pgica.ntxent_small(a, b, inv_tau, True)[0]
                (loss * g).backward()
                assert a.grad.dtype == dtype and b.grad.dtype == dtype
                assert torch.equal(a.grad, (da * g).to(dtype)), (n, g, via, "da")
                assert torch.equal(b.grad, (db * g).to(dtype)), (n, g, via, "db")
