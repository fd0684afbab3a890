"""Tile-level exactness of the tensor-core heads.

A global norm such as rel(out, ref) < 1e-2 does not notice one 128 x 128 tile of G lost in the exchange ring or
scheduled twice: at the benchmarked shapes that moves dW by a fraction of a percent.  The tests here check every row.

1. Exact inputs.  Every backward kernel builds G from fast_exp2(z * c - lse * log2 e).  With x supported on columns
   [k/2, k) and y on [0, k/2), z == 0 exactly; with lse == 0 every exponential is exp2(0) = 1, so

       G_ij = r_coef_i (1 - [j == r_tgt_i]) + c_coef_j (1 - [i == c_tgt_j]).

   Coefficients in {-2..2} (or a power of two), entries in {-3..3}: G is exact in bf16 and every partial sum of G y
   and G^T x is an integer (times a power of two) below 2^24, exact in fp32 in any summation order.  The closed-form
   reference (`closed_form`) then has to equal the kernel bit for bit.  The forward kernels get integer operands, so
   z is an exact integer: `similarity`, `tgt`, `ztgt` and `diag` are bit-exact, lse per row / column within a few
   fp32 ulps of fp64.
2. Where the arithmetic is approximate (the shared-exponential NT-Xent path, GPT-2-like logits), an fp64 reference
   from the same bf16 operands and a per-row error bound derived from the kernel's arithmetic (`row_bound`).
3. Every check is applied to the reference with a planted fault (`planted_faults`) and must reject it.

The helpers are plain torch and run on the CPU as well; the tests not marked `gpu` check them there.
"""
import ctypes
import math

import pytest
import torch

TILE = 128
LN2 = math.log(2.0)
LOG2E = 1.0 / LN2


# ================================================================================================ input builders
def int_operands(mx, my, k, gen, device="cpu", lo=-3, hi=3):
    """bf16 integer operands with disjoint supports: x in columns [k/2, k), y in [0, k/2) -> x y^T == 0 exactly."""
    h = k // 2
    x = torch.zeros(mx, k)
    y = torch.zeros(my, k)
    x[:, h:] = torch.randint(lo, hi + 1, (mx, k - h), generator=gen).float()
    y[:, :h] = torch.randint(lo, hi + 1, (my, h), generator=gen).float()
    return x.to(torch.bfloat16).to(device), y.to(torch.bfloat16).to(device)


def int_stats(n, ntgt, gen, device="cpu", coef=None):
    """(lse = 0, coef in {-2..2}, tgt) for n rows (or columns) whose targets index ntgt entries.  Every third target
    is -1; a few are pinned to tile edges (0, 127, 128, ntgt - 1)."""
    c = torch.randint(-2, 3, (n,), generator=gen).float() if coef is None else torch.full((n,), float(coef))
    t = torch.randint(0, ntgt, (n,), generator=gen, dtype=torch.int32)
    t[::3] = -1
    for i, v in zip((1, 2, 4, 5), (0, ntgt - 1, 127, 128)):
        if i < n:
            t[i] = min(v, ntgt - 1)
    return torch.zeros(n, device=device), c.to(device), t.to(device)


def ntxent_stats(ra, rb, off, coef, device):
    """Row / column statistics exactly as pgica_ntxent_coef builds them (positives at (i, i + off)), lse = 0."""
    rows = torch.arange(ra, device=device)
    cols = torch.arange(rb, device=device) - off
    ctgt = torch.where((cols >= 0) & (cols < ra), cols, torch.full_like(cols, -1))
    return ((torch.zeros(ra, device=device), torch.full((ra,), float(coef), device=device), (rows + off).int()),
            (torch.zeros(rb, device=device), torch.full((rb,), float(coef), device=device), ctgt.int()))


def swap(row, col):
    return col, row


# ================================================================================================ references
def closed_form(x, y, row=None, col=None):
    """out = G y for z == 0, lse == 0 (every exponential 1): O((mx + my) k) fp64 work, exact for integer data.

        row term: out_i += r_coef_i (sum_j y_j - y_{r_tgt_i})
        col term: out_i += sum_j c_coef_j y_j - sum_{j : c_tgt_j == i} c_coef_j y_j
    """
    X, Y = x.double(), y.double()
    out = torch.zeros_like(X)
    if row is not None:
        _, rc, rt = row
        rt = rt.long()
        v = rt >= 0
        yt = torch.zeros_like(X)
        yt[v] = Y[rt[v]]
        out += rc.double()[:, None] * (Y.sum(0)[None, :] - yt)
    if col is not None:
        _, cc, ct = col
        ct = ct.long()
        cy = cc.double()[:, None] * Y
        out += cy.sum(0)[None, :]
        v = ct >= 0
        out.index_add_(0, ct[v], -cy[v])
    return out


def g_block(x, y, scale, row, col, ri, cj, parts=False):
    """fp64 G on rows ri x columns cj, straight from the definition in pgica.h.  parts=True also returns
    E = |r_coef| P_row + |c_coef| P_col, the exponential part (what an error of the exponentials scales with)."""
    z = scale * (x[ri].double() @ y[cj].double().T)
    g = torch.zeros_like(z)
    e = torch.zeros_like(z)
    if row is not None:
        lse, coef, tgt = (t[ri] for t in row)
        p = torch.exp(z - lse.double()[:, None])
        g += coef.double()[:, None] * (p - (tgt.long()[:, None] == cj[None, :]).double())
        e += coef.double().abs()[:, None] * p
    if col is not None:
        lse, coef, tgt = (t[cj] for t in col)
        p = torch.exp(z - lse.double()[None, :])
        g += coef.double()[None, :] * (p - (tgt.long()[None, :] == ri[:, None]).double())
        e += coef.double().abs()[None, :] * p
    return (g, e) if parts else g


def dense_reference(x, y, scale, row, col):
    """(G y, G^T x) with G materialised in fp64 (small problems only)."""
    ri = torch.arange(x.shape[0], device=x.device)
    cj = torch.arange(y.shape[0], device=x.device)
    g = g_block(x, y, scale, row, col, ri, cj)
    return g @ y.double(), g.T @ x.double()


# ================================================================================================ planted faults
def planted_faults(x, y, scale, row, col):
    """The faults every check must see, as a change dG of G on a block: [(name, ri, cj, dG)].

    tile_dropped / tile_twice: the 128 x 128 tile holding the target of a scored row (or column), removed or added
    once more; onehot_moved: that row's target one-hot on the neighbouring column; lse_ln2: that row's lse
    (column term only: that column's lse) too large by ln 2, i.e. its exponentials halved."""
    dev = x.device
    mx, my = x.shape[0], y.shape[0]
    stats = row if row is not None else col
    _, coef, tgt = stats
    cand = torch.nonzero((coef != 0) & (tgt >= 0)).flatten()
    assert cand.numel() > 0, "degenerate statistics: no scored row with a target"
    i = int(cand[cand.numel() // 2])
    t = int(tgt[i])
    c = float(coef[i])
    if row is not None:
        fi, fj = i, t
    else:
        fi, fj = t, i
    t2 = t + 1 if t + 1 < (my if row is not None else mx) else t - 1
    ri = torch.arange((fi // TILE) * TILE, min(mx, (fi // TILE + 1) * TILE), device=dev)
    cj = torch.arange((fj // TILE) * TILE, min(my, (fj // TILE + 1) * TILE), device=dev)
    tile = g_block(x, y, scale, row, col, ri, cj)
    faults = [("tile_dropped", ri, cj, -tile), ("tile_twice", ri, cj, tile)]
    move = torch.tensor([[c, -c]], dtype=torch.float64, device=dev)
    if row is not None:
        faults.append(("onehot_moved", torch.tensor([i], device=dev), torch.tensor([t, t2], device=dev), move))
        ri1, cj1 = torch.tensor([i], device=dev), torch.arange(my, device=dev)
        z = scale * (x[ri1].double() @ y.double().T)
        dg = -0.5 * c * torch.exp(z - float(row[0][i]))
    else:
        faults.append(("onehot_moved", torch.tensor([t, t2], device=dev), torch.tensor([i], device=dev), move.T))
        ri1, cj1 = torch.arange(mx, device=dev), torch.tensor([i], device=dev)
        z = scale * (x.double() @ y[cj1].double().T)
        dg = -0.5 * c * torch.exp(z - float(col[0][i]))
    faults.append(("lse_ln2", ri1, cj1, dg))
    return faults


def fault_deltas(fault, x, y):
    """-> ((rows of out_x, change), (rows of out_y, change)) of one planted fault."""
    _, ri, cj, dg = fault
    return (ri, dg @ y[cj].double()), (cj, dg.T @ x[ri].double())


# ================================================================================================ checkers
def exact_ok(out, ref):
    """Bit-exact: fp32 outputs equal the exact values; bf16 outputs equal their round-to-nearest."""
    if out.dtype == torch.bfloat16:
        return torch.equal(out, ref.float().to(torch.bfloat16))
    return torch.equal(out.double(), ref)


def assert_exact_and_sensitive(outs, refs, faults, x, y, what):
    """outs / refs: (out_x, out_y) with None where a product is not computed.  The kernel equals the closed form bit for
    bit, and the same comparison rejects each planted fault."""
    for o, r, side in zip(outs, refs, ("x", "y")):
        if o is None:
            continue
        assert exact_ok(o, r), (what, side, float((o.double() - r).abs().max()),
                                int(((o.double() - r) != 0).any(1).sum()))
    for f in faults:
        deltas = fault_deltas(f, x, y)
        rejected = False
        for o, r, (rows, d) in zip(outs, refs, deltas):
            if o is not None and not exact_ok(o[rows], r[rows] + d):
                rejected = True
        assert rejected, (what, f[0], "planted fault not rejected")


def row_bound(g_abs_ynorm, flip_ynorm, e_ynorm, n_terms, eps_p, kappa=4.0):
    """Per-row bound on ||out_i - ref_i||_2 for out = G y computed as the kernels do, ref = bf16(G) y in fp64.

    The kernel forms G~_ij = coef (P~_ij - onehot) in fp32 from approximate exponentials, rounds it to bf16 (round to
    nearest) and accumulates bf16(G~) y in fp32 on the tensor cores.  The reference keeps that rounding of G (it is
    part of what the kernel defines) but takes G in fp64.  Three error terms; only the statistical one (C) carries a
    safety factor kappa = 4, the other two are worst-case sums:

    * rounding flips.  |G~_ij - G_ij| <= d_ij := eps_p E_ij + 2^-23 |G_ij| (the exponentials' error below, the fp32
      rounding of G~).  bf16(G~_ij) differs from bf16(G_ij) only if a rounding midpoint lies within d_ij of G_ij, and
      then by one bf16 spacing s_ij.  Summed without any independence assumption (rows of an adversarial batch round
      alike):
          A_i = sum_j s_ij [dist(G_ij, midpoint) <= d_ij] ||y_j||.
      (A coarser 2^-9 ||(G^2 . Y^2)_i||^(1/2) against an unrounded reference was tried first.  It is wrong for this
      purpose: in a flat softmax the target element G_it ~ -coef dominates it and hides an lse error of a whole row,
      and it assumes the roundings of different j are independent, which mixed-sign groups of near-equal rows break.)
    * the exponentials: P~ = P (1 + d), |d| <= eps_p (ex2.approx, the fp32 rounding of the argument z c - lse log2 e,
      the fp32 accumulation of z over k, and the error of the lse the backward is given, see the callers):
          B_i = eps_p sum_j E_ij ||y_j||,   E = |coef| P   (the absolute exp-approximation term; kept as a margin,
      since without a flip the exponentials' error is absorbed by the rounding to bf16).
    * fp32 accumulation of the n_terms products on the tensor cores: at most n_terms / 16 + 1 roundings of partial
      sums bounded by sum_j |G_ij| |y_jc|, each <= 2^-23 of it, independent:
          C_i = 2^-23 sqrt(n_terms / 16 + 1) sum_j |G_ij| ||y_j||.
    bound_i = A_i + B_i + kappa C_i.
    """
    return flip_ynorm + eps_p * e_ynorm + kappa * 2.0 ** -23 * math.sqrt(n_terms / 16 + 1) * g_abs_ynorm


def bf16_flips(g, d):
    """s_ij [dist(G_ij, nearest bf16 rounding midpoint) <= d_ij]: the change of bf16(G) a perturbation <= d can make."""
    g32 = g.float()
    gb = g32.bfloat16().double()
    _, e = torch.frexp(g32)
    s = torch.ldexp(torch.ones_like(g), (e - 8).to(torch.int32))          # bf16 spacing at |G| (8 significant bits)
    near = ((gb - g).abs() - s / 2).abs() <= d + (g32.double() - g).abs()
    return gb, s * near


def rows_within(out, ref, bound):
    """-> (all rows within their bound, largest error / bound)"""
    err = (out.double() - ref).norm(dim=1)
    ratio = err / bound.clamp_min(1e-300)
    return bool((ratio <= 1.0).all()), float(ratio.max())


class Reference:
    """bf16(G) y and bf16(G)^T x in fp64 and the per-row bounds (row_bound) of both, G materialised a block of rows at a
    time."""

    def __init__(self, x, y, scale, row, col, eps_p, chunk=2048):
        X, Y = x.double(), y.double()
        yn, xn = Y.norm(dim=1), X.norm(dim=1)
        self.out_x = torch.empty_like(X)
        self.out_y = torch.zeros_like(Y)
        bx = [torch.empty(x.shape[0], dtype=torch.float64, device=x.device) for _ in range(3)]
        by = [torch.zeros(y.shape[0], dtype=torch.float64, device=x.device) for _ in range(3)]
        cj = torch.arange(y.shape[0], device=x.device)
        for r0 in range(0, x.shape[0], chunk):
            ri = torch.arange(r0, min(x.shape[0], r0 + chunk), device=x.device)
            g, e = g_block(x, y, scale, row, col, ri, cj, parts=True)
            ga = g.abs()
            gb, flip = bf16_flips(g, eps_p * e + 2.0 ** -23 * ga)
            self.out_x[ri] = gb @ Y
            self.out_y += gb.T @ X[ri]
            for dst, v in zip(bx, (ga @ yn, flip @ yn, e @ yn)):
                dst[ri] = v
            for dst, v in zip(by, (ga.T @ xn[ri], flip.T @ xn[ri], e.T @ xn[ri])):
                dst += v
            del g, e, ga, gb, flip
        self.bounds = (row_bound(*bx, y.shape[0], eps_p), row_bound(*by, x.shape[0], eps_p))


def assert_bounded_and_sensitive(outs, ref, bounds, faults, x, y, what, report):
    """Every row within its bound; each planted fault puts some row outside it (its largest error / bound reported as
    the margin by which the check sees the fault)."""
    for o, r, b, side in zip(outs, (ref.out_x, ref.out_y), bounds, ("x", "y")):
        ok, worst = rows_within(o, r, b)
        report(f"{what} out_{side}", worst)
        assert ok, (what, side, worst)
    for f in faults:
        seen = max(rows_within(o[rows], r[rows] + d, b[rows])[1]
                   for o, r, b, (rows, d) in zip(outs, (ref.out_x, ref.out_y), bounds, fault_deltas(f, x, y)))
        print(f"[fault error/bound] {what} {f[0]}: {seen:.3g}")
        assert seen > 1.0, (what, f[0], "planted fault not rejected")


def ulps(v, n):
    """n fp32 ulps of max(1, |v|) (2^-23 relative: never smaller than the true ulp)."""
    return n * 2.0 ** -23 * v.double().abs().clamp_min(1.0)


def within(got, ref, tol):
    """-> (every entry within its tolerance, largest error / tolerance)"""
    ratio = (got.double() - ref).abs() / tol
    return bool((ratio <= 1.0).all()), float(ratio.max())


# ================================================================================================ CPU tests
@pytest.mark.parametrize("mx,my,k", [(300, 270, 64), (129, 1000, 512), (5, 7, 16)])
def test_builders_give_zero_logits(mx, my, k):
    """The exact tests rest on x y^T == 0 in bf16 and on integer entries that bf16 holds exactly."""
    gen = torch.Generator().manual_seed(mx + my)
    x, y = int_operands(mx, my, k, gen)
    assert torch.equal(x.double() @ y.double().T, torch.zeros(mx, my, dtype=torch.float64))
    for t in (x, y):
        assert torch.equal(t.double(), t.double().round()) and float(t.double().abs().max()) <= 3
        assert int((t != 0).sum()) > t.numel() // 4                         # not degenerate
    _, coef, tgt = int_stats(mx, my, gen)
    assert bool(((coef >= -2) & (coef <= 2)).all()) and int((coef != 0).sum()) > 0
    assert bool((tgt == -1).any()) and bool(((tgt >= -1) & (tgt < my)).all())


@pytest.mark.parametrize("mode", ["row", "col", "both", "ntxent"])
@pytest.mark.parametrize("mx,my,k", [(300, 270, 64), (129, 391, 32), (1, 130, 16)])
def test_closed_form_equals_dense_fp64(mode, mx, my, k):
    """The O((mx + my) k) closed form equals G y and G^T x with G materialised in fp64, on ragged shapes."""
    gen = torch.Generator().manual_seed(7 * mx + my)
    if mode == "ntxent":                                   # positives (i, i + off) need rows_a <= rows_b
        mx, my = min(mx, my), max(mx, my)
    x, y = int_operands(mx, my, k, gen)
    if mode == "ntxent":
        row, col = ntxent_stats(mx, my, (my - mx) // 2, 2.0 ** -13, "cpu")
    else:
        row = int_stats(mx, my, gen) if mode in ("row", "both") else None
        col = int_stats(my, mx, gen) if mode in ("col", "both") else None
    ox, oy = closed_form(x, y, row, col), closed_form(y, x, *swap(row, col))
    dx, dy = dense_reference(x, y, 1.0, row, col)
    assert torch.equal(ox, dx) and torch.equal(oy, dy)
    assert float(ox.abs().max()) > 0 and float(oy.abs().max()) > 0


@pytest.mark.parametrize("mode", ["row", "col", "both"])
def test_exact_checker_rejects_planted_faults(mode):
    """The bit-exact comparison accepts the closed form and rejects each planted fault (CPU-sized problem)."""
    gen = torch.Generator().manual_seed(11)
    mx, my, k = 300, 700, 64
    x, y = int_operands(mx, my, k, gen)
    row = int_stats(mx, my, gen) if mode in ("row", "both") else None
    col = int_stats(my, mx, gen) if mode in ("col", "both") else None
    refs = (closed_form(x, y, row, col), closed_form(y, x, *swap(row, col)))
    outs = tuple(r.float() for r in refs)
    faults = planted_faults(x, y, 1.0, row, col)
    assert [f[0] for f in faults] == ["tile_dropped", "tile_twice", "onehot_moved", "lse_ln2"]
    assert_exact_and_sensitive(outs, refs, faults, x, y, mode)
    # and on each side alone, when only one product is computed
    assert_exact_and_sensitive((outs[0], None), refs, faults, x, y, mode)
    # a kernel output with one tile lost fails the comparison
    bad = refs[0].clone()
    (rows, d), _ = fault_deltas(faults[0], x, y)
    bad[rows] += d
    assert not exact_ok(bad.float(), refs[0])


@pytest.mark.parametrize("peaked", [False, True])
def test_row_bound_accepts_emulation_and_rejects_faults(peaked):
    """The per-row bound holds for an fp32 emulation of the kernel (bf16 G, approximate exponentials, fp32 sums) and
    rejects every planted fault, on a CPU-sized softmax-gradient problem with flat or peaked rows."""
    gen = torch.Generator().manual_seed(5 + peaked)
    mx, my, k = 256, 1500, 128
    x = torch.randn(mx, k, generator=gen).bfloat16()
    y = (torch.randn(my, k, generator=gen) * 0.1).bfloat16()
    tgt = torch.randint(0, my, (mx,), generator=gen, dtype=torch.int32)
    if peaked:
        x = (x.float() + 30 * y.float()[tgt.long()]).bfloat16()
    z = x.double() @ y.double().T
    lse = torch.logsumexp(z, 1)
    coef = torch.randn(mx, generator=gen)
    tgt[::7] = -1
    row = (lse.float(), coef, tgt)
    eps_p = 2.0 ** -20
    ref = Reference(x, y, 1.0, row, None, eps_p, chunk=100)
    bounds = ref.bounds
    # emulation: exponentials with a relative error of eps_p / 2, G rounded to bf16, fp32 products
    ri, cj = torch.arange(mx), torch.arange(my)
    g = g_block(x, y, 1.0, row, None, ri, cj)
    noise = (torch.rand(mx, my, generator=gen, dtype=torch.float64) - 0.5) * eps_p
    gb = (g + coef.double()[:, None] * torch.exp(z - lse[:, None]) * noise).float().bfloat16().float()
    outs = (gb @ y.float(), gb.T @ x.float())
    assert_bounded_and_sensitive(outs, ref, bounds, planted_faults(x, y, 1.0, row, None), x, y, "emulation",
                                 lambda *a: None)
    # a row lse off by ln 2 is outside the forward tolerance as well
    assert not within(lse + LN2 * (ri == 3), lse, ulps(lse, 16))[0]


# ================================================================================================ GPU tests
@pytest.fixture(scope="module")
def pg(cuda_device):
    import preference_guided_image_captioning_alignment_b200 as pkg
    from preference_guided_image_captioning_alignment_b200 import _lib
    lib = _lib.load()
    assert lib.pgica_device_check() == 0, lib.pgica_last_error()
    return pkg


@pytest.fixture(autouse=True)
def _reset_library_options():
    yield
    try:
        from preference_guided_image_captioning_alignment_b200 import _lib
        for name, value in (("sggf_plan_r2", 0), ("sggf_plan_c2", 0), ("sgg_fused", 1), ("sgg_cluster", 0),
                            ("sggf_col_groups", 1)):
            _lib.set_option(name, value)
    except Exception:
        pass


def set_plan(plan):
    from preference_guided_image_captioning_alignment_b200 import _lib
    r2, c2 = (int(v) for v in plan.split(",")) if plan else (0, 0)
    _lib.set_option("sggf_plan_r2", r2)
    _lib.set_option("sggf_plan_c2", c2)


def report(what, worst):
    print(f"[worst error/bound] {what}: {worst:.3g}")


def card():
    """Card name and power limit, printed beside the ratios."""
    import subprocess
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = "?"
    return f"{name}, power limit {out}"


# ------------------------------------------------------------------------------------------------ 1. exact backward
SGG_SHAPES = [(128, 128, 256, "row"), (77, 90, 64, "col"), (300, 1000, 512, "both"), (200, 333, 1024, "row"),
              (128 * 37 + 5, 700, 1024, "col"), (520, 128 * 9 + 1, 1024, "both"), (4500, 260, 512, "row"),
              (333, 777, 1536, "both"), (640, 1500, 1024, "row")]


@pytest.mark.gpu
@pytest.mark.parametrize("mx,my,k,mode", SGG_SHAPES)
def test_softmax_grad_gemm_exact(pg, cuda_device, mx, my, k, mode):
    """pgica_softmax_grad_gemm with exact G: the cluster kernel (L2 exchange ring), the single-CTA kernel
    (sgg_cluster = 1) and, for k = 1536 or k < 512, the path for k not a multiple of 512; fp32 and bf16 outputs."""
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(mx * 3 + my)
    x, y = int_operands(mx, my, k, gen, cuda_device)
    row = int_stats(mx, my, gen, cuda_device) if mode in ("row", "both") else None
    col = int_stats(my, mx, gen, cuda_device) if mode in ("col", "both") else None
    ref = closed_form(x, y, row, col)
    faults = planted_faults(x, y, 1.0, row, col)
    for cluster in (0, 1):
        _lib.set_option("sgg_cluster", cluster)
        out = F.softmax_grad_gemm(x, y, 1.0, row=row, col=col)
        assert_exact_and_sensitive((out, None), (ref, None), faults, x, y, f"sgg cluster={cluster}")
        ob = F.softmax_grad_gemm(x, y, 1.0, row=row, col=col, out_dtype=torch.bfloat16)
        assert exact_ok(ob, ref), ("bf16", cluster)


DUAL_CASES = [(128, 128, 512, "row", None), (300, 1000, 512, "both", None), (200, 333, 1024, "row", None),
              (128 * 5 + 7, 128 * 9 + 1, 1024, "row", "2,4"), (128 * 7, 128 * 6, 512, "both", "3,2"),
              (128 * 2, 128 * 11, 1024, "col", "4,6"), (2048, 5003, 1024, "row", None),
              (128 * 6 + 1, 128 * 10 + 1, 2048, "both", "2,3"), (129, 5003, 1536, "both", "1,2"),
              (1000, 3001, 1024, "both", "2,2")]


@pytest.mark.gpu
@pytest.mark.parametrize("mx,my,k,mode,plan", DUAL_CASES)
def test_softmax_grad_gemm_dual_exact(pg, cuda_device, mx, my, k, mode, plan):
    """pgica_softmax_grad_gemm_dual with exact G, both products: the planner's split and pinned plans that force
    several chunks (OutY accumulated in place over chunks), k from 512 to 2048, one-row and one-column tails."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(mx * 5 + my)
    x, y = int_operands(mx, my, k, gen, cuda_device)
    row = int_stats(mx, my, gen, cuda_device) if mode in ("row", "both") else None
    col = int_stats(my, mx, gen, cuda_device) if mode in ("col", "both") else None
    refs = (closed_form(x, y, row, col), closed_form(y, x, *swap(row, col)))
    faults = planted_faults(x, y, 1.0, row, col)
    set_plan(plan)
    outs = F.softmax_grad_gemm_dual(x, y, 1.0, row=row, col=col)
    assert_exact_and_sensitive(outs, refs, faults, x, y, f"dual plan={plan}")
    bx, oy = F.softmax_grad_gemm_dual(x, y, 1.0, row=row, col=col, out_x_dtype=torch.bfloat16)
    assert exact_ok(bx, refs[0]) and exact_ok(oy, refs[1])


@pytest.mark.gpu
@pytest.mark.parametrize("mx,my,k", [(100, 5003, 1024), (470, 50257, 1024), (300, 3000, 512), (513, 9000, 1536),
                                     (257, 20001, 2048)])
def test_dual_column_groups_exact(pg, cuda_device, mx, my, k):
    """Column groups (partial OutX add-reduced into zeros) for sggf_col_groups in {0, 1, 2, 5}: bit-exact each time;
    rows of the OutX allocation past mx are left untouched."""
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(mx + 13 * my)
    x, y = int_operands(mx, my, k, gen, cuda_device)
    row = int_stats(mx, my, gen, cuda_device)
    refs = (closed_form(x, y, row, None), closed_form(y, x, None, row))
    faults = planted_faults(x, y, 1.0, row, None)
    lib = _lib.load()
    pad = 200
    for groups in (0, 1, 2, 5):
        _lib.set_option("sggf_col_groups", groups)
        out_x = torch.full((mx + pad, k), 7.0, device=cuda_device)
        out_y = torch.empty(my, k, device=cuda_device)
        need = ctypes.c_size_t(0)
        _lib.check(lib.pgica_softmax_grad_gemm_dual_workspace_bytes(mx, my, k, ctypes.byref(need)))
        ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=cuda_device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        _lib.check(lib.pgica_softmax_grad_gemm_dual(p(x), p(y), mx, my, k, 1.0, p(row[0]), p(row[1]), p(row[2]), None,
                                                    None, None, p(out_x), 0, p(out_y), 0, p(ws), need.value,
                                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        assert_exact_and_sensitive((out_x[:mx], out_y), refs, faults, x, y, f"col_groups={groups}")
        assert bool((out_x[mx:] == 7.0).all()), ("rows past mx written", groups)


def lmhead_int_inputs(nseq, T, d, V, seed, device):
    """Integer hidden / weight with disjoint supports, labels with tile-edge values, a 0/1 mask, integer grad_seq."""
    gen = torch.Generator().manual_seed(seed)
    h, W = int_operands(nseq * T, V, d, gen, device)
    labels = torch.randint(0, V, (nseq, T), generator=gen)
    edge = torch.tensor([0, 127, 128, 255, 256, V - 1])
    labels[:, 1:1 + edge.numel()] = edge
    lens = torch.randint(T // 2, T + 1, (nseq,), generator=gen)
    mask = (torch.arange(T)[None, :] < lens[:, None]).long()
    gseq = torch.randint(-2, 3, (nseq,), generator=gen).float()
    gseq[gseq == 0] = 1.0
    return h.view(nseq, T, d), W, labels.to(device), mask.to(device), gseq.to(device)


def lmhead_row_stats(labels, mask, gseq):
    """What prep_rows + row_coef(sign = -1) must produce, restated: row r = (b, t) has label[b, t + 1] and weight
    mask[b, t + 1]; the last position of every sequence has label -1, weight 0; ncoef = -grad_seq[b] * weight.
    (Labels are in the vocabulary here.)"""
    nseq, T = labels.shape
    tgt = torch.cat([labels[:, 1:], torch.full((nseq, 1), -1, device=labels.device, dtype=labels.dtype)], 1)
    w = torch.cat([mask[:, 1:].double(), torch.zeros(nseq, 1, device=labels.device, dtype=torch.float64)], 1)
    tgt = tgt.reshape(-1).int()                       # labels of masked rows are kept; their coefficient is 0
    ncoef = (-gseq.double()[:, None] * w).reshape(-1)
    return torch.zeros(nseq * T, device=labels.device), ncoef, tgt


@pytest.mark.gpu
@pytest.mark.parametrize("nseq,T,plan", [(32, 128, None), (32, 128, "8,11"), (32, 128, "16,9"), (64, 512, None)])
def test_lmhead_backward_chain_exact(pg, cuda_device, nseq, T, plan):
    """The whole LM-head backward (prep_rows -> row_coef -> dual kernel) at the benchmarked shapes: cfg2 (4096 x 50257
    x 1024) with the planner's split and pinned splits, and one rank's cfg4 slice (32768 rows, 8 chunks, dW
    accumulated in place).  lse = 0 and integer operands: dH and dW are bit-exact."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    d, V = 1024, 50257
    h, W, labels, mask, gseq = lmhead_int_inputs(nseq, T, d, V, nseq * T, cuda_device)
    rl, rw = F.prep_rows(labels, mask, V)
    row = lmhead_row_stats(labels, mask, gseq)
    assert torch.equal(rl, row[2]) and torch.equal(rw.double(), -row[1] / gseq.double().repeat_interleave(T))
    hf = h.reshape(-1, d)
    refs = (closed_form(hf, W, row, None), closed_form(W, hf, None, row))
    faults = planted_faults(hf, W, 1.0, row, None)
    set_plan(plan)
    zero = torch.zeros(nseq * T, device=cuda_device)
    dh, dw = F.lmhead_logprob_bwd(h, W, rl, rw, zero, gseq, False, dhidden_dtype=torch.float32)
    assert_exact_and_sensitive((dh.reshape(-1, d), dw), refs, faults, hf, W, f"lmhead plan={plan}")
    if nseq * T <= 4096:
        dhb, _ = F.lmhead_logprob_bwd(h, W, rl, rw, zero, gseq, False, dhidden_dtype=torch.bfloat16)
        assert exact_ok(dhb.reshape(-1, d), refs[0])


@pytest.mark.gpu
def test_lmhead_backward_progress_exact(pg, cuda_device):
    """pgica_lmhead_logprob_bwd_progress beside pgica_peer_allreduce_progress at world = 1, three epochs on the same
    counters: dW and dH bit-exact every time."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    nseq, T, d, V, rows_per_seg = 32, 128, 1024, 50257, 6400
    h, W, labels, mask, gseq = lmhead_int_inputs(nseq, T, d, V, 99, cuda_device)
    rl, rw = F.prep_rows(labels, mask, V)
    row = lmhead_row_stats(labels, mask, gseq)
    hf = h.reshape(-1, d)
    refs = (closed_form(hf, W, row, None), closed_form(W, hf, None, row))
    faults = planted_faults(hf, W, 1.0, row, None)
    zero = torch.zeros(nseq * T, device=cuda_device)
    pairs = (V + 255) // 256
    rows = pairs * 256
    nseg = (rows + rows_per_seg - 1) // rows_per_seg
    buf = torch.zeros(rows * d + 64 * (nseg + 1), dtype=torch.float32, device=cuda_device)
    dw = buf[: V * d].view(V, d)
    progress = torch.zeros(nseg, dtype=torch.int32, device=cuda_device)
    local_sync = torch.zeros(2, dtype=torch.int32, device=cuda_device)
    seg_begin = [min(s * rows_per_seg, rows) * d for s in range(nseg + 1)]
    seg_pairs = [(min((s + 1) * rows_per_seg, rows) - s * rows_per_seg) // 256 for s in range(nseg)]
    side = torch.cuda.Stream(device=cuda_device)
    for epoch in (1, 2, 3):
        dw.zero_()
        torch.cuda.synchronize()
        dh, inc = F.lmhead_logprob_bwd_progress(h, W, rl, rw, zero, gseq, dw, progress, rows_per_seg, False,
                                                dhidden_dtype=torch.float32)
        targets = [epoch * inc * n for n in seg_pairs]
        F.peer_allreduce_progress([buf.data_ptr()], [buf.data_ptr() + 4 * rows * d], 0, progress, targets, seg_begin,
                                  epoch, local_sync, 0, stream=side)
        side.synchronize()
        torch.cuda.synchronize()
        assert progress.tolist() == targets
        assert_exact_and_sensitive((dh.reshape(-1, d), dw), refs, faults, hf, W, f"progress epoch {epoch}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 1, 129, 700])
def test_lmhead_rows_bwd_compacted_exact(pg, cuda_device, n):
    """pgica_lmhead_rows_bwd on compacted rows (few row blocks: the X-holders share each sweep over the vocabulary in
    column groups) for sggf_col_groups in {0, 1, 2, 5}: dH and dW bit-exact."""
    from preference_guided_image_captioning_alignment_b200 import _lib
    d, V = 1024, 50257
    gen = torch.Generator().manual_seed(n)
    hc, W = int_operands(n, V, d, gen, cuda_device)
    row = int_stats(n, V, gen, cuda_device)
    if n == 1:
        row[1].fill_(-2.0)
        row[2].fill_(V - 1)
    refs = (closed_form(hc, W, row, None), closed_form(W, hc, None, row))
    faults = planted_faults(hc, W, 1.0, row, None)
    lib = _lib.load()
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_lmhead_rows_workspace_bytes(n, d, V, ctypes.byref(need)))
    ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=cuda_device)
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    for groups in (0, 1, 2, 5):
        _lib.set_option("sggf_col_groups", groups)
        dh = torch.empty(n, d, device=cuda_device)
        dw = torch.empty(V, d, device=cuda_device)
        _lib.check(lib.pgica_lmhead_rows_bwd(p(hc), p(W), p(row[2]), p(row[0]), p(row[1]), n, d, V, p(dh), 0, p(dw), 0,
                                             p(ws), ws.numel(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        assert_exact_and_sensitive((dh, dw), refs, faults, hc, W, f"rows_bwd col_groups={groups}")


@pytest.mark.gpu
@pytest.mark.parametrize("ra,rb,off", [(16384, 16384, 0), (4096, 32768, 0), (4096, 32768, 3 * 4096), (300, 1000, 200)])
def test_ntxent_backward_two_exponentials_exact(pg, cuda_device, ra, rb, off):
    """pgica_ntxent_bwd (two exponentials per element) at the benchmarked sizes: inv_tau = 2, grad = 1 and a
    power-of-two grad_mult, so every coefficient is a power of two and dA, dB are exact."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    D, inv_tau, mult = 512, 2.0, 2.0 ** -15
    gen = torch.Generator().manual_seed(ra + rb + off)
    a, b = int_operands(ra, rb, D, gen, cuda_device)
    row, col = ntxent_stats(ra, rb, off, mult * inv_tau, cuda_device)
    refs = (closed_form(a, b, row, col), closed_form(b, a, col, row))
    faults = planted_faults(a, b, inv_tau, row, col)
    one = torch.ones((), device=cuda_device)
    outs = F.ntxent_bwd(a, b, inv_tau, off, row[0], col[0], one, mult)
    assert_exact_and_sensitive(outs, refs, faults, a, b, f"ntxent_bwd {ra}x{rb}+{off}")


# ------------------------------------------------------------------------------------------------ 1. exact forward
def sparse_int_rows(n, k, nnz, gen, device):
    """bf16 rows with nnz entries in {-1, 1} at random positions: |<a_i, b_j>| <= nnz, small integer logits."""
    x = torch.zeros(n, k)
    pos = torch.argsort(torch.rand(n, k, generator=gen), dim=1)[:, :nnz]
    x.scatter_(1, pos, (torch.randint(0, 2, (n, nnz), generator=gen) * 2 - 1).float())
    return x.to(torch.bfloat16).to(device)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,k", [(300, 1000, 512), (129, 257, 64), (513, 5003, 1024), (128, 128, 2048),
                                         (1, 33, 8)])
def test_similarity_integer_exact(pg, cuda_device, rows, cols, k):
    """pgica_similarity reproduces the integer product bit for bit in every tile, ragged tails included."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(rows * cols)
    a = torch.randint(-3, 4, (rows, k), generator=gen).bfloat16().to(cuda_device)
    b = torch.randint(-3, 4, (cols, k), generator=gen).bfloat16().to(cuda_device)
    ref = a.double() @ b.double().T
    sim = F.similarity(a, b, 1.0)
    assert torch.equal(sim.double(), ref)
    for i0, j0 in ((0, 0), (rows // 2, cols // 2), (rows - 1, cols - 1)):   # a tile's worth off must be seen
        bad = ref.clone()
        bad[(i0 // TILE) * TILE:(i0 // TILE + 1) * TILE, (j0 // TILE) * TILE:(j0 // TILE + 1) * TILE] = 0
        assert not torch.equal(sim.double(), bad)


def lse_faults(z, lse, i, dim=1):
    """Planted forward faults on row i of logits z (dim = 0: column i): a 32-wide chunk dropped, lse off by ln 2."""
    zi = z[i] if dim == 1 else z[:, i]
    c0 = (zi.numel() // 2 // 32) * 32
    dropped = torch.logsumexp(torch.cat([zi[:c0], zi[c0 + 32:]]), 0)
    return {"chunk_dropped": dropped, "lse_ln2": lse[i] + LN2}


@pytest.mark.gpu
@pytest.mark.parametrize("nseq,T,d,V", [(4, 100, 1024, 50257), (32, 128, 1024, 50257), (3, 17, 512, 1000)])
def test_lmhead_forward_integer_logits(pg, cuda_device, nseq, T, d, V):
    """gemm_lse through lmhead_logprob_fwd on integer logits: ztgt bit-exact for labels 0, 127, 128, 255, 256, V - 1,
    and 0 for -1 and >= V; lse per row within 16 fp32 ulps of max(1, |lse|) of fp64 (exact z: the error is the fp32
    sum of about V / 32 chunk partials and ex2.approx, a few ulps); a dropped 32-column chunk (about 32 / V) and an
    lse off by ln 2 are both rejected."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(V + T)
    h = sparse_int_rows(nseq * T, d, 64, gen, cuda_device)
    W = sparse_int_rows(V, d, 64, gen, cuda_device)
    labels = torch.randint(0, V, (nseq, T), generator=gen)
    special = torch.tensor([0, 127, 128, 255, 256, V - 1, -1, V, V + 5])
    labels[0, 1:1 + special.numel()] = special
    labels = labels.to(cuda_device)
    _, lse, ztgt, rl, _, _ = F.lmhead_logprob_fwd(h.view(nseq, T, d), W, labels, None, False)
    z = h.double() @ W.double().T
    lse_ref = torch.logsumexp(z, 1)
    tgt = torch.cat([labels[:, 1:], torch.full((nseq, 1), -1, device=cuda_device)], 1).reshape(-1)
    valid = (tgt >= 0) & (tgt < V)
    zt = torch.where(valid, z.gather(1, tgt.clamp(0, V - 1)[:, None]).squeeze(1), torch.zeros_like(lse_ref))
    assert torch.equal(ztgt.double(), zt)
    assert bool((ztgt[6:9] == 0).all())                              # rows scoring labels -1, V, V + 5
    moved = (tgt + 1) % V
    zt_moved = torch.where(valid, z.gather(1, moved.clamp(0, V - 1)[:, None]).squeeze(1), torch.zeros_like(lse_ref))
    assert not torch.equal(ztgt.double(), zt_moved)                  # a target one-hot on the next column is seen
    tol = ulps(lse_ref, 16)
    ok, worst = within(lse, lse_ref, tol)
    report(f"lmhead fwd lse {nseq}x{T}x{V}", worst)
    assert ok
    i = int(torch.nonzero(valid).flatten()[0])
    for name, v in lse_faults(z, lse_ref, i).items():
        assert not within(lse[i:i + 1], v.reshape(1), tol[i:i + 1])[0], name


@pytest.mark.gpu
@pytest.mark.parametrize("ra,rb,k,off", [(4096, 32768, 512, 8192), (300, 1000, 512, 200), (16384, 16384, 512, 0),
                                         (1000, 3001, 128, 1500)])
def test_ntxent_forward_one_pass_integer_logits(pg, cuda_device, ra, rb, k, off):
    """The one-pass rowcol forward (pgica_ntxent_fwd_bounded) on integer logits |z| <= 32 (inside its bound at
    inv_tau = 1): diag bit-exact, lse_row per row and lse_col per column within 16 fp32 ulps of fp64.  A dropped
    32-column chunk (row side) and a dropped 32-row group (column side) shift by about 32 / cols and 32 / rows."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    gen = torch.Generator().manual_seed(ra + rb + k)
    a = sparse_int_rows(ra, k, 32, gen, cuda_device)
    b = sparse_int_rows(rb, k, 32, gen, cuda_device)
    lse_row, diag, lse_col = F.ntxent_fwd(a, b, 1.0, off, bounded=True)
    z = a.double() @ b.double().T
    idx = torch.arange(ra, device=cuda_device)
    assert torch.equal(diag.double(), z[idx, idx + off])
    lr, lc = torch.logsumexp(z, 1), torch.logsumexp(z, 0)
    for got, ref, dim, name in ((lse_row, lr, 1, "lse_row"), (lse_col, lc, 0, "lse_col")):
        tol = ulps(ref, 16)
        ok, worst = within(got, ref, tol)
        report(f"ntxent fwd {name} {ra}x{rb}+{off}", worst)
        assert ok, name
        i = got.numel() // 2
        for fname, v in lse_faults(z, ref, i, dim).items():
            assert not within(got[i:i + 1], v.reshape(1), tol[i:i + 1])[0], (name, fname)


# ------------------------------------------------------------------------------------------------ 2. fp64 bounds
def unit_rows(x):
    return torch.nn.functional.normalize(x.float(), dim=-1).bfloat16()


def ntxent_ref_stats(a, b, inv_tau, off):
    z = inv_tau * (a.double() @ b.double().T)
    idx = torch.arange(a.shape[0], device=a.device)
    out = torch.logsumexp(z, 1), z[idx, idx + off], torch.logsumexp(z, 0)
    del z
    return out


def dot_err(k, scale, xn_max, yn_max):
    """Bound on |z~ - z| for one fp32 tensor-core dot product over k: (k/16 + 1) roundings of partial sums bounded by
    sum |x||y| <= ||x|| ||y|| (Cauchy-Schwarz), each <= 2^-23 of it; times the logit scale."""
    return scale * (k / 16 + 1) * 2.0 ** -23 * xn_max * yn_max


def check_ntxent_bounded(a, b, inv_tau, off, what, grad=1.0, mult=None):
    """Bounded (one-pass / shared-exponential) NT-Xent forward and backward against fp64, every row and column.

    Forward: lse_row, lse_col within tol = 16 fp32 ulps of max(1, |lse|) plus the logit error dot_err (an error of
    every z shifts lse by at most as much); diag within dot_err.  Backward: dA = G B, dB = G^T A with
    G = c (P_row + P_col - onehots), c = grad * mult * inv_tau, bound per row from row_bound with
    eps_p = 3 * 2^-22 (three ex2.approx per element: the shared exponential and the two factors)
          + ln 2 * 2^-23 * 4 * (inv_tau log2 e + max |lse| log2 e) (fp32 arguments z c - c and c - lse log2 e)
          + ln 2 * log2 e * dot_err (fp32 accumulation of z)
          + max |lse - lse_fp64| of the forward outputs the backward is given (measured, after the forward passed)."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    ra, rb, k = a.shape[0], b.shape[0], a.shape[1]
    mult = mult if mult is not None else 0.5 / rb
    lse_row, diag, lse_col = F.ntxent_fwd(a, b, inv_tau, off, bounded=True)
    lr, dg, lc = ntxent_ref_stats(a, b, inv_tau, off)
    an, bn = a.double().norm(dim=1), b.double().norm(dim=1)
    dz = dot_err(k, inv_tau, float(an.max()), float(bn.max()))
    for got, ref, name in ((lse_row, lr, "lse_row"), (lse_col, lc, "lse_col")):
        tol = ulps(ref, 16) + dz
        ok, worst = within(got, ref, tol)
        report(f"{what} {name}", worst)
        assert ok, name
        i = got.numel() // 2
        assert not within(got[i:i + 1], (ref[i] + LN2).reshape(1), tol[i:i + 1])[0]
    ok, worst = within(diag, dg, torch.full_like(dg, dz))
    report(f"{what} diag", worst)
    assert ok
    gl = torch.full((1,), grad, device=a.device)
    da, db = F.ntxent_bwd(a, b, inv_tau, off, lse_row, lse_col, gl, mult, bounded=True)
    row, col = ntxent_stats(ra, rb, off, grad * mult * inv_tau, a.device)
    row, col = (lr,) + row[1:], (lc,) + col[1:]                 # the reference runs on the fp64 statistics
    lmax = float(torch.cat([lr.abs(), lc.abs()]).max())
    lse_err = float(torch.cat([lse_row.double() - lr, lse_col.double() - lc]).abs().max())
    eps_p = 3 * 2.0 ** -22 + LN2 * 2.0 ** -23 * 4 * (inv_tau + lmax) * LOG2E + dz + lse_err
    ref = Reference(a, b, inv_tau, row, col, eps_p)
    bounds = ref.bounds
    faults = planted_faults(a, b, inv_tau, row, col)
    assert_bounded_and_sensitive((da, db), ref, bounds, faults, a, b, f"{what} bwd", report)
    return lse_row, lse_col, da, db


@pytest.mark.gpu
@pytest.mark.parametrize("ra,rb,off", [(16384, 16384, 0), (4096, 32768, 0), (4096, 32768, 4096),
                                       (4096, 32768, 28672)])
def test_ntxent_bounded_benchmarked_sizes_fp64(pg, cuda_device, ra, rb, off):
    """The NT-Xent path bench.py times (bounded=True, D = 512, tau = 0.5) against fp64 at its sizes: lse_row, diag,
    lse_col, dA and dB checked per row / column."""
    print(card())
    D = 512
    g = torch.Generator().manual_seed(ra + off)
    b = unit_rows(torch.randn(rb, D, generator=g)).to(cuda_device)
    a = unit_rows(b[off:off + ra].float().cpu() + 0.7 * torch.randn(ra, D, generator=g)).to(cuda_device)
    check_ntxent_bounded(a, b, 2.0, off, f"ntxent bounded {ra}x{rb}+{off}")


def adversarial_pairs(n, D, gen):
    """Unit rows: every b_j close to one direction u; in every 32-row group of a, half the rows are +u (logits near
    +1 / tau) and half -u (near -1 / tau), so the group's shared shift is as far from half its rows as it can be."""
    u = torch.randn(D, generator=gen)
    b = unit_rows(u[None, :] + 0.15 * u.norm() / math.sqrt(D) * torch.randn(n, D, generator=gen))
    sign = torch.where(torch.arange(n) % 2 == 0, 1.0, -1.0)
    a = unit_rows(sign[:, None] * u[None, :] + 0.05 * u.norm() / math.sqrt(D) * torch.randn(n, D, generator=gen))
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("tau", [0.5, 0.07, 0.03])
def test_ntxent_bounded_adversarial_groups_fp64(pg, cuda_device, tau):
    """The shared-shift scheme at its hardest: mixed-sign rows in every 32-row group, tau from 0.5 down to 0.03."""
    g = torch.Generator().manual_seed(int(1 / tau))
    a, b = adversarial_pairs(2048, 512, g)
    check_ntxent_bounded(a.to(cuda_device), b.to(cuda_device), 1.0 / tau, 0, f"ntxent adversarial tau={tau}")


@pytest.mark.gpu
def test_ntxent_bounded_falls_back_below_tau_bound(pg, cuda_device):
    """tau = 0.0288 is outside the bounded scheme: the call takes the two-pass / two-exponential path and equals it bit
    for bit (lse_row, lse_col, dB); dA is add-reduced over column groups, so equal to rounding."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    g = torch.Generator().manual_seed(288)
    a, b = adversarial_pairs(2048, 512, g)
    a, b = a.to(cuda_device), b.to(cuda_device)
    inv_tau = 1.0 / 0.0288
    assert inv_tau * LOG2E * 2 >= 100.0
    f1 = F.ntxent_fwd(a, b, inv_tau, 0, bounded=True)
    f2 = F.ntxent_fwd(a, b, inv_tau, 0)
    assert torch.equal(f1[0], f2[0]) and torch.equal(f1[2], f2[2]) and torch.equal(f1[1], f2[1])
    gl = torch.ones(1, device=cuda_device)
    da1, db1 = F.ntxent_bwd(a, b, inv_tau, 0, f2[0], f2[2], gl, 2.0 ** -12, bounded=True)
    da2, db2 = F.ntxent_bwd(a, b, inv_tau, 0, f2[0], f2[2], gl, 2.0 ** -12)
    assert torch.equal(db1, db2)
    assert float((da1.double() - da2.double()).norm() / da2.double().norm()) < 1e-6


def gpt2_like_inputs(nseq, T, d, V, seed, device):
    """Logits like a trained LM head: a common offset of -100 (one hidden coordinate 10 against weights -10), a
    per-row spread of a few units, and every 8th row peaked on its label with p_target > 1 - 1e-6."""
    gen = torch.Generator().manual_seed(seed)
    W = torch.randn(V, d, generator=gen) * 0.05
    W[:, 0] = -10.0
    W = W.bfloat16()
    h = torch.randn(nseq * T, d, generator=gen) * 1.5
    h[:, 0] = 10.0
    labels = torch.randint(0, V, (nseq, T), generator=gen)
    nxt = torch.cat([labels[:, 1:], labels[:, :1]], 1).reshape(-1)
    peaked = torch.arange(nseq * T) % 8 == 0
    h[peaked, 1:] += 20.0 * W[nxt[peaked], 1:].float()
    h = h.bfloat16()
    lens = torch.randint(T // 2, T + 1, (nseq,), generator=gen)
    mask = (torch.arange(T)[None, :] < lens[:, None]).long()
    gseq = torch.randn(nseq, generator=gen)
    return h.view(nseq, T, d).to(device), W.to(device), labels.to(device), mask.to(device), gseq.to(device), peaked


@pytest.mark.gpu
def test_lmhead_cfg2_gpt2_like_logits_fp64(pg, cuda_device):
    """cfg2 (4096 x 50257 x 1024) with GPT-2-like logits against fp64, per row: lse and ztgt within the logit error
    dot_err (plus 16 ulps for lse), seq_logp within the sum of its rows' tolerances, dH per row and dW per vocabulary
    row within row_bound, eps_p = 2^-21 + ln 2 (2^-23 * 4 * max|lse| log2 e + log2 e * dot_err) + max |lse - lse_fp64|
    (the backward runs on the forward's lse, whose error is measured once the forward has passed)."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    print(card())
    nseq, T, d, V = 32, 128, 1024, 50257
    h, W, labels, mask, gseq, peaked = gpt2_like_inputs(nseq, T, d, V, 2024, cuda_device)
    seq, lse, ztgt, rl, rw, _ = F.lmhead_logprob_fwd(h, W, labels, mask, False)
    dh, dw = F.lmhead_logprob_bwd(h, W, rl, rw, lse, gseq, False, dhidden_dtype=torch.float32)
    hf = h.reshape(-1, d)
    n = nseq * T
    lse_ref = torch.empty(n, dtype=torch.float64, device=cuda_device)
    zt_ref = torch.zeros(n, dtype=torch.float64, device=cuda_device)
    _, ncoef, tgt = lmhead_row_stats(labels, mask, gseq)
    tl = tgt.long()
    pt = torch.zeros(n, dtype=torch.float64, device=cuda_device)
    for r0 in range(0, n, 1024):
        z = hf[r0:r0 + 1024].double() @ W.double().T
        lse_ref[r0:r0 + 1024] = torch.logsumexp(z, 1)
        t = tl[r0:r0 + 1024]
        v = t >= 0
        zz = z.gather(1, t.clamp_min(0)[:, None]).squeeze(1)
        zt_ref[r0:r0 + 1024] = torch.where(v, zz, torch.zeros_like(zz))
        pt[r0:r0 + 1024] = torch.where(v, torch.exp(zz - lse_ref[r0:r0 + 1024]), torch.zeros_like(zz))
    pk = peaked.to(cuda_device) & (tl >= 0)
    assert float(pt[pk].min()) > 1 - 1e-6 and float(lse_ref.mean()) < -70      # the inputs are what they claim
    hn, wn = hf.double().norm(dim=1), W.double().norm(dim=1)
    dz = dot_err(d, 1.0, float(hn.max()), float(wn.max()))
    scored = tl >= 0
    ok, worst = within(ztgt[scored], zt_ref[scored], torch.full_like(zt_ref[scored], dz))
    report("cfg2 gpt2-like ztgt", worst)
    assert ok
    ltol = ulps(lse_ref, 16) + dz
    ok, worst = within(lse, lse_ref, ltol)
    report("cfg2 gpt2-like lse", worst)
    assert ok
    i = int(torch.nonzero(pk).flatten()[0])
    assert not within(lse[i:i + 1], (lse_ref[i] + LN2).reshape(1), ltol[i:i + 1])[0]
    t2 = int(tl[i]) + 1 if int(tl[i]) + 1 < V else int(tl[i]) - 1
    zmoved = float(hf[i].double() @ W[t2].double())
    assert abs(float(ztgt[i]) - zmoved) > dz                                     # a moved target is seen in ztgt
    w = -ncoef / gseq.double().repeat_interleave(T)
    seq_ref = ((zt_ref - lse_ref) * w).view(nseq, T).sum(1)
    seq_tol = ((ltol + dz) * w.abs()).view(nseq, T).sum(1)
    ok, worst = within(seq, seq_ref, seq_tol)
    report("cfg2 gpt2-like seq_logp", worst)
    assert ok
    row = (lse_ref, ncoef, tgt)
    eps_p = (2.0 ** -21 + LN2 * (2.0 ** -23 * 4 * float(lse_ref.abs().max()) * LOG2E + LOG2E * dz)
             + float((lse.double() - lse_ref).abs().max()))
    ref = Reference(hf, W, 1.0, row, None, eps_p, chunk=1024)
    bounds = ref.bounds
    faults = planted_faults(hf, W, 1.0, row, None)
    assert_bounded_and_sensitive((dh.reshape(-1, d), dw), ref, bounds, faults, hf, W, "cfg2 gpt2-like bwd", report)
