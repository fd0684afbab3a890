"""Compacted DPO head with the row count kept on the device (functional.lmhead_compact_fwd_bucketed / _bwd_bucketed,
the *_dev entry points of csrc/compact.cu) and its CUDA-graph step (graphs.GraphedCompactDPOStep).

CPU: the host bucket rule against a numpy restatement of prep_rows, the ABI prototypes and argument refusals, and a
numpy restatement of the device compaction that shows every index stays in bounds when the masks score more rows
than the bucket holds.  GPU (one B200): cfg2's shape (16 pairs, T = 128, d = 1024, V = 50257) at the reference's
caption statistics (470 / 1555 / 4064 scored rows) and a ragged small case, against the fp64 oracle with the per-row
bounds of test_kernel_exactness.py and against the eager compacted path; stale values across replays; the overflow
flag; no host synchronisation in a replay."""
import ctypes

import numpy as np
import pytest
import torch

from test_kernel_exactness import (LN2, LOG2E, Reference, card, dot_err, report, rows_within,  # noqa: F401
                                   ulps, within)

NEW_ENTRY_POINTS = {"pgica_compact_rows_dev": 8, "pgica_gather_rows_bf16_dev": 11, "pgica_gather_u32_dev": 6,
                    "pgica_scatter_u32_dev": 6, "pgica_scatter_rows_dev": 9}


# ================================================================================================ numpy restatements
def prep_rows_weight(mask, nseq, T):
    """pgica_prep_rows' row weight, restated: w[b, t] = float32(mask[b, t + 1]) for t < T - 1, else 0 (an out-of-vocabulary
    label only turns a nonzero weight into NaN, which is still nonzero)."""
    w = np.zeros((nseq, T), dtype=np.float32)
    if T > 1:
        if mask is None:
            w[:, :-1] = 1.0
        else:
            m = mask.numpy() if mask.dtype != torch.bool else mask.numpy().astype(np.uint8)
            if mask.dtype in (torch.int64, torch.int32, torch.float32, torch.bool, torch.uint8):
                w[:, :-1] = m[:, 1:].astype(np.float32)
            else:  # functional.mask_kind hands any other dtype over as float32
                w[:, :-1] = mask.float().numpy()[:, 1:]
    return w.reshape(-1)


def compact_restated(row_weight, set_rows, rows_launch):
    """compact_rows_dev_kernel, restated: -> (index[rows_launch], slot[R], info[2 nset + 2])."""
    R = int(sum(set_rows))
    scored = row_weight != 0  # NaN != 0
    pos = np.cumsum(scored) - scored
    slot = np.where(scored, pos, -1).astype(np.int32)
    n = int(scored.sum())
    index = np.full(rows_launch, -1, dtype=np.int32)
    keep = scored & (pos < rows_launch)
    index[pos[keep]] = np.nonzero(keep)[0]
    begin = np.concatenate([[0], np.cumsum(set_rows)]).astype(np.int64)
    offsets = [int(pos[b]) for b in begin[:-1]]
    counts = [(offsets[s + 1] if s + 1 < len(set_rows) else n) - offsets[s] for s in range(len(set_rows))]
    assert begin[-1] == R
    return index, slot, np.array(counts + offsets + [n, int(n > rows_launch)], dtype=np.int32)


def caption_masks(nseq, T, total, seed):
    """int64 masks of captions (ones on [0, L_b)) whose scored rows (L_b - 1 each) sum to `total`."""
    gen = np.random.default_rng(seed)
    lens = np.full(nseq, 1 + total // nseq)
    lens[: total % nseq] += 1
    for _ in range(4 * nseq):  # shuffle lengths around, keeping the total
        i, j = gen.integers(0, nseq, 2)
        k = int(gen.integers(0, 4))
        if lens[i] - k >= 2 and lens[j] + k <= T:
            lens[i] -= k
            lens[j] += k
    assert int((lens - 1).sum()) == total and lens.max() <= T
    m = torch.zeros(nseq, T, dtype=torch.int64)
    for b, L in enumerate(lens):
        m[b, :L] = 1
    return m


# ================================================================================================ CPU tests
@pytest.mark.parametrize("kind", ["int64", "bool", "float32", "float64", "int32", "none", "zero_rows", "T1"])
def test_bucket_rule_matches_prep_rows(kind):
    from preference_guided_image_captioning_alignment_b200.graphs import BUCKET_ROWS, bucket_rows, scored_rows
    gen = torch.Generator().manual_seed(7)
    nseq, T = 6, 1 if kind == "T1" else 19
    m = (torch.rand(nseq, T, generator=gen) < 0.6)
    mask = {"int64": m.long(), "bool": m, "int32": m.int(), "none": None, "T1": m.long(),
            "float32": m.float() * torch.randn(nseq, T, generator=gen), "float64": m.double() * 1e-50,
            "zero_rows": m.long() * (torch.arange(nseq)[:, None] % 2)}[kind]
    if kind == "float32":
        mask[0, 3], mask[1, 4] = float("nan"), -0.0
    n = int((prep_rows_weight(mask, nseq, T) != 0).sum())
    assert scored_rows(mask, nseq, T) == n
    if kind == "float64":
        assert n == 0  # 1e-50 is 0 in the float32 the kernel reads
    if kind == "zero_rows":
        assert prep_rows_weight(mask, nseq, T).reshape(nseq, T)[0::2].sum() == 0
    assert bucket_rows(n) == max(1, -(-n // BUCKET_ROWS)) * BUCKET_ROWS
    assert bucket_rows(0) == bucket_rows(1) == BUCKET_ROWS and bucket_rows(257) == 512


def test_device_count_prototypes_and_refusals():
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F
    protos = _lib.parse_header()
    for name, nargs in NEW_ENTRY_POINTS.items():
        assert name in protos and len(protos[name][1]) == nargs, name
    lib = _lib.load()
    host = (ctypes.c_int32 * 4096)()
    hp = ctypes.cast(host, ctypes.c_void_p)
    rows = (ctypes.c_int64 * 2)(64, 64)
    # bad sizes are refused before any pointer is looked at
    assert lib.pgica_compact_rows_dev(hp, 0, rows, 256, hp, hp, hp, None) == -1
    assert lib.pgica_compact_rows_dev(hp, 9, rows, 256, hp, hp, hp, None) == -1
    assert lib.pgica_compact_rows_dev(hp, 2, (ctypes.c_int64 * 2)(64, 0), 256, hp, hp, hp, None) == -1
    assert lib.pgica_compact_rows_dev(hp, 2, rows, 0, hp, hp, hp, None) == -1
    assert b"rows_launch" in lib.pgica_last_error()
    srcs = (ctypes.c_void_p * 2)(hp.value, hp.value)
    bf = (ctypes.c_int32 * 2)(0, 0)
    assert lib.pgica_gather_rows_bf16_dev(2, srcs, bf, rows, hp, 256, 1001, hp, None, None, None) == -1
    assert b"d % 8" in lib.pgica_last_error()
    assert lib.pgica_gather_rows_bf16_dev(2, srcs, bf, rows, hp, 256, 64, hp, hp, None, None) == -1
    assert lib.pgica_gather_u32_dev(hp, 0, hp, 256, hp, None) == -1
    assert lib.pgica_scatter_u32_dev(hp, 256, hp, 0, hp, None) == -1
    assert lib.pgica_scatter_rows_dev(hp, 0, 256, hp, 128, 6, hp, 0, None) == -1
    # well-formed calls on host memory are refused: a kernel must never be handed a host pointer
    for rc in (lib.pgica_compact_rows_dev(hp, 2, rows, 256, hp, hp, hp, None),
               lib.pgica_gather_rows_bf16_dev(2, srcs, bf, rows, hp, 256, 64, hp, None, None, None),
               lib.pgica_gather_u32_dev(hp, 128, hp, 256, hp, None),
               lib.pgica_scatter_u32_dev(hp, 256, hp, 128, hp, None),
               lib.pgica_scatter_rows_dev(hp, 0, 256, hp, 128, 64, hp, 0, None)):
        assert rc == -1
        err = lib.pgica_last_error()
        assert b"not device memory" in err or b"cannot query pointer" in err, err
    with pytest.raises(_lib.PgicaError):
        F.lmhead_compact_fwd_bucketed([torch.zeros(2, 5, 8)], torch.zeros(11, 8, dtype=torch.bfloat16),
                                      [torch.zeros(2, 5, dtype=torch.long)], [None], 256)


@pytest.mark.parametrize("rows_launch", [256, 512, 1024])
def test_compaction_restatement_stays_in_bounds(rows_launch):
    """The clamping of the device-count kernels, restated: with masks that score more rows than rows_launch every index
    a kernel dereferences is inside its buffer, the dropped rows' lse becomes NaN and their dH zero."""
    gen = np.random.default_rng(rows_launch)
    set_rows = [16 * 128, 16 * 128]
    w = (gen.random(sum(set_rows)) < 0.3).astype(np.float32)
    w[5] = np.nan
    R = len(w)
    index, slot, info = compact_restated(w, set_rows, rows_launch)
    n = int((w != 0).sum())
    assert info[-2] == n and info[-1] == int(n > rows_launch) and info[:2].sum() == n
    assert info[2] == 0 and info[3] == info[0]
    # gather_rows_dev / gather_u32_dev: index[p] is used only inside [0, R); padding positions read nothing
    used = index[(index >= 0) & (index < R)]
    assert used.size == min(n, rows_launch) and np.all(w[used] != 0)
    assert np.all(index[min(n, rows_launch):] == -1)
    # scatter_u32_dev / scatter_rows_dev: slot[r] is used only inside [0, rows_launch)
    src = np.arange(rows_launch, dtype=np.float32) + 1
    p = slot
    lse = np.where(p < 0, 0.0, np.where(p < rows_launch, src[np.clip(p, 0, rows_launch - 1)], np.nan))
    assert np.all(np.isnan(lse) == (p >= rows_launch))
    assert np.all(lse[w == 0] == 0)
    dropped = (w != 0) & (p >= rows_launch)
    assert dropped.sum() == max(0, n - rows_launch)
    ok = (p >= 0) & (p < rows_launch)
    assert np.array_equal(index[p[ok]], np.nonzero(ok)[0])  # slot and index are inverse on the kept rows


# ================================================================================================ GPU tests
V_CFG2, D_CFG2, B_CFG2, T_CFG2 = 50257, 1024, 16, 128
ROW_COUNTS = [470, 1555, 4064]


@pytest.fixture(scope="module")
def pg(cuda_device):
    import preference_guided_image_captioning_alignment_b200 as pkg
    from preference_guided_image_captioning_alignment_b200 import _lib
    assert _lib.load().pgica_device_check() == 0
    return pkg


@pytest.fixture(scope="module")
def cfg2(cuda_device):
    """Policy / reference weights and hidden states of cfg2's shape; labels in the vocabulary."""
    gen = torch.Generator().manual_seed(2025)
    dev = cuda_device
    W = (torch.randn(V_CFG2, D_CFG2, generator=gen) * 0.05).bfloat16().to(dev)
    Wr = (W.float().cpu() + 0.01 * torch.randn(V_CFG2, D_CFG2, generator=gen)).bfloat16().to(dev)
    H = torch.randn(2 * B_CFG2, T_CFG2, D_CFG2, generator=gen).to(dev)
    Hr = (H.cpu() + 0.1 * torch.randn(2 * B_CFG2, T_CFG2, D_CFG2, generator=gen)).to(dev)
    y = torch.randint(0, V_CFG2, (2 * B_CFG2, T_CFG2), generator=gen).to(dev)
    return W, Wr, H, Hr, y


def eager_step(F, H, W, y, m, Hr, Wr, ln, beta=0.1):
    """The eager compacted path: lmhead_compact_fwd / _bwd (one host read of the row counts), DPO scalar head."""
    B = H.shape[0] // 2
    ms = [None, None] if m is None else [m[:B], m[B:]]
    (pc, pr), ctx = F.lmhead_compact_fwd([H[:B], H[B:]], W, [y[:B], y[B:]], ms, ln)
    rc = rr = None
    if Wr is not None:
        (rc, rr), _ = F.lmhead_compact_fwd([Hr[:B], Hr[B:]], Wr, [y[:B], y[B:]], ms, ln)
    loss, metrics, dpc = F.dpo_loss_fwd(pc, pr, rc, rr, beta, 0.0, B)
    g = F.dpo_grad_seq(dpc, torch.ones(1, device=H.device))
    dhs, dw = F.lmhead_compact_bwd(ctx, W, [g[:B], g[B:]], dhidden_dtypes=[H.dtype, H.dtype])
    return dict(loss=loss, metrics=metrics, seq=torch.cat([pc, pr]), dh=torch.cat(dhs), dw=dw,
                lse=torch.cat(ctx.lse))


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300))


def assert_step_matches(step, ref, mask, what):
    """Graphed step against the eager compacted path: loss, metrics, dH, dW to fp32 reordering, unscored rows of dH and
    lse exact zeros."""
    torch.cuda.synchronize()
    assert abs(float(step.loss) - float(ref["loss"])) <= 1e-5 * max(1.0, abs(float(ref["loss"]))), what
    torch.testing.assert_close(step.metrics, ref["metrics"], rtol=1e-5, atol=1e-5)
    assert rel(step.dweight, ref["dw"]) < 1e-5, (what, rel(step.dweight, ref["dw"]))
    assert rel(step.dhidden, ref["dh"]) < 1e-5, (what, rel(step.dhidden, ref["dh"]))
    ctx = step.graphs[step.rows_launch][2][0]
    T = step.hidden.shape[1]
    unscored = torch.ones_like(step.labels, dtype=torch.bool)
    if mask is not None:
        unscored[:, :-1] = mask.to(step.labels.device)[:, 1:] == 0
    else:
        unscored[:, :-1] = False
    assert torch.count_nonzero(step.dhidden[unscored]) == 0, what
    assert torch.count_nonzero(ctx.lse.view(-1, T)[unscored]) == 0, what
    torch.testing.assert_close(ctx.lse.view(-1, T)[~unscored], ref["lse"].view(-1, T)[~unscored], rtol=0, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROW_COUNTS + ["ragged"])
def test_bucketed_against_fp64_oracle(pg, cuda_device, cfg2, n):
    """Bucketed forward / backward on the scored rows of two sets: index plumbing bit-exact against the numpy
    restatement, per-row lse / target logit / sequence log-prob against fp64 (tolerances of test_kernel_exactness),
    dH per scored row and dW per vocabulary row within row_bound, unscored dH rows exact zeros; the same seqs as the
    eager compacted path."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    from preference_guided_image_captioning_alignment_b200.graphs import bucket_rows, scored_rows
    print(card())
    dev = cuda_device
    W = cfg2[0]
    if n == "ragged":  # different set shapes, one fp32 and one bf16 set, float and bool masks, d = 512
        gen = torch.Generator().manual_seed(11)
        d, V = 512, 1000
        W = (torch.randn(V, d, generator=gen) * 0.05).bfloat16().to(dev)
        hs = [torch.randn(3, 37, d, generator=gen).to(dev), torch.randn(5, 21, d, generator=gen).bfloat16().to(dev)]
        ys = [torch.randint(0, V, (3, 37), generator=gen).to(dev), torch.randint(0, V, (5, 21), generator=gen).to(dev)]
        ms = [(torch.rand(3, 37, generator=gen) < 0.5).float() * 2.5, torch.rand(5, 21, generator=gen) < 0.3]
        ln = True
    else:
        _, _, H, _, y = cfg2
        d, V, B = D_CFG2, V_CFG2, B_CFG2
        m = caption_masks(2 * B, T_CFG2, n, seed=n)
        hs, ys, ms = [H[:B], H[B:]], [y[:B], y[B:]], [m[:B], m[B:]]
        ln = n == 1555
    total = sum(scored_rows(mm, *mm.shape) for mm in ms)
    rows_launch = bucket_rows(total)
    msd = [mm.to(dev) for mm in ms]
    seqs, ref_seqs, ctx = F.lmhead_compact_fwd_bucketed(hs, W, ys, msd, rows_launch, ln)
    assert ref_seqs is None
    gen = torch.Generator().manual_seed(3)
    gseqs = [torch.randn(h.shape[0], generator=gen).to(dev) for h in hs]
    dhs, dw = F.lmhead_compact_bwd_bucketed(ctx, W, gseqs, dhidden_dtypes=[torch.float32, torch.float32])
    torch.cuda.synchronize()
    # ---- plumbing, bit for bit
    w_np = np.concatenate([prep_rows_weight(mm, *mm.shape) for mm in ms])
    set_rows = [h.shape[0] * h.shape[1] for h in hs]
    index, slot, info = compact_restated(w_np, set_rows, rows_launch)
    assert np.array_equal(ctx.index.cpu().numpy(), index)
    assert np.array_equal(ctx.slot.cpu().numpy(), slot)
    assert np.array_equal(ctx.info.cpu().numpy(), info) and info[-1] == 0 and info[-2] == total
    tgt_all = torch.cat([torch.cat([yy[:, 1:], torch.full_like(yy[:, :1], -1)], 1).reshape(-1) for yy in ys])
    keep = torch.from_numpy(index[:total]).long().to(dev)
    lab = ctx.label_c.long()
    assert torch.equal(lab[:total], tgt_all[keep]) and bool((lab[total:] == -1).all())
    hall = torch.cat([h.reshape(-1, d).bfloat16() for h in hs])
    hc = hall[keep]
    assert torch.equal(ctx.hidden_c[:total], hc) and torch.count_nonzero(ctx.hidden_c[total:]) == 0
    # ---- forward against fp64
    Wd = W.double()
    z = hc.double() @ Wd.T
    lse_ref = torch.logsumexp(z, 1)
    zt_ref = z.gather(1, lab[:total, None]).squeeze(1)
    del z
    dz = dot_err(d, 1.0, float(hc.double().norm(dim=1).max()), float(Wd.norm(dim=1).max()))
    ltol = ulps(lse_ref, 16) + dz
    lse_all, zt_all = ctx.lse, ctx.ztgt
    ok, worst = within(lse_all[keep], lse_ref, ltol)
    report(f"bucketed {n} lse", worst)
    assert ok
    ok, worst = within(zt_all[keep], zt_ref, torch.full_like(zt_ref, dz))
    report(f"bucketed {n} ztgt", worst)
    assert ok
    unscored = torch.ones(len(w_np), dtype=torch.bool, device=dev)
    unscored[keep] = False
    assert torch.count_nonzero(lse_all[unscored]) == 0 and torch.count_nonzero(zt_all[unscored]) == 0
    wd = torch.from_numpy(w_np).double().to(dev)
    begin = np.concatenate([[0], np.cumsum(set_rows)])
    lp = torch.zeros(len(w_np), dtype=torch.float64, device=dev)
    lp[keep] = zt_ref - lse_ref
    tol_r = torch.zeros_like(lp)
    tol_r[keep] = ltol + dz
    ncoef = torch.zeros(len(w_np), dtype=torch.float64, device=dev)
    eager_seqs, _ = F.lmhead_compact_fwd(hs, W, ys, msd, ln)
    for s, h in enumerate(hs):
        nseq, T = h.shape[:2]
        ws = wd[begin[s]:begin[s + 1]].view(nseq, T)
        den = ws.sum(1) if ln else torch.ones(nseq, dtype=torch.float64, device=dev)
        seq_ref = (lp[begin[s]:begin[s + 1]].view(nseq, T) * ws).sum(1) / den
        seq_tol = (tol_r[begin[s]:begin[s + 1]].view(nseq, T) * ws.abs()).sum(1) / den.abs() + ulps(seq_ref, 64)
        ok, worst = within(seqs[s], seq_ref, seq_tol)
        report(f"bucketed {n} seq set {s}", worst)
        assert ok
        torch.testing.assert_close(seqs[s], eager_seqs[s], rtol=1e-6, atol=1e-5)
        ncoef[begin[s]:begin[s + 1]] = (-gseqs[s].double()[:, None] * ws / den[:, None]).reshape(-1)
    # ---- backward against fp64: dH on the scored rows, dW on every vocabulary row
    row = (lse_ref, ncoef[keep], lab[:total].int())
    eps_p = (2.0 ** -21 + LN2 * (2.0 ** -23 * 4 * float(lse_ref.abs().max()) * LOG2E + LOG2E * dz)
             + float((lse_all[keep].double() - lse_ref).abs().max()))
    ref = Reference(hc, W, 1.0, row, None, eps_p, chunk=1024)
    dh_all = torch.cat([x.reshape(-1, d) for x in dhs])
    for out, r, b, side in ((dh_all[keep], ref.out_x, ref.bounds[0], "dH"), (dw, ref.out_y, ref.bounds[1], "dW")):
        ok, worst = rows_within(out, r, b)
        report(f"bucketed {n} {side}", worst)
        assert ok, (side, worst)
    assert torch.count_nonzero(dh_all[unscored]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("with_ref", [False, True])
@pytest.mark.parametrize("ln", [False, True])
def test_graphed_step_matches_eager(pg, cuda_device, cfg2, with_ref, ln):
    """GraphedCompactDPOStep (fp32 master weight, cast to bf16 inside the forward graph) against the eager compacted path
    at the three caption statistics, one step object replaying each: loss, metrics, dH, dW, lse; unscored dH rows exact
    zeros."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    W, Wr, H, Hr, y = cfg2
    head = pg.FusedDPOHead(beta=0.1, length_normalize=ln)
    m0 = caption_masks(2 * B_CFG2, T_CFG2, ROW_COUNTS[0], seed=1)
    step = pg.GraphedCompactDPOStep(head, W.float(), Wr if with_ref else None, H, y.cpu(), m0,
                                    Hr if with_ref else None)
    for n in ROW_COUNTS:
        m = caption_masks(2 * B_CFG2, T_CFG2, n, seed=n + 1).pin_memory()
        step.copy_inputs(H, y.cpu().pin_memory(), m, Hr if with_ref else None)
        step.launch()
        value = step.loss_value()
        ref = eager_step(F, H, W, y, m.to(cuda_device), Hr, Wr if with_ref else None, ln)
        assert abs(value - float(ref["loss"])) <= 1e-5 * max(1.0, abs(float(ref["loss"])))
        assert_step_matches(step, ref, m, f"n={n} ref={with_ref} ln={ln}")
    assert sorted(step.graphs) == [512, 1792, 4096]


@pytest.mark.gpu
def test_replays_leave_no_stale_values(pg, cuda_device, cfg2):
    """Mask A, then mask B with fewer scored rows in the same bucket, then mask C in a smaller bucket, then A again:
    every replay's dH, lse, sequence log-probs and gradients are those of its own mask."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    from preference_guided_image_captioning_alignment_b200.graphs import bucket_rows
    W, Wr, H, Hr, y = cfg2
    head = pg.FusedDPOHead(beta=0.1)
    mA = caption_masks(2 * B_CFG2, T_CFG2, 1555, seed=21)
    mB = caption_masks(2 * B_CFG2, T_CFG2, 1540, seed=22)
    mC = caption_masks(2 * B_CFG2, T_CFG2, 470, seed=23)
    assert bucket_rows(1555) == bucket_rows(1540) != bucket_rows(470)
    step = pg.GraphedCompactDPOStep(head, W.float(), Wr, H, y.cpu(), mA, Hr)
    gen = torch.Generator().manual_seed(5)
    for k, m in enumerate((mA, mB, mC, mA)):
        Hk = H + 0.5 * torch.randn(H.shape, generator=gen).to(cuda_device)  # new hidden states every step
        step.copy_inputs(Hk, y.cpu().pin_memory(), m.pin_memory(), Hr)
        step.launch()
        ref = eager_step(F, Hk, W, y, m.to(cuda_device), Hr, Wr, False)
        step.loss_value()
        assert_step_matches(step, ref, m, f"replay {k}")
        ctx = step.graphs[step.rows_launch][2][0]
        torch.testing.assert_close(F.seq_reduce(ctx.lse, ctx.ztgt, ctx.row_weight, 2 * B_CFG2, T_CFG2), ref["seq"],
                                   rtol=1e-6, atol=1e-5)


@pytest.mark.gpu
def test_overflow_sets_flag_and_loss_raises(pg, cuda_device, cfg2):
    """Device masks that score more rows than the host's bucket: nothing out of bounds, the flag is set, the loss is
    NaN and loss_value() raises; the next consistent step is correct again."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    W, Wr, H, Hr, y = cfg2
    head = pg.FusedDPOHead(beta=0.1)
    m = caption_masks(2 * B_CFG2, T_CFG2, 470, seed=31)
    step = pg.GraphedCompactDPOStep(head, W.float(), Wr, H, y.cpu(), m, Hr)
    step.copy_inputs(H, y.cpu().pin_memory(), m.pin_memory(), Hr)
    step.launch()
    step.loss_value()
    step.mask.fill_(1)  # the device now scores 4064 rows; the host still picked the 512-row bucket
    step.launch()
    with pytest.raises(RuntimeError, match="bucket"):
        step.loss_value()
    torch.cuda.synchronize()
    assert torch.isnan(step.loss)
    ctx = step.graphs[512][2][0]
    assert ctx.info.tolist()[-2:] == [4064, 1]
    assert torch.count_nonzero(step.dhidden[:, -1]) == 0  # never-scored rows stay exact zeros
    step.copy_inputs(H, y.cpu().pin_memory(), m.pin_memory(), Hr)
    step.launch()
    step.loss_value()
    assert_step_matches(step, eager_step(F, H, W, y, m.to(cuda_device), Hr, Wr, False), m, "after overflow")


@pytest.mark.gpu
def test_replay_issues_no_host_synchronisation(pg, cuda_device, cfg2):
    """Once a bucket's graphs exist, copy_inputs + launch neither synchronise nor read anything back (sync debug mode
    raises on any synchronising call), and the profiler sees no synchronising runtime call."""
    W, Wr, H, Hr, y = cfg2
    head = pg.FusedDPOHead(beta=0.1)
    m = caption_masks(2 * B_CFG2, T_CFG2, 470, seed=41).pin_memory()
    yp = y.cpu().pin_memory()
    step = pg.GraphedCompactDPOStep(head, W.float(), Wr, H, yp, m, Hr)
    step.copy_inputs(H, yp, m, Hr)
    step.launch()
    step.loss_value()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.cuda.set_sync_debug_mode("error")
        try:
            for _ in range(3):
                step.copy_inputs(H, yp, m, Hr)
                step.launch()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
    names = {e.key for e in prof.key_averages()}
    assert not names & {"cudaStreamSynchronize", "cudaEventSynchronize", "cudaMemcpy"}, names
    assert sum(e.count for e in prof.key_averages() if e.key == "cudaGraphLaunch") == 6
    assert step.loss_value() == step.loss_value()
