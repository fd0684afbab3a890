"""Tensor-level wrappers over the C ABI (include/pgica.h): allocate outputs with torch, pass raw device
pointers and the current CUDA stream.  No arithmetic happens here — PyTorch is only memory and streams.
"""
import ctypes

import torch

from . import _lib

MASK_NONE, MASK_I64, MASK_F32, MASK_U8, MASK_I32 = 0, 1, 2, 3, 4


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.PgicaError(
                "pgica ops run on a B200 only (got a %s tensor); there is no CPU fallback" % t.device.type)


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def as_bf16(x):
    """bf16 contiguous view/copy of a float tensor; fp32 goes through the library's cast kernel."""
    _need_cuda(x)
    if x.dtype == torch.bfloat16:
        return x.contiguous()
    if x.dtype != torch.float32:
        x = x.float()
    x = x.contiguous()
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    if x.numel():
        _lib.check(_lib.load().pgica_cast_f32_to_bf16(_p(x), x.numel(), _p(y), _stream()))
    return y


def mask_kind(mask):
    if mask is None:
        return MASK_NONE, None
    if mask.dtype == torch.int64:
        return MASK_I64, mask.contiguous()
    if mask.dtype == torch.float32:
        return MASK_F32, mask.contiguous()
    if mask.dtype in (torch.bool, torch.uint8):
        return MASK_U8, mask.contiguous().view(torch.uint8)
    if mask.dtype == torch.int32:
        return MASK_I32, mask.contiguous()
    return MASK_F32, mask.float().contiguous()


# ----------------------------------------------------------------------------------------- K1/K3 core
def gemm_lse(a, b, scale=1.0, labels=None, diag_offset=0, want_tgt=True):
    """lse[i] = logsumexp_j scale*<a_i, b_j>;  tgt[i] = scale*<a_i, b_label(i)>.  a, b bf16 [*, k]."""
    _need_cuda(a, b, labels)
    lib = _lib.load()
    rows, k = a.shape
    cols = b.shape[0]
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_gemm_lse_workspace_bytes(rows, cols, k, ctypes.byref(need)))
    ws = _ws(need.value, a.device)
    lse = torch.empty(rows, dtype=torch.float32, device=a.device)
    tgt = torch.empty(rows, dtype=torch.float32, device=a.device) if want_tgt else None
    _lib.check(lib.pgica_gemm_lse(_p(a), _p(b), rows, cols, k, float(scale), _p(labels), int(diag_offset), _p(lse),
                                  _p(tgt), _p(ws), need.value, _stream()))
    return lse, tgt


def similarity(a, b, scale=1.0):
    """Dense fp32 (rows, cols) matrix scale*<a_i, b_j> (scoring API; the loss path never calls this)."""
    _need_cuda(a, b)
    lib = _lib.load()
    rows, k = a.shape
    cols = b.shape[0]
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_gemm_lse_workspace_bytes(rows, cols, k, ctypes.byref(need)))
    ws = _ws(need.value, a.device)
    sim = torch.empty(rows, cols, dtype=torch.float32, device=a.device)
    lse = torch.empty(rows, dtype=torch.float32, device=a.device)
    _lib.check(lib.pgica_similarity(_p(a), _p(b), rows, cols, k, float(scale), _p(sim), _p(lse), _p(ws), need.value,
                                    _stream()))
    return sim


# ----------------------------------------------------------------------------------------- K2/K4 core
def softmax_grad_gemm(x, y, scale=1.0, row=None, col=None, out_dtype=torch.float32):
    """out = G(x y^T) y with G built from row stats (lse, coef, tgt) and/or column stats (see pgica.h)."""
    _need_cuda(x, y)
    lib = _lib.load()
    mx, k = x.shape
    my = y.shape[0]
    out = torch.empty(mx, k, dtype=out_dtype, device=x.device)
    r = row if row is not None else (None, None, None)
    c = col if col is not None else (None, None, None)
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_softmax_grad_gemm_workspace_bytes(mx, my, k, ctypes.byref(need)))
    ws = _ws(need.value, x.device)
    _lib.check(lib.pgica_softmax_grad_gemm(_p(x), _p(y), mx, my, k, float(scale), _p(r[0]), _p(r[1]), _p(r[2]),
                                           _p(c[0]), _p(c[1]), _p(c[2]), _p(out),
                                           1 if out_dtype == torch.bfloat16 else 0, _p(ws), need.value, _stream()))
    return out


def softmax_grad_gemm_dual(x, y, scale=1.0, row=None, col=None, out_x_dtype=torch.float32, out_y_dtype=torch.float32):
    """(out_x, out_y) = (G y, G^T x) from one recomputation of G(x y^T) (pgica_softmax_grad_gemm_dual)."""
    _need_cuda(x, y)
    lib = _lib.load()
    mx, k = x.shape
    my = y.shape[0]
    out_x = torch.empty(mx, k, dtype=out_x_dtype, device=x.device)
    out_y = torch.empty(my, k, dtype=out_y_dtype, device=x.device)
    r = row if row is not None else (None, None, None)
    c = col if col is not None else (None, None, None)
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_softmax_grad_gemm_dual_workspace_bytes(mx, my, k, ctypes.byref(need)))
    ws = _ws(need.value, x.device)
    _lib.check(lib.pgica_softmax_grad_gemm_dual(_p(x), _p(y), mx, my, k, float(scale), _p(r[0]), _p(r[1]), _p(r[2]),
                                                _p(c[0]), _p(c[1]), _p(c[2]), _p(out_x),
                                                1 if out_x_dtype == torch.bfloat16 else 0, _p(out_y),
                                                1 if out_y_dtype == torch.bfloat16 else 0, _p(ws), need.value,
                                                _stream()))
    return out_x, out_y


# ----------------------------------------------------------------------------------------- Stage-2 head
def lmhead_logprob_fwd(hidden, weight, labels, mask=None, length_normalize=False, want_nll=False):
    """hidden bf16 [nseq, T, d], weight bf16 [V, d], labels int64 [nseq, T] -> seq_logp [nseq] + saved ctx."""
    _need_cuda(hidden, weight, labels, mask)
    lib = _lib.load()
    nseq, T, d = hidden.shape
    V = weight.shape[0]
    dev = hidden.device
    kind, mask_c = mask_kind(mask)
    labels = labels.contiguous()
    if labels.dtype != torch.int64:
        labels = labels.long()
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_lmhead_logprob_workspace_bytes(nseq, T, d, V, ctypes.byref(need)))
    ws = _ws(need.value, dev)
    f32 = dict(dtype=torch.float32, device=dev)
    seq_logp = torch.empty(nseq, **f32)
    lse = torch.empty(nseq * T, **f32)
    ztgt = torch.empty(nseq * T, **f32)
    row_label = torch.empty(nseq * T, dtype=torch.int32, device=dev)
    row_weight = torch.empty(nseq * T, **f32)
    nll = torch.empty(1, **f32) if want_nll else None
    _lib.check(lib.pgica_lmhead_logprob_fwd(_p(hidden), _p(weight), _p(labels), _p(mask_c), kind, nseq, T, d, V,
                                            1 if length_normalize else 0, _p(seq_logp), _p(lse), _p(ztgt),
                                            _p(row_label), _p(row_weight), _p(nll), _p(ws), need.value, _stream()))
    return seq_logp, lse, ztgt, row_label, row_weight, nll


def sum_into(dst, sources, max_ctas=0):
    """dst += sum(sources) (fp32, same shape, contiguous); the grid is capped at max_ctas CTAs."""
    _need_cuda(dst, *sources)
    lib = _lib.load()
    arr = (ctypes.c_void_p * len(sources))(*[s.data_ptr() for s in sources])
    _lib.check(lib.pgica_sum_into_f32(_p(dst), arr, len(sources), dst.numel(), int(max_ctas), _stream()))
    return dst


def lmhead_logprob_bwd(hidden, weight, row_label, row_weight, lse, grad_seq, length_normalize=False,
                       need_dhidden=True, need_dweight=True, dhidden_dtype=torch.bfloat16,
                       dweight_dtype=torch.float32, dweight_out=None):
    _need_cuda(hidden, weight, grad_seq)
    lib = _lib.load()
    nseq, T, d = hidden.shape
    V = weight.shape[0]
    dev = hidden.device
    dh = torch.empty(nseq, T, d, dtype=dhidden_dtype, device=dev) if need_dhidden else None
    dw = None
    if need_dweight:
        if dweight_out is not None:  # caller-owned destination (e.g. a symmetric-memory buffer for the peer all-reduce)
            if tuple(dweight_out.shape) != (V, d) or not dweight_out.is_contiguous():
                raise ValueError("dweight_out must be a contiguous (V, d) tensor")
            dw, dweight_dtype = dweight_out, dweight_out.dtype
        else:
            dw = torch.empty(V, d, dtype=dweight_dtype, device=dev)
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_lmhead_logprob_workspace_bytes(nseq, T, d, V, ctypes.byref(need)))
    ws = _ws(need.value, dev)
    grad_seq = grad_seq.contiguous().float()
    _lib.check(lib.pgica_lmhead_logprob_bwd(_p(hidden), _p(weight), _p(row_label), _p(row_weight), _p(lse),
                                            _p(grad_seq), nseq, T, d, V, 1 if length_normalize else 0, _p(dh),
                                            1 if dhidden_dtype == torch.bfloat16 else 0, _p(dw),
                                            1 if dweight_dtype == torch.bfloat16 else 0, _p(ws), ws.numel(),
                                            _stream()))
    return dh, dw


def dpo_loss_fwd(pc, pr, rc=None, rr=None, beta=0.1, label_smoothing=0.0, n_global=None):
    _need_cuda(pc, pr, rc, rr)
    lib = _lib.load()
    n = pc.numel()
    f32 = dict(dtype=torch.float32, device=pc.device)
    loss = torch.empty((), **f32)
    metrics = torch.empty(5, **f32)
    dpc = torch.empty(n, **f32)
    _lib.check(lib.pgica_dpo_loss_fwd(_p(pc), _p(pr), _p(rc), _p(rr), n, int(n_global or n), float(beta),
                                      float(label_smoothing), _p(loss), _p(metrics), _p(dpc), _stream()))
    return loss, metrics, dpc


def scale_by_scalar(a, scalar, mult=1.0):
    lib = _lib.load()
    out = torch.empty_like(a)
    _lib.check(lib.pgica_scale_by_scalar(_p(a), _p(scalar), float(mult), a.numel(), _p(out), _stream()))
    return out


def dpo_grad_seq(dpc, grad_loss):
    """[dloss/dpc * g ; -dloss/dpc * g]: upstream gradient of the stacked (chosen ++ rejected) sequence log-probs."""
    lib = _lib.load()
    n = dpc.numel()
    out = torch.empty(2 * n, dtype=torch.float32, device=dpc.device)
    g = grad_loss.reshape(1)
    _lib.check(lib.pgica_scale_by_scalar(_p(dpc), _p(g), 1.0, n, _p(out), _stream()))
    _lib.check(lib.pgica_scale_by_scalar(_p(dpc), _p(g), -1.0, n, ctypes.c_void_p(out.data_ptr() + 4 * n), _stream()))
    return out


# ----------------------------------------------------------------------------------------- Stage-1 head
def ntxent_fwd(a, b, inv_tau, diag_offset=0, bounded=False):
    """Row LSE, diagonal and column-LSE (partial) of the (rows_a x rows_b) similarity slice.  bounded=True: the caller
    guarantees unit-norm rows (|<a_i, b_j>| <= 1) — both LSEs then come from ONE pass over the tiles
    (pgica_ntxent_fwd_bounded) instead of two."""
    _need_cuda(a, b)
    lib = _lib.load()
    ra, dim = a.shape
    rb = b.shape[0]
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_ntxent_workspace_bytes(ra, rb, dim, ctypes.byref(need)))
    ws = _ws(need.value, a.device)
    f32 = dict(dtype=torch.float32, device=a.device)
    lse_row, diag, lse_col = torch.empty(ra, **f32), torch.empty(ra, **f32), torch.empty(rb, **f32)
    fn = lib.pgica_ntxent_fwd_bounded if bounded else lib.pgica_ntxent_fwd
    _lib.check(fn(_p(a), _p(b), ra, rb, dim, float(inv_tau), int(diag_offset), _p(lse_row), _p(diag), _p(lse_col), _p(ws),
                  need.value, _stream()))
    return lse_row, diag, lse_col


def ntxent_loss(lse_row, diag, lse_col_owned, inv_denom):
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=lse_row.device)
    _lib.check(lib.pgica_ntxent_loss(_p(lse_row), _p(diag), _p(lse_col_owned), lse_row.numel(), float(inv_denom),
                                     _p(loss), _stream()))
    return loss


def lse_combine(parts):
    """parts fp32 [nparts, n] -> logsumexp over dim 0."""
    lib = _lib.load()
    parts = parts.contiguous()
    out = torch.empty(parts.shape[1], dtype=torch.float32, device=parts.device)
    _lib.check(lib.pgica_lse_combine(_p(parts), parts.shape[0], parts.shape[1], _p(out), _stream()))
    return out


def ntxent_bwd(a, b, inv_tau, diag_offset, lse_row, lse_col, grad_loss, grad_mult, need_da=True, need_db=True,
               da_dtype=torch.float32, db_dtype=torch.float32, bounded=False):
    """bounded=True: unit-norm rows promised (as in ntxent_fwd) — one exponential per element instead of two."""
    _need_cuda(a, b, grad_loss)
    lib = _lib.load()
    ra, dim = a.shape
    rb = b.shape[0]
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_ntxent_workspace_bytes(ra, rb, dim, ctypes.byref(need)))
    ws = _ws(need.value, a.device)
    da = torch.empty(ra, dim, dtype=da_dtype, device=a.device) if need_da else None
    db = torch.empty(rb, dim, dtype=db_dtype, device=a.device) if need_db else None
    grad_loss = grad_loss.reshape(1).float().contiguous()
    fn = lib.pgica_ntxent_bwd_bounded if bounded else lib.pgica_ntxent_bwd
    _lib.check(fn(_p(a), _p(b), ra, rb, dim, float(inv_tau), int(diag_offset), _p(lse_row), _p(lse_col), _p(grad_loss),
                  float(grad_mult), _p(da), 1 if da_dtype == torch.bfloat16 else 0, _p(db),
                  1 if db_dtype == torch.bfloat16 else 0, _p(ws), need.value, _stream()))
    return da, db


def rownorm_fwd(x, eps=1e-12, split=False):
    """-> (unit rows bf16, 1/norm, x as used[, left3, right3 when split])."""
    _need_cuda(x)
    lib = _lib.load()
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    rows, dim = x.shape
    y = torch.empty(rows, dim, dtype=torch.bfloat16, device=x.device)
    inv = torch.empty(rows, dtype=torch.float32, device=x.device)
    l3 = torch.empty(rows, 3 * dim, dtype=torch.bfloat16, device=x.device) if split else None
    r3 = torch.empty(rows, 3 * dim, dtype=torch.bfloat16, device=x.device) if split else None
    _lib.check(lib.pgica_rownorm_fwd(_p(x), 1 if x.dtype == torch.bfloat16 else 0, rows, dim, float(eps), _p(y),
                                     _p(inv), _p(l3), _p(r3), _stream()))
    return (y, inv, x, l3, r3) if split else (y, inv, x)


def rownorm_bwd(x, inv_norm, g, second=-1):
    """g is (rows, dim), or (rows, pitch) with the gradient in columns [0, dim) + [second, second + dim)."""
    lib = _lib.load()
    g = g.contiguous()
    rows, dim = x.shape
    dx = torch.empty(rows, dim, dtype=torch.float32, device=x.device)
    _lib.check(lib.pgica_rownorm_bwd(_p(x), 1 if x.dtype == torch.bfloat16 else 0, _p(inv_norm), _p(g),
                                     1 if g.dtype == torch.bfloat16 else 0, rows, dim, g.shape[1], int(second),
                                     _p(dx), _stream()))
    return dx


# ----------------------------------------------------------------------------------------- logits path
def lmhead_logprob_bwd_progress(hidden, weight, row_label, row_weight, lse, grad_seq, dweight_out, progress,
                                rows_per_segment, length_normalize=False, dhidden_dtype=torch.bfloat16):
    """Backward of the LM head that publishes its progress on dweight (pgica_lmhead_logprob_bwd_progress): dweight_out is
    a caller-owned fp32 (V, d) tensor (inside a symmetric buffer), `progress` a uint32/int32 device tensor with one
    counter per `rows_per_segment` rows.  -> (dhidden, increments one 256-row pair of dweight contributes)"""
    _need_cuda(hidden, weight, grad_seq, dweight_out, progress)
    lib = _lib.load()
    nseq, T, d = hidden.shape
    V = weight.shape[0]
    dev = hidden.device
    if tuple(dweight_out.shape) != (V, d) or dweight_out.dtype != torch.float32 or not dweight_out.is_contiguous():
        raise ValueError("dweight_out must be a contiguous fp32 (V, d) tensor")
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_lmhead_logprob_workspace_bytes(nseq, T, d, V, ctypes.byref(need)))
    ws = _ws(need.value, dev)
    dh = torch.empty(nseq, T, d, dtype=dhidden_dtype, device=dev)
    inc = ctypes.c_int32(0)
    _lib.check(lib.pgica_lmhead_logprob_bwd_progress(_p(hidden), _p(weight), _p(row_label), _p(row_weight), _p(lse),
                                                     _p(grad_seq.float().contiguous()), nseq, T, d, V,
                                                     1 if length_normalize else 0, _p(dh),
                                                     1 if dhidden_dtype == torch.bfloat16 else 0, _p(dweight_out),
                                                     _p(progress), int(rows_per_segment), ctypes.byref(inc), _p(ws),
                                                     ws.numel(), _stream()))
    return dh, inc.value


def peer_allreduce_progress(buf_ptrs, flag_ptrs, rank, progress, targets, seg_begin, epoch, local_sync, max_ctas=0,
                            stream=None, multicast_ptr=0):
    """Launch the progress-gated peer all-reduce (pgica_peer_allreduce_progress) on `stream` (default: current).
    multicast_ptr: the buffer through an NVSwitch multicast mapping (0: sums over unicast peer loads)."""
    lib = _lib.load()
    world, nseg = len(buf_ptrs), len(seg_begin) - 1
    bufs = (ctypes.c_void_p * world)(*[int(q) for q in buf_ptrs])
    flags = (ctypes.c_void_p * world)(*[int(q) for q in flag_ptrs])
    tg = (ctypes.c_uint32 * nseg)(*[int(t) & 0xFFFFFFFF for t in targets]) if progress is not None else None
    sb = (ctypes.c_int64 * (nseg + 1))(*[int(v) for v in seg_begin])
    st = ctypes.c_void_p(stream.cuda_stream) if stream is not None else _stream()
    mc = ctypes.c_void_p(int(multicast_ptr)) if multicast_ptr else None
    _lib.check(lib.pgica_peer_allreduce_progress(bufs, flags, mc, world, int(rank), _p(progress), tg, sb, nseg,
                                                 int(epoch) & 0xFFFFFFFF, _p(local_sync), int(max_ctas), st))


def prep_rows(labels, mask, vocab):
    _need_cuda(labels, mask)
    lib = _lib.load()
    nseq, T = labels.shape
    kind, mask_c = mask_kind(mask)
    labels = labels.contiguous()
    if labels.dtype != torch.int64:
        labels = labels.long()
    row_label = torch.empty(nseq * T, dtype=torch.int32, device=labels.device)
    row_weight = torch.empty(nseq * T, dtype=torch.float32, device=labels.device)
    _lib.check(lib.pgica_prep_rows(_p(labels), _p(mask_c), kind, nseq, T, int(vocab), _p(row_label), _p(row_weight),
                                   _stream()))
    return row_label, row_weight


def seq_reduce(lse, ztgt, row_weight, nseq, T, length_normalize=False):
    lib = _lib.load()
    out = torch.empty(nseq, dtype=torch.float32, device=lse.device)
    _lib.check(lib.pgica_seq_reduce(_p(lse), _p(ztgt), _p(row_weight), nseq, T, 1 if length_normalize else 0, _p(out),
                                    None, _stream()))
    return out


def row_coef(grad_seq, row_weight, nseq, T, length_normalize=False, sign=1.0):
    lib = _lib.load()
    coef = torch.empty(nseq * T, dtype=torch.float32, device=row_weight.device)
    grad_seq = grad_seq.contiguous().float()
    _lib.check(lib.pgica_row_coef(_p(grad_seq), _p(row_weight), nseq, T, 1 if length_normalize else 0, float(sign),
                                  _p(coef), _stream()))
    return coef


def logits_lse(logits, row_label):
    _need_cuda(logits)
    lib = _lib.load()
    nseq, T, V = logits.shape
    lse = torch.empty(nseq * T, dtype=torch.float32, device=logits.device)
    ztgt = torch.empty(nseq * T, dtype=torch.float32, device=logits.device)
    _lib.check(lib.pgica_logits_lse(_p(logits), 1 if logits.dtype == torch.bfloat16 else 0, _p(row_label), nseq, T, V,
                                    _p(lse), _p(ztgt), _stream()))
    return lse, ztgt


def logits_grad(logits, row_label, lse, coef):
    lib = _lib.load()
    nseq, T, V = logits.shape
    dlogits = torch.empty_like(logits)
    _lib.check(lib.pgica_logits_grad(_p(logits), 1 if logits.dtype == torch.bfloat16 else 0, _p(row_label), _p(lse),
                                     _p(coef), nseq, T, V, _p(dlogits), _stream()))
    return dlogits


def ntxent_small_supported(rows, dim):
    return bool(_lib.load().pgica_ntxent_small_supported(int(rows), int(dim)))


def ntxent_small(a, b, inv_tau, reduce_mean=True):
    """Whole symmetric NT-Xent (loss + unit-upstream gradients) of bf16 (B, D) operands, B <= 128, in one launch.
    -> (loss[], lse_row[B], lse_col[B], da[B, D] fp32, db[B, D] fp32)"""
    _need_cuda(a, b)
    lib = _lib.load()
    n, dim = a.shape
    f32 = dict(dtype=torch.float32, device=a.device)
    loss = torch.empty((), **f32)
    lse_row, lse_col = torch.empty(n, **f32), torch.empty(n, **f32)
    da, db = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
    _lib.check(lib.pgica_ntxent_small(_p(a), _p(b), n, dim, float(inv_tau), 1 if reduce_mean else 0, _p(loss),
                                      _p(lse_row), _p(lse_col), _p(da), _p(db), _stream()))
    return loss, lse_row, lse_col, da, db


def split3(x):
    """fp32 (rows, dim) -> bf16 (rows, 3*dim) pair ([hi|lo|hi], [hi|hi|lo]) WITHOUT normalising (pgica_split3_bf16)."""
    _need_cuda(x)
    lib = _lib.load()
    x = x.float().contiguous()
    rows, dim = x.shape
    l3 = torch.empty(rows, 3 * dim, dtype=torch.bfloat16, device=x.device)
    r3 = torch.empty(rows, 3 * dim, dtype=torch.bfloat16, device=x.device)
    _lib.check(lib.pgica_split3_bf16(_p(x), rows, dim, _p(l3), _p(r3), _stream()))
    return l3, r3


def ntxent_small_split(a_left3, b_right3, dim, inv_tau, reduce_mean=True):
    """ntxent_small on split fp32 operands: similarity over depth 3*dim, gradients (B, dim) fp32."""
    _need_cuda(a_left3, b_right3)
    lib = _lib.load()
    n = a_left3.shape[0]
    f32 = dict(dtype=torch.float32, device=a_left3.device)
    loss = torch.empty((), **f32)
    lse_row, lse_col = torch.empty(n, **f32), torch.empty(n, **f32)
    da, db = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
    _lib.check(lib.pgica_ntxent_small_split(_p(a_left3), _p(b_right3), n, dim, float(inv_tau), 1 if reduce_mean else 0,
                                            _p(loss), _p(lse_row), _p(lse_col), _p(da), _p(db), _stream()))
    return loss, lse_row, lse_col, da, db


# ----------------------------------------------------------------------------------------- SURVEY 8(f) row 2
def grad_norm_clip(grads, max_norm, clip=True):
    """Global L2 norm of a list of gradient tensors (fp32 / bf16, contiguous), finite check and in-place clip in three
    launches (pgica_grad_norm_clip).  Returns a (3,) fp32 device tensor: total_norm, clip_coef, is_finite."""
    grads = [g for g in grads if g is not None and g.numel() > 0]
    if not grads:
        raise ValueError("grad_norm_clip: no gradients")
    _need_cuda(*grads)
    for g in grads:
        if g.dtype not in (torch.float32, torch.bfloat16) or not g.is_contiguous():
            raise ValueError("grad_norm_clip: gradients must be contiguous fp32 or bf16 tensors")
    lib = _lib.load()
    n = len(grads)
    ptrs = (ctypes.c_void_p * n)(*[g.data_ptr() for g in grads])
    numels = (ctypes.c_int64 * n)(*[g.numel() for g in grads])
    kinds = (ctypes.c_int32 * n)(*[1 if g.dtype == torch.bfloat16 else 0 for g in grads])
    # the workspace (chunk table + partial sums) is kept for the next call on the same tensors: optimiser steps
    # clip the same gradient buffers every time, and the table then need not be rebuilt and uploaded
    key = tuple((g.data_ptr(), g.numel(), g.dtype) for g in grads)
    cached = _GRADCLIP_CACHE.get("entry")
    flags = 1 if clip else 0
    if cached is not None and cached[0] == key:
        ws = cached[1]
        flags |= 2
    else:
        need = ctypes.c_size_t(0)
        _lib.check(lib.pgica_grad_norm_clip_workspace_bytes(numels, n, ctypes.byref(need)))
        ws = _ws(need.value, grads[0].device)
        _GRADCLIP_CACHE["entry"] = (key, ws)
    stats = torch.empty(3, dtype=torch.float32, device=grads[0].device)
    _lib.check(lib.pgica_grad_norm_clip(ptrs, numels, kinds, n, float(max_norm), flags, _p(stats), _p(ws),
                                        ws.numel(), _stream()))
    return stats


_GRADCLIP_CACHE = {}


def adamw_step(params, grads, exp_avgs, exp_avg_sqs, steps, lr, beta1, beta2, eps, weight_decay, grad_stats=None):
    """One AdamW step (decoupled weight decay, torch's single-tensor arithmetic) over lists of contiguous fp32 tensors
    of one device, in place, in two launches (pgica_adamw_step): p, exp_avg and exp_avg_sq updated, then every 0-dim
    fp32 `steps[i]` incremented.  `grad_stats` (optional): the (3,) tensor of grad_norm_clip(..., clip=False); the
    update then runs on g * grad_stats[1], and writes nothing at all when grad_stats[2] == 0 (non-finite norm)."""
    n = len(params)
    if n == 0:
        return
    if not (len(grads) == len(exp_avgs) == len(exp_avg_sqs) == len(steps) == n):
        raise ValueError("adamw_step: params, grads, exp_avgs, exp_avg_sqs and steps must have the same length")
    _need_cuda(*params, *grads, *exp_avgs, *exp_avg_sqs, *steps, grad_stats)
    dev = params[0].device
    for i in range(n):
        p, quad = params[i], (params[i], grads[i], exp_avgs[i], exp_avg_sqs[i])
        for t in quad:
            if t.dtype != torch.float32 or not t.is_contiguous() or t.layout != torch.strided:
                raise ValueError("adamw_step: tensor %d: params, grads and state must be contiguous fp32" % i)
            if t.numel() != p.numel() or t.device != dev:
                raise ValueError("adamw_step: tensor %d: numel or device differs from its parameter" % i)
        if steps[i].dtype != torch.float32 or steps[i].numel() != 1 or steps[i].device != dev:
            raise ValueError("adamw_step: tensor %d: step must be a one-element fp32 tensor on the parameter's device" % i)
    if grad_stats is not None and (grad_stats.dtype != torch.float32 or grad_stats.numel() < 3
                                   or not grad_stats.is_contiguous() or grad_stats.device != dev):
        raise ValueError("adamw_step: grad_stats must be the (3,) fp32 output of grad_norm_clip on the same device")
    lib = _lib.load()
    ptrs = lambda ts: (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])
    numels = (ctypes.c_int64 * n)(*[p.numel() for p in params])
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_adamw_workspace_bytes(n, ctypes.byref(need)))
    ws = _ws(need.value, dev)
    _lib.check(lib.pgica_adamw_step(ptrs(params), ptrs(grads), ptrs(exp_avgs), ptrs(exp_avg_sqs), ptrs(steps), numels, n,
                                    float(lr), float(beta1), float(beta2), float(eps), float(weight_decay),
                                    _p(grad_stats), _p(ws), ws.numel(), _stream()))


# ----------------------------------------------------------------------------------------- compacted Stage-2 head
class CompactRows:
    """What the forward of the compacted head keeps for the backward (device tensors + host counts)."""
    __slots__ = ("hidden_c", "label_c", "lse_c", "index", "counts", "row_weight", "shapes", "n", "length_normalize",
                 "lse", "ztgt")


def lmhead_compact_fwd(hiddens, weight_bf16, labels, masks, length_normalize=False):
    """Sequence log-probs of one or more sequence sets (e.g. preferred, rejected) against ONE LM-head weight, computed
    on the scored rows only: hiddens[s] (B_s, T_s, d) fp32 or bf16, labels[s] (B_s, T_s), masks[s] (B_s, T_s) or None.
    The scored rows of all sets are gathered (and cast to bf16) into one dense matrix, so the LM-head GEMM runs once
    over sum_s n_s rows instead of sum_s B_s*T_s.  One host read (the row counts).  -> ([seq_logp_s], CompactRows)"""
    _need_cuda(weight_bf16, *hiddens, *labels, *[m for m in masks if m is not None])
    lib = _lib.load()
    dev = weight_bf16.device
    V, d = weight_bf16.shape
    f32 = dict(dtype=torch.float32, device=dev)
    nset = len(hiddens)
    counts_dev = torch.empty(nset, dtype=torch.int32, device=dev)
    index, row_weight, row_label, shapes, srcs = [], [], [], [], []
    for s in range(nset):
        h = hiddens[s]
        if h.dim() != 3 or h.shape[-1] != d:
            raise ValueError("lmhead_compact_fwd: hidden (nseq, T, d) expected")
        if h.dtype not in (torch.float32, torch.bfloat16):
            h = h.float()
        h = h.contiguous()
        nseq, T, _ = h.shape
        rl, rw = prep_rows(labels[s], masks[s], V)
        idx = torch.empty(nseq * T, dtype=torch.int32, device=dev)
        _lib.check(lib.pgica_compact_rows(_p(rw), nseq * T, _p(idx), ctypes.c_void_p(counts_dev.data_ptr() + 4 * s),
                                          _stream()))
        index.append(idx), row_weight.append(rw), row_label.append(rl), shapes.append((nseq, T)), srcs.append(h)
    counts = [int(c) for c in counts_dev.tolist()]  # the one device->host read of the compacted path
    n = sum(counts)
    ctx = CompactRows()
    ctx.index, ctx.counts, ctx.row_weight, ctx.shapes, ctx.n = index, counts, row_weight, shapes, n
    ctx.length_normalize = bool(length_normalize)
    ctx.hidden_c = torch.empty(max(n, 1), d, dtype=torch.bfloat16, device=dev)
    ctx.label_c = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    ctx.lse_c = torch.zeros(max(n, 1), **f32)
    ztgt_c = torch.zeros(max(n, 1), **f32)
    off = 0
    for s in range(nset):
        if counts[s]:
            _lib.check(lib.pgica_gather_rows_bf16(_p(srcs[s]), 1 if srcs[s].dtype == torch.bfloat16 else 0,
                                                  _p(index[s]), counts[s], d,
                                                  ctypes.c_void_p(ctx.hidden_c.data_ptr() + 2 * d * off),
                                                  _p(row_label[s]), ctypes.c_void_p(ctx.label_c.data_ptr() + 4 * off),
                                                  _stream()))
        off += counts[s]
    if n:
        need = ctypes.c_size_t(0)
        _lib.check(lib.pgica_gemm_lse_workspace_bytes(n, V, d, ctypes.byref(need)))
        ws = _ws(need.value, dev)
        _lib.check(lib.pgica_gemm_lse(_p(ctx.hidden_c), _p(weight_bf16), n, V, d, 1.0, _p(ctx.label_c), 0,
                                      _p(ctx.lse_c), _p(ztgt_c), _p(ws), need.value, _stream()))
    seqs, off = [], 0
    ctx.lse, ctx.ztgt = [], []
    for s in range(nset):
        nseq, T = shapes[s]
        lse = torch.empty(nseq * T, **f32)
        ztgt = torch.empty(nseq * T, **f32)
        for src, dst in ((ctx.lse_c, lse), (ztgt_c, ztgt)):
            _lib.check(lib.pgica_scatter_u32(ctypes.c_void_p(src.data_ptr() + 4 * off), _p(index[s]), counts[s],
                                             _p(dst), nseq * T, _stream()))
        seqs.append(seq_reduce(lse, ztgt, row_weight[s], nseq, T, length_normalize))
        ctx.lse.append(lse), ctx.ztgt.append(ztgt)
        off += counts[s]
    return seqs, ctx


def lmhead_compact_bwd(ctx, weight_bf16, grad_seqs, need_dhidden=True, need_dweight=True, dhidden_dtypes=None,
                       dweight_dtype=torch.float32):
    """Backward of lmhead_compact_fwd: ONE dual-kernel launch over the compacted rows of all sequence sets.
    -> ([dhidden_s] in the (B_s, T_s, d) layout, zeros at unscored rows; dweight (V, d))"""
    lib = _lib.load()
    dev = weight_bf16.device
    V, d = weight_bf16.shape
    n, nset = ctx.n, len(ctx.shapes)
    dhidden_dtypes = dhidden_dtypes or [torch.float32] * nset
    if n == 0:
        dhs = [torch.zeros(ns, T, d, dtype=dt, device=dev) for (ns, T), dt in zip(ctx.shapes, dhidden_dtypes)]
        return (dhs if need_dhidden else None), (torch.zeros(V, d, dtype=dweight_dtype, device=dev)
                                                 if need_dweight else None)
    ncoef_c = torch.empty(n, dtype=torch.float32, device=dev)
    off = 0
    for s in range(nset):
        nseq, T = ctx.shapes[s]
        coef = row_coef(grad_seqs[s], ctx.row_weight[s], nseq, T, ctx.length_normalize, -1.0)
        _lib.check(lib.pgica_gather_u32(_p(coef), _p(ctx.index[s]), ctx.counts[s],
                                        ctypes.c_void_p(ncoef_c.data_ptr() + 4 * off), _stream()))
        off += ctx.counts[s]
    # the compacted dhidden is fp32 when any consumer wants fp32 (the trainer's hidden states are fp32)
    dhc_dtype = torch.bfloat16 if all(dt == torch.bfloat16 for dt in dhidden_dtypes) else torch.float32
    dhc = torch.empty(n, d, dtype=dhc_dtype, device=dev) if need_dhidden else None
    dw = torch.empty(V, d, dtype=dweight_dtype, device=dev) if need_dweight else None
    need = ctypes.c_size_t(0)
    _lib.check(lib.pgica_lmhead_rows_workspace_bytes(n, d, V, ctypes.byref(need)))
    ws = _ws(need.value, dev)
    _lib.check(lib.pgica_lmhead_rows_bwd(_p(ctx.hidden_c), _p(weight_bf16), _p(ctx.label_c), _p(ctx.lse_c), _p(ncoef_c),
                                         n, d, V, _p(dhc), 1 if dhc_dtype == torch.bfloat16 else 0, _p(dw),
                                         1 if dweight_dtype == torch.bfloat16 else 0, _p(ws), ws.numel(), _stream()))
    dhs = None
    if need_dhidden:
        dhs, off = [], 0
        for s in range(nset):
            nseq, T = ctx.shapes[s]
            dh = torch.empty(nseq, T, d, dtype=dhidden_dtypes[s], device=dev)
            _lib.check(lib.pgica_scatter_rows(ctypes.c_void_p(dhc.data_ptr() + dhc.element_size() * d * off),
                                              1 if dhc_dtype == torch.bfloat16 else 0, _p(ctx.index[s]),
                                              ctx.counts[s], d, _p(dh), 1 if dh.dtype == torch.bfloat16 else 0,
                                              nseq * T, _stream()))
            dhs.append(dh)
            off += ctx.counts[s]
    return dhs, dw


# ----------------------------------------------------------------------------------------- SURVEY 8(f) rows 3, 4
def xattn_ln_fwd(x, u, w, out_bias, gamma, beta, eps):
    """y = LayerNorm(x + out_bias + sum_h w[..., h] * u[:, h]) (pgica_xattn_ln_fwd).  -> (y, mean, rstd)"""
    _need_cuda(x, u, w, out_bias, gamma, beta)
    lib = _lib.load()
    B, T, E = x.shape
    H = u.shape[1]
    y = torch.empty_like(x)
    mean = torch.empty(B * T, dtype=torch.float32, device=x.device)
    rstd = torch.empty(B * T, dtype=torch.float32, device=x.device)
    _lib.check(lib.pgica_xattn_ln_fwd(_p(x), _p(u), _p(w), _p(out_bias), _p(gamma), _p(beta), B, T, E, H, float(eps), _p(y),
                                      _p(mean), _p(rstd), _stream()))
    return y, mean, rstd


def xattn_ln_bwd(dy, x, u, w, out_bias, gamma, mean, rstd):
    """-> (dx, du, dgamma_part [B, E], dbeta_part [B, E], dpre_sum_part [B, E])"""
    lib = _lib.load()
    B, T, E = x.shape
    H = u.shape[1]
    f32 = dict(dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x)
    du = torch.empty(B, H, E, **f32)
    dg, db, dp = torch.empty(B, E, **f32), torch.empty(B, E, **f32), torch.empty(B, E, **f32)
    _lib.check(lib.pgica_xattn_ln_bwd(_p(dy), _p(x), _p(u), _p(w), _p(out_bias), _p(gamma), _p(mean), _p(rstd), B, T, E, H,
                                      _p(dx), _p(du), _p(dg), _p(db), _p(dp), _stream()))
    return dx, du, dg, db, dp


def ln_l2norm_fwd(z, gamma, beta, eps_ln, eps_norm):
    """e = LayerNorm(z), n = e / max(||e||, eps_norm) in one launch.  -> (e, n, stats [rows, 3])"""
    _need_cuda(z, gamma, beta)
    lib = _lib.load()
    rows, D = z.shape
    e, n = torch.empty_like(z), torch.empty_like(z)
    stats = torch.empty(rows, 3, dtype=torch.float32, device=z.device)
    _lib.check(lib.pgica_ln_l2norm_fwd(_p(z), _p(gamma), _p(beta), rows, D, float(eps_ln), float(eps_norm), _p(e), _p(n),
                                       _p(stats), _stream()))
    return e, n, stats


def ln_l2norm_bwd(z, gamma, beta, stats, de, dn):
    """-> (dz, dgamma_part [ceil(rows / 8), D], dbeta_part)"""
    lib = _lib.load()
    rows, D = z.shape
    nb = (rows + 7) // 8
    dz = torch.empty_like(z)
    dg = torch.empty(nb, D, dtype=torch.float32, device=z.device)
    db = torch.empty(nb, D, dtype=torch.float32, device=z.device)
    _lib.check(lib.pgica_ln_l2norm_bwd(_p(z), _p(gamma), _p(beta), _p(stats), _p(de), _p(dn), rows, D, _p(dz), _p(dg),
                                       _p(db), _stream()))
    return dz, dg, db


# ----------------------------------------------------------------------------------------- device guard
def _device_guard(fn):
    """Run `fn` with the device of its first CUDA tensor argument current: the stream handed to the C ABI
    (`_stream()`) and every allocation then belong to the tensors' device, whatever device the caller had selected."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for a in args:
            if isinstance(a, (list, tuple)) and a:
                a = a[0]
            if isinstance(a, torch.Tensor) and a.is_cuda:
                dev = a.device
                break
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


for _name, _fn in list(globals().items()):
    if callable(_fn) and getattr(_fn, "__module__", None) == __name__ and not _name.startswith("_") \
            and _name not in ("mask_kind", "ntxent_small_supported", "CompactRows"):
        globals()[_name] = _device_guard(_fn)
del _name, _fn
