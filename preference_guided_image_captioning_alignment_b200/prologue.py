"""SURVEY.md §8(f) rows 3 and 4: the pieces of the reference model right next to the two loss heads, fused.

Row 4 — `CaptionDecoder`'s cross-attention (pkg/models/model.py:528-535, 594-601) attends to ONE key/value token (the
projected image), so softmax over keys is 1 and `attention_norm(text + attended)` is a LayerNorm of a broadcast add:
`collapsed_cross_attention_ln`.  Attention dropout (training) survives as a keep-mask per (batch, position, head).

Row 3 — the projection heads end in a LayerNorm whose output the model L2-normalises for the contrastive head
(model.py:136-142, 338-344, 826-829): `ln_l2norm` gives both tensors from one launch, forward and backward.

`fuse_cross_attention` / `fuse_projection_tail` wire them into live reference modules WITHOUT touching the module tree
or the model's forward: the patched sub-modules hand a small carrier object (or tensor subclass) to the very next
operation of the reference code (`text + attended` -> `attention_norm(...)`;  `F.normalize(embeddings)`), which is
where the fused kernel runs.  Everything else that touches the carriers sees ordinary tensors.
"""
import types

import torch
import torch.nn as nn
import torch.nn.functional as TF

from . import functional as F


# ============================================================================================ row 4
class _XAttnLN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, u, w, out_bias, gamma, beta, eps):
        x, u = x.contiguous(), u.contiguous()
        w = None if w is None else w.contiguous()
        y, mean, rstd = F.xattn_ln_fwd(x, u, w, out_bias, gamma, beta, eps)
        ctx.save_for_backward(x, u, w, out_bias, gamma, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, u, w, out_bias, gamma, mean, rstd = ctx.saved_tensors
        dx, du, dg, db, dp = F.xattn_ln_bwd(dy.contiguous().float(), x, u, w, out_bias, gamma, mean, rstd)
        return dx, du, None, (dp.sum(0) if out_bias is not None else None), dg.sum(0), db.sum(0), None


def collapsed_cross_attention_ln(text: torch.Tensor, vision: torch.Tensor, mha: nn.MultiheadAttention,
                                 norm: nn.LayerNorm, keep_weights: torch.Tensor = None) -> torch.Tensor:
    """norm(text + mha(query=text, key=vision, value=vision)[0]) for a single key/value token.

    text (B, T, E) fp32, vision (B, 1, E) or (B, E).  In training with mha.dropout > 0 a keep-mask is drawn per
    (batch, position, head) — the weights nn.MultiheadAttention would apply to its (all-ones) attention matrix — unless
    `keep_weights` (B, T, H), already scaled by 1 / (1 - p), is given.  Differentiable w.r.t. text, vision and every
    parameter the reference block would train (the query / key projections get exact zeros, as they do there)."""
    B, T, E = text.shape
    H = mha.num_heads
    hd = E // H
    if not mha._qkv_same_embed_dim:
        raise ValueError("collapsed_cross_attention_ln expects a MultiheadAttention with one in_proj_weight")
    vis = vision.reshape(B, E).to(text.dtype)
    wv = mha.in_proj_weight[2 * E:]
    v = vis @ wv.t()
    if mha.in_proj_bias is not None:
        v = v + mha.in_proj_bias[2 * E:]
    wo = mha.out_proj.weight
    p = float(mha.dropout) if mha.training else 0.0
    if keep_weights is None and p > 0.0:
        keep_weights = (torch.rand(B, T, H, device=text.device) >= p).to(torch.float32) / (1.0 - p)
    if keep_weights is None:
        u = (v @ wo.t()).unsqueeze(1)                                             # (B, 1, E): heads already summed
    else:
        u = torch.einsum("bhd,ehd->bhe", v.view(B, H, hd), wo.view(E, H, hd))     # (B, H, E): one slice per head
        keep_weights = keep_weights.to(torch.float32)                             # a bool / fp16 / fp64 mask as well
    return _XAttnLN.apply(text.float(), u.float(), keep_weights, mha.out_proj.bias, norm.weight, norm.bias, norm.eps)


class CollapsedAttention:
    """What the patched cross-attention returns as `attended`: the block, still unevaluated.  `text + attended`
    (model.py:601) turns it into a PendingResidual, which the patched attention_norm evaluates in one fused launch."""

    def __init__(self, mha, vision, shape, device):
        self.mha, self.vision, self.shape, self.device = mha, vision, torch.Size(shape), device
        self.dtype = torch.float32

    def __radd__(self, text):
        return PendingResidual(text, self)

    __add__ = __radd__

    def materialize(self):
        """The dense (B, T, E) attended tensor, for code that wants it after all."""
        B, T, E = self.shape
        zeros = torch.zeros(B, T, E, device=self.device)
        return type(self.mha).forward(self.mha, zeros, self.vision, self.vision)[0]


class PendingResidual:
    def __init__(self, text, attended):
        self.text, self.attended = text, attended
        self.shape, self.device, self.dtype = text.shape, text.device, text.dtype

    def materialize(self):
        return self.text + self.attended.materialize()


def _xattn_forward(self, query, key, value, key_padding_mask=None, need_weights=True, attn_mask=None, **kw):
    E = self.embed_dim
    dropout = self.training and self.dropout > 0.0
    ok = (self.batch_first and key is value and query.is_cuda and query.dim() == 3 and key.dim() == 3 and
          key.shape[1] == 1 and key_padding_mask is None and attn_mask is None and self._qkv_same_embed_dim and
          self.bias_k is None and not self.add_zero_attn and query.dtype == torch.float32 and
          E % 4 == 0 and E <= 4096 and not (dropout and self.num_heads > 32))    # the kernel's limits
    if not ok:
        return type(self).forward(self, query, key, value, key_padding_mask=key_padding_mask, need_weights=need_weights,
                                  attn_mask=attn_mask, **kw)
    return CollapsedAttention(self, key, query.shape, query.device), None


def _fusable_norm(norm):
    """A LayerNorm the kernels can apply: an fp32 weight and bias over the last dimension."""
    return (norm.weight is not None and norm.bias is not None and norm.weight.dtype == torch.float32 and
            norm.bias.dtype == torch.float32 and len(norm.normalized_shape) == 1)


def _norm_forward(self, inp):
    if isinstance(inp, PendingResidual) and _fusable_norm(self):
        att = inp.attended
        return collapsed_cross_attention_ln(inp.text, att.vision, att.mha, self)
    if isinstance(inp, (CollapsedAttention, PendingResidual)):
        inp = inp.materialize()
    return TF.layer_norm(inp, self.normalized_shape, self.weight, self.bias, self.eps)


def fuse_cross_attention(decoder):
    """Patch `decoder.cross_attention` / `decoder.attention_norm` (a reference CaptionDecoder) on the instances."""
    mha, norm = decoder.cross_attention, decoder.attention_norm
    if not isinstance(mha, nn.MultiheadAttention) or not isinstance(norm, nn.LayerNorm):
        raise TypeError("fuse_cross_attention expects nn.MultiheadAttention + nn.LayerNorm")
    if "forward" not in mha.__dict__:
        mha.forward = types.MethodType(_xattn_forward, mha)
    if "forward" not in norm.__dict__:
        norm.forward = types.MethodType(_norm_forward, norm)
    return decoder


def unfuse_cross_attention(decoder):
    decoder.cross_attention.__dict__.pop("forward", None)
    decoder.attention_norm.__dict__.pop("forward", None)
    return decoder


# ============================================================================================ row 3
class _LnL2Norm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, gamma, beta, eps_ln, eps_norm):
        z = z.contiguous().float()
        e, n, stats = F.ln_l2norm_fwd(z, gamma, beta, eps_ln, eps_norm)
        ctx.save_for_backward(z, gamma, beta, stats)
        return e, n

    @staticmethod
    def backward(ctx, de, dn):
        z, gamma, beta, stats = ctx.saved_tensors
        de = None if de is None else de.contiguous().float()
        dn = None if dn is None else dn.contiguous().float()
        if de is None and dn is None:
            return None, None, None, None, None
        dz, dg, db = F.ln_l2norm_bwd(z, gamma, beta, stats, de, dn)
        return dz, dg.sum(0), db.sum(0), None, None


def ln_l2norm(z: torch.Tensor, norm: nn.LayerNorm, eps_norm: float = 1e-12):
    """(LayerNorm(z), F.normalize(LayerNorm(z), dim=-1)) for (rows, D) inputs: the tail of the projection heads and
    the normalisation in front of the contrastive head (model.py:141, 343, 828-829), one launch each way."""
    if z.shape[-1] > 2048:
        raise ValueError(f"ln_l2norm: dim {z.shape[-1]} > 2048, the largest row its backward takes")
    return _LnL2Norm.apply(z, norm.weight, norm.bias, norm.eps, eps_norm)


class NormalizedCarrier(torch.Tensor):
    """The LayerNorm output of a projection head that already knows its L2-normalised twin: F.normalize(t, p=2, dim=-1)
    on it returns the twin (computed by the same launch); every other operation sees a plain tensor."""

    @classmethod
    def __torch_function__(cls, func, types_, args=(), kwargs=None):
        kwargs = kwargs or {}
        if func is TF.normalize and args and isinstance(args[0], NormalizedCarrier):
            t = args[0]
            p = kwargs.get("p", args[1] if len(args) > 1 else 2.0)
            dim = kwargs.get("dim", args[2] if len(args) > 2 else 1)
            eps = kwargs.get("eps", args[3] if len(args) > 3 else 1e-12)
            out = kwargs.get("out", args[4] if len(args) > 4 else None)
            twin = getattr(t, "_pgica_normalized", None)
            if twin is not None and out is None and float(p) == 2.0 and dim in (-1, t.dim() - 1) and \
                    float(eps) == 1e-12:
                return twin
        from torch.utils._pytree import tree_map
        plain = lambda x: x.as_subclass(torch.Tensor) if isinstance(x, NormalizedCarrier) else x
        with torch._C.DisableTorchFunctionSubclass():
            return func(*tree_map(plain, args), **tree_map(plain, kwargs))


def _proj_norm_forward(self, z):
    if not (z.is_cuda and z.dim() == 2 and z.dtype == torch.float32 and z.shape[-1] <= 1024 and _fusable_norm(self)):
        return TF.layer_norm(z, self.normalized_shape, self.weight, self.bias, self.eps)
    e, n = ln_l2norm(z, self)
    out = e.as_subclass(NormalizedCarrier)
    n._pgica_unit_norm = True  # read by losses.ContrastiveLoss: unit-norm rows by construction
    out._pgica_normalized = n
    return out


def fuse_projection_tail(encoder):
    """Patch the final LayerNorm of `encoder.projection` (a reference VisionEncoder / TextEncoder) on the instance."""
    last = encoder.projection[-1]
    if not isinstance(last, nn.LayerNorm):
        raise TypeError("fuse_projection_tail expects projection[-1] to be nn.LayerNorm")
    if "forward" not in last.__dict__:
        last.forward = types.MethodType(_proj_norm_forward, last)
    return encoder


def unfuse_projection_tail(encoder):
    encoder.projection[-1].__dict__.pop("forward", None)
    return encoder
