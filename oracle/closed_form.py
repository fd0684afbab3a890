"""float64 numpy restatement of the reference loss heads, with analytic gradients.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Paths cite the reference repository,
"pkg/" = src/preference_guided_image_captioning_alignment/.
"""
import numpy as np

F64 = np.float64


def _logsumexp(z, axis):
    m = np.max(z, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return (m + np.log(np.sum(np.exp(z - m), axis=axis, keepdims=True))).squeeze(axis)


def l2_normalize(x, eps=1e-12):
    """F.normalize(x, p=2, dim=-1) — pkg/models/components.py:74-75, pkg/models/model.py:828-829."""
    x = np.asarray(x, F64)
    n = np.maximum(np.sqrt(np.sum(x * x, axis=-1, keepdims=True)), eps)
    return x / n, n


def l2_normalize_bwd(x, g, eps=1e-12):
    """Gradient of F.normalize(x, dim=-1) for the upstream gradient g: (g - u <u, g>) / ||x|| with u = x / ||x||.  A
    row with ||x|| < eps was divided by the constant eps (torch's clamp_min passes no gradient to the norm below its
    bound): g / eps, no projection."""
    x = np.asarray(x, F64)
    g = np.asarray(g, F64)
    u, n = l2_normalize(x, eps)
    proj = np.where(np.sqrt(np.sum(x * x, axis=-1, keepdims=True)) < eps, 0.0, np.sum(u * g, axis=-1, keepdims=True))
    return (g - u * proj) / n


def effective_temperature(temperature, clamp_tau, min_temp=0.1, max_temp=2.0):
    """torch.clamp(self.temperature, min_temp, max_temp) — pkg/models/components.py:78 (ctor :45-59).
    The trainer-facing loss (pkg/models/model.py:988) divides by the raw temperature."""
    return float(min(max(temperature, min_temp), max_temp)) if clamp_tau else float(temperature)


def ntxent(x, y, temperature, normalize=False, clamp_tau=False, reduction="mean", row_offset=0):
    """Symmetric NT-Xent / InfoNCE loss and its gradients.

    components variant: pkg/models/components.py:117-145 (normalize=True, clamp_tau=True, reduction mean|sum)
    trainer variant:    pkg/models/model.py:970-1000   (normalize=False, clamp_tau=False, mean)

    x: (b, D) rows i, y: (B, D) columns j; positives are (i, i + row_offset).  With b == B and
    row_offset == 0 this is the reference; b < B is one rank's row slice of the global-negatives extension.
    Returns dict(loss, lse_row, lse_col, dx, dy, sim) — sim = S, the (b, B) scaled similarity.
    """
    x = np.asarray(x, F64)
    y = np.asarray(y, F64)
    b, B = x.shape[0], y.shape[0]
    tau = effective_temperature(temperature, clamp_tau)
    if normalize:
        a, _ = l2_normalize(x)
        c, _ = l2_normalize(y)
    else:
        a, c = x, y
    S = a @ c.T / tau
    lse_r = _logsumexp(S, axis=1)
    lse_c = _logsumexp(S, axis=0)
    idx = np.arange(b)
    diag = S[idx, idx + row_offset]
    if b == B:
        col_term = np.sum(lse_c - diag)
    else:  # a row slice sees only part of every column: the column half of the loss is not defined locally
        col_term = np.nan
    row_term = np.sum(lse_r - diag)
    denom = B if reduction == "mean" else 1.0
    loss = 0.5 * (row_term + col_term) / denom
    onehot = np.zeros_like(S)
    onehot[idx, idx + row_offset] = 1.0
    dS = (np.exp(S - lse_r[:, None]) + np.exp(S - lse_c[None, :]) - 2.0 * onehot) / (2.0 * denom)
    da = dS @ c / tau
    dc = dS.T @ a / tau
    if normalize:
        dx, dy = l2_normalize_bwd(x, da), l2_normalize_bwd(y, dc)
    else:
        dx, dy = da, dc
    return dict(loss=loss, lse_row=lse_r, lse_col=lse_c, dx=dx, dy=dy, sim=S)


def token_logprobs(logits, labels):
    """log_softmax + gather at the shifted labels — pkg/models/components.py:339-352,
    pkg/models/model.py:1069-1079.  logits (B, T, V), labels (B, T) -> (B, T-1) log-probs, lse, z_tgt."""
    z = np.asarray(logits, F64)[:, :-1, :]
    yl = np.asarray(labels)[:, 1:]
    lse = _logsumexp(z, axis=-1)
    zt = np.take_along_axis(z, yl[..., None], axis=-1)[..., 0]
    return zt - lse, lse, zt


def sequence_logprobs(logits, labels, mask=None, length_normalize=False):
    """compute_sequence_logprobs (masked SUM, pkg/models/components.py:321-362) or
    PreferenceLoss._compute_log_probs (masked MEAN, pkg/models/model.py:1052-1085)."""
    lp, _, _ = token_logprobs(logits, labels)
    m = np.ones_like(lp) if mask is None else np.asarray(mask, F64)[:, 1:]
    s = np.sum(lp * m, axis=-1)
    if length_normalize:
        with np.errstate(invalid="ignore", divide="ignore"):
            s = s / np.sum(m, axis=-1)
    return s


def lm_head_logits(hidden, weight):
    """GPT2LMHeadModel.lm_head: nn.Linear without bias (transformers modeling_gpt2.py:651,706; reached from
    pkg/models/model.py:604-610).  hidden (B, T, d), weight (V, d) -> (B, T, V)."""
    return np.asarray(hidden, F64) @ np.asarray(weight, F64).T


def lmhead_sequence_logprobs(hidden, weight, labels, mask=None, length_normalize=False, grad_seq=None):
    """LM head + sequence log-prob, and — when grad_seq (B,) = dLoss/dseq_logp is given — the gradients
    dhidden (B, T, d) and dweight (V, d) (SURVEY.md Appendix A)."""
    h = np.asarray(hidden, F64)
    W = np.asarray(weight, F64)
    z = h @ W.T
    lp, lse, zt = token_logprobs(z, labels)
    Bn, T = np.asarray(labels).shape
    m = np.ones((Bn, T - 1), F64) if mask is None else np.asarray(mask, F64)[:, 1:]
    seq = np.sum(lp * m, axis=-1)
    lens = np.sum(m, axis=-1)
    if length_normalize:
        with np.errstate(invalid="ignore", divide="ignore"):
            seq = seq / lens
    out = dict(seq_logp=seq, lse=lse, z_tgt=zt, token_logp=lp)
    if grad_seq is not None:
        g = np.asarray(grad_seq, F64)[:, None] * m
        if length_normalize:
            g = g / lens[:, None]
        p = np.exp(z[:, :-1, :] - lse[..., None])
        dz = -p * g[..., None]
        yl = np.asarray(labels)[:, 1:]
        bi, ti = np.meshgrid(np.arange(Bn), np.arange(T - 1), indexing="ij")
        dz[bi, ti, yl] += g
        dh = np.zeros_like(h)
        dh[:, :-1, :] = dz @ W
        dW = np.einsum("btv,btd->vd", dz, h[:, :-1, :])
        out.update(dhidden=dh, dweight=dW)
    return out


def _logsigmoid(x):
    return -np.logaddexp(0.0, -x)


def _sigmoid(x):
    return np.exp(_logsigmoid(x))


def dpo_loss(pc, pr, rc=None, rr=None, beta=0.1, reference_free=False, label_smoothing=0.0):
    """DPOPreferenceLoss.forward — pkg/models/components.py:192-249.  Also the trainer-facing
    PreferenceLoss tail (pkg/models/model.py:1046-1048) when rc = rr = None.
    Returns dict(loss, metrics{5 keys}, d_pc, d_pr, d_rc, d_rr)."""
    pc = np.asarray(pc, F64)
    pr = np.asarray(pr, F64)
    pol = pc - pr
    if reference_free or rc is None:
        ref = np.zeros_like(pol)
    else:
        ref = np.asarray(rc, F64) - np.asarray(rr, F64)
    x = beta * (pol - ref)
    n = x.shape[0]
    if label_smoothing > 0:
        t = 1.0 - label_smoothing
        per = -(t * _logsigmoid(x) + (1.0 - t) * _logsigmoid(-x))
        dx = -(t * _sigmoid(-x) - (1.0 - t) * _sigmoid(x))
    else:
        per = -_logsigmoid(x)
        dx = -_sigmoid(-x)
    loss = per.mean()
    d_pc = beta * dx / n
    metrics = dict(
        dpo_loss=float(loss),
        reward_margin=float((pol - ref).mean()),
        reward_accuracy=float((pol > ref).astype(F64).mean()),
        policy_chosen_logprob=float(pc.mean()),
        policy_rejected_logprob=float(pr.mean()),
    )
    has_ref = not (reference_free or rc is None)
    return dict(loss=loss, metrics=metrics, d_pc=d_pc, d_pr=-d_pc,
                d_rc=(-d_pc if has_ref else None), d_rr=(d_pc if has_ref else None))


def preference_loss_from_logits(pref_logits, rej_logits, pref_labels, rej_labels, pref_mask, rej_mask, beta=0.1):
    """PreferenceLoss.forward — pkg/models/model.py:1016-1050 (length-normalised, no reference)."""
    lw = sequence_logprobs(pref_logits, pref_labels, pref_mask, length_normalize=True)
    ll = sequence_logprobs(rej_logits, rej_labels, rej_mask, length_normalize=True)
    return dpo_loss(lw, ll, beta=beta)["loss"], lw, ll


def dpo_head(hc, hr, W, yc, yr, mc=None, mr=None, ref=None, beta=0.1, length_normalize=False,
             label_smoothing=0.0):
    """Whole Stage-2 head at the hidden-state level: LM head -> sequence log-probs for chosen / rejected under
    the policy (and the frozen reference `ref` = dict(hc, hr, W)) -> DPO loss; plus policy gradients.
    Composition of lm_head (modeling_gpt2.py:706), components.py:321-362 and components.py:192-249."""
    fc = lmhead_sequence_logprobs(hc, W, yc, mc, length_normalize)
    fr = lmhead_sequence_logprobs(hr, W, yr, mr, length_normalize)
    rc = rr = None
    if ref is not None:
        rc = lmhead_sequence_logprobs(ref["hc"], ref["W"], yc, mc, length_normalize)["seq_logp"]
        rr = lmhead_sequence_logprobs(ref["hr"], ref["W"], yr, mr, length_normalize)["seq_logp"]
    head = dpo_loss(fc["seq_logp"], fr["seq_logp"], rc, rr, beta=beta, label_smoothing=label_smoothing)
    gc = lmhead_sequence_logprobs(hc, W, yc, mc, length_normalize, grad_seq=head["d_pc"])
    gr = lmhead_sequence_logprobs(hr, W, yr, mr, length_normalize, grad_seq=head["d_pr"])
    return dict(loss=head["loss"], metrics=head["metrics"], pc=fc["seq_logp"], pr=fr["seq_logp"], rc=rc, rr=rr,
                dhc=gc["dhidden"], dhr=gr["dhidden"], dW=gc["dweight"] + gr["dweight"])


def grad_norm_clip(grads, max_norm):
    """NaNSafeGradientNorm.forward (pkg/models/components.py:283-318) + torch.nn.utils.clip_grad_norm_ in float64:
    total L2 norm over all gradients (norm of the per-tensor norms, :300-303), finite flag (:306), and the gradients
    multiplied by min(1, max_norm / (total + 1e-6)) when finite, untouched otherwise (:308-315)."""
    grads = [np.asarray(g, dtype=np.float64) for g in grads]
    with np.errstate(over="ignore", invalid="ignore"):
        total = float(np.sqrt(sum(float(np.sum(g * g)) for g in grads)))
    finite = bool(np.isfinite(total))
    coef = min(1.0, max_norm / (total + 1e-6)) if finite else 1.0
    return {"total_norm": total, "is_finite": finite, "clip_coef": coef,
            "clipped": [g * coef if finite else g.copy() for g in grads]}
