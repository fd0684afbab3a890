"""Retrieval-style scoring on the similarity kernel (SURVEY.md §8(f) row 5).

    compute_similarity   PreferenceGuidedCaptioningModel.compute_similarity, pkg/models/model.py:925-954:
                         (B, B) matrix  image_embeddings @ text_embeddings.T / temperature
    paired_scores        the per-pair score the CLIP-score loop collects one `.item()` at a time
                         (pkg/evaluation/metrics.py:380-439: logits_per_image of ONE image and ONE caption =
                         logit_scale * cos(image, caption)), for a whole batch in one launch
    retrieval_ranks_both rank of the matching caption among all captions and of the matching image among all images,
                         any number of captions per image (pgica_retrieval_ranks: no score matrix is stored)
    retrieval_ranks      the image -> caption half of it, caption i matching image i
    retrieval_recall     recall@k in both directions from those ranks

All of them run on `pgica_similarity` / `pgica_gemm_lse` / `pgica_retrieval_ranks` (tcgen05 GEMM, csrc/gemm_lse.cu).  fp32 embeddings go in as their
two-term bf16 split (depth 3*D), so scores agree with the reference's fp32 matmul to ~1e-6 relative; bf16 embeddings
are used as they are.  Forward-only (evaluation); no CPU path.
"""
import torch

from . import functional as F


def _operands(a, b):
    if a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16:
        return a.contiguous(), b.contiguous()
    al, _ = F.split3(a)
    _, br = F.split3(b)
    return al, br


@torch.no_grad()
def compute_similarity(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor,
                       temperature: float = 0.07) -> torch.Tensor:
    """(B_i, D), (B_t, D) embeddings as given (the model normalises them, model.py:826-829) -> (B_i, B_t) fp32
    similarity / temperature."""
    a, b = _operands(image_embeddings, text_embeddings)
    return F.similarity(a, b, 1.0 / float(temperature))


@torch.no_grad()
def paired_scores(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor, logit_scale: float = 100.0,
                  normalize: bool = True) -> torch.Tensor:
    """score[i] = logit_scale * <img_i, txt_i> (cosine when `normalize`): the CLIP-score of pair i.  (B,) fp32.
    Uses the diagonal gather of the GEMM+LSE kernel, so the (B, B) matrix is never written."""
    if normalize:
        _, _, _, al, _ = F.rownorm_fwd(image_embeddings, 1e-12, split=True)
        _, _, _, _, br = F.rownorm_fwd(text_embeddings, 1e-12, split=True)
    else:
        al, br = _operands(image_embeddings, text_embeddings)
    _, diag = F.gemm_lse(al, br, float(logit_scale), None, 0, want_tgt=True)
    return diag


def _owners(text_to_image, n_img, n_txt):
    """Validated int32 owner vector (or None for the default pairing); raises ValueError before any launch."""
    if text_to_image is None:
        return None
    if not isinstance(text_to_image, torch.Tensor) or text_to_image.dtype not in (torch.int32, torch.int64):
        raise ValueError("text_to_image must be an int32 or int64 tensor")
    if text_to_image.shape != (n_txt,):
        raise ValueError(f"text_to_image has shape {tuple(text_to_image.shape)}, expected ({n_txt},)")
    lo, hi = (int(v) for v in torch.stack([text_to_image.min(), text_to_image.max()]).tolist())
    if lo < -1 or hi >= n_img:
        raise ValueError(f"text_to_image values must lie in [-1, {n_img}); got [{lo}, {hi}]")
    return text_to_image.to(torch.int32).contiguous()


@torch.no_grad()
def retrieval_ranks_both(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor,
                         text_to_image: torch.Tensor = None):
    """Ranks of the matching items in both directions, from two passes over the similarity tiles (pgica_retrieval_ranks);
    the (Ni, Nt) score matrix is never stored.  S = image_embeddings @ text_embeddings.T in fp32 as compute_similarity
    computes it; caption j belongs to image text_to_image[j] (-1: none; default: caption j to image j for j < Ni).

        image_rank[i] = #captions scoring above image i's best own caption (-1 if image i owns none)
        text_rank[j]  = #images scoring above caption j's own image (-1 if caption j has none)

    Strict '>': ties count for the positive.  Returns two int64 (Ni,), (Nt,) tensors on the device."""
    if image_embeddings.dim() != 2 or text_embeddings.dim() != 2:
        raise ValueError("embeddings must be 2-D (N, D)")
    n_img, n_txt = image_embeddings.shape[0], text_embeddings.shape[0]
    if n_img == 0 or n_txt == 0 or image_embeddings.shape[1] == 0:
        raise ValueError("retrieval ranks need at least one image, one caption and D > 0")
    if image_embeddings.shape[1] != text_embeddings.shape[1]:
        raise ValueError(f"embedding widths differ: {image_embeddings.shape[1]} vs {text_embeddings.shape[1]}")
    owners = _owners(text_to_image, n_img, n_txt)
    F._need_cuda(image_embeddings, text_embeddings, owners)
    a, b = _operands(image_embeddings, text_embeddings)
    image_rank, text_rank = F.retrieval_ranks(a, b, owners)
    return image_rank.long(), text_rank.long()


@torch.no_grad()
def retrieval_ranks(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor) -> torch.Tensor:
    """rank[i] = number of captions that score strictly higher than caption i for image i (0 = retrieved first);
    -1 for the images past the last caption."""
    return retrieval_ranks_both(image_embeddings, text_embeddings)[0]


@torch.no_grad()
def retrieval_recall(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor, text_to_image: torch.Tensor = None,
                     ks=(1, 5, 10)) -> dict:
    """Recall@k in both directions: {"image_to_text": {k: r}, "text_to_image": {k: r}} as Python floats (NaN when no
    item has a match).  Images that own no caption and captions without an image are left out of the denominators."""
    image_rank, text_rank = retrieval_ranks_both(image_embeddings, text_embeddings, text_to_image)
    ks = [int(k) for k in ks]
    counts = torch.stack([torch.stack([((r >= 0) & (r < k)).sum() for k in ks] + [(r >= 0).sum()])
                          for r in (image_rank, text_rank)]).tolist()  # one device-to-host read
    out = {}
    for name, row in zip(("image_to_text", "text_to_image"), counts):
        n = row[-1]
        out[name] = {k: (row[i] / n if n else float("nan")) for i, k in enumerate(ks)}
    return out


def model_compute_similarity(self, images, captions, caption_mask):
    """Bound over PreferenceGuidedCaptioningModel.compute_similarity by install(): same signature and result
    (pkg/models/model.py:925-954), the final matmul on the similarity kernel."""
    outputs = self(images=images, caption_ids=captions, caption_mask=caption_mask, mode="contrastive")
    img, txt = outputs["image_embeddings"], outputs["text_embeddings"]
    if not img.is_cuda:
        return torch.matmul(img, txt.t()) / self.temperature
    return compute_similarity(img, txt, self.temperature)
