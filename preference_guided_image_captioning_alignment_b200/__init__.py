"""B200-native (sm_100a) fused alignment loss heads: Stage-1 NT-Xent and Stage-2 DPO.

Drop-in for the loss-head hot path of A-SHOJAEI/preference-guided-image-captioning-alignment:

    losses.ContrastiveLoss / losses.PreferenceLoss         <- pkg/models/model.py:957-1085 (what the trainer uses)
    components.ContrastiveLoss / DPOPreferenceLoss /
        TemperatureScaledSimilarity / compute_sequence_logprobs   <- pkg/models/components.py
    components.FusedDPOHead / lmhead_sequence_logprobs      hidden-state level: logits never materialised
    graphs.GraphedDPOStep / GraphedContrastiveStep          one or two CUDA-graph launches per head step (forward + backward)
    distributed.global_ntxent / GlobalContrastiveLoss       NT-Xent with negatives from every rank
    scoring.compute_similarity / paired_scores              retrieval-style scoring on the similarity kernel
    optim.FusedAdamW                                        AdamW with the NaN-safe global-norm clip folded into one update pass
    install()                                               rebinds the reference's names to the above

Everything computes in hand-written CUDA (csrc/, exported through the C ABI in include/pgica.h).  There is no
CPU or PyTorch fallback: on a machine without a B200 the ops raise.
"""
from . import _lib  # noqa: F401  (ctypes binding; the library itself is loaded on first use)
from .components import (DPOPreferenceLoss, FusedDPOHead, NaNSafeGradientNorm, TemperatureScaledSimilarity,  # noqa: F401
                         compute_sequence_logprobs, lmhead_sequence_logprobs)
from .graphs import GraphedContrastiveStep, GraphedDPOStep  # noqa: F401
from .install import fuse_model, install, unfuse_model, uninstall  # noqa: F401
from .prologue import collapsed_cross_attention_ln, ln_l2norm  # noqa: F401
from .losses import ContrastiveLoss, DeferredLoss, LazyLogits, PreferenceLoss  # noqa: F401
from .optim import FusedAdamW  # noqa: F401
from .scoring import compute_similarity, paired_scores, retrieval_ranks  # noqa: F401

__all__ = ["ContrastiveLoss", "PreferenceLoss", "DPOPreferenceLoss", "FusedDPOHead", "TemperatureScaledSimilarity",
           "compute_sequence_logprobs", "lmhead_sequence_logprobs", "LazyLogits", "GraphedDPOStep", "GraphedContrastiveStep", "NaNSafeGradientNorm",
           "install", "uninstall", "fuse_model", "unfuse_model", "collapsed_cross_attention_ln", "ln_l2norm", "DeferredLoss", "compute_similarity", "paired_scores", "retrieval_ranks",
           "FusedAdamW"]
