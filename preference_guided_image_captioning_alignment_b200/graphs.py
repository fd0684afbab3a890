"""CUDA-graph capture of a whole DPO-head training step (forward + backward through the module API).

The head's step is ~20 short launches around three long ones; issued one by one from Python the host needs longer
to enqueue them than the B200 needs to run them (bench.py: 2.2 ms of host time against 1.7 ms of device time on
BASELINE config 2).  `GraphedDPOStep` records `FusedDPOHead.forward_stacked(...)` and its backward once into two CUDA
graphs over static input buffers and replays them: two `cudaGraphLaunch` calls per step, same kernels, same results.
The loss is copied to pinned host memory at the end of the FORWARD graph, so the host can read it (and go on to
enqueue the next step) while the backward graph is still running — the device never waits for the host.

    step = GraphedDPOStep(head, weight, ref_weight, hidden_like, labels_like, mask_like, ref_hidden_like, n_global)
    step.copy_inputs(hidden, labels, mask, ref_hidden)      # async copies into the static buffers
    step.launch()                                           # forward graph, event, backward graph
    value = step.loss_value()                               # waits for the forward graph only
    step.dweight, step.dhidden                              # gradients (valid once the stream has caught up)
"""
from typing import Optional

import torch


class GraphedDPOStep:
    def __init__(self, head, weight: torch.Tensor, ref_weight: Optional[torch.Tensor], hidden: torch.Tensor,
                 labels: torch.Tensor, mask: Optional[torch.Tensor], ref_hidden: Optional[torch.Tensor] = None,
                 n_global: Optional[int] = None, warmup: int = 2):
        if not hidden.is_cuda:
            raise RuntimeError("GraphedDPOStep needs CUDA tensors (there is no CPU path)")
        self.head = head
        self.weight = weight if weight.requires_grad else weight.detach().requires_grad_(True)
        self.ref_weight = ref_weight
        self.n_global = n_global
        # static inputs: the graphs read these addresses on every replay
        self.hidden = hidden.detach().clone().requires_grad_(True)
        self.labels = labels.clone()
        self.mask = None if mask is None else mask.clone()
        self.ref_hidden = None if ref_hidden is None else ref_hidden.detach().clone()
        self.loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
        self.forward_done = torch.cuda.Event()
        side = torch.cuda.Stream(device=hidden.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):  # first-use work (attribute setting, occupancy queries, allocator growth)
                loss, _ = self._forward()
                torch.autograd.grad(loss, (self.hidden, self.weight))
        torch.cuda.current_stream().wait_stream(side)
        self.fwd_graph = torch.cuda.CUDAGraph()
        self.bwd_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.fwd_graph):
            self.loss, self.metrics = self._forward()
            self.loss_host.copy_(self.loss.detach(), non_blocking=True)
        with torch.cuda.graph(self.bwd_graph, pool=self.fwd_graph.pool()):
            self.dhidden, self.dweight = torch.autograd.grad(self.loss, (self.hidden, self.weight))

    def _forward(self):
        return self.head.forward_stacked(self.hidden, self.weight, self.labels, self.mask, self.ref_hidden,
                                         self.ref_weight, self.n_global)

    def copy_inputs(self, hidden, labels=None, mask=None, ref_hidden=None):
        """Asynchronous copies (e.g. from pinned host memory) into the graphs' static input buffers."""
        with torch.no_grad():
            self.hidden.copy_(hidden, non_blocking=True)
            if labels is not None:
                self.labels.copy_(labels, non_blocking=True)
            if mask is not None and self.mask is not None:
                self.mask.copy_(mask, non_blocking=True)
            if ref_hidden is not None and self.ref_hidden is not None:
                self.ref_hidden.copy_(ref_hidden, non_blocking=True)

    def launch(self):
        """Enqueue the step on the current stream: forward (+ loss to pinned memory), then backward."""
        self.fwd_graph.replay()
        self.forward_done.record()
        self.bwd_graph.replay()

    def loss_value(self) -> float:
        """The step's loss as a Python float; waits for the forward graph only."""
        self.forward_done.synchronize()
        return self.loss_host.item()

    def replay(self) -> torch.Tensor:
        """launch() and return the loss as a device tensor (no host synchronisation)."""
        self.launch()
        return self.loss


# Row-bucket granularity of GraphedCompactDPOStep: one CTA-pair row block of the tensor-core kernels.
BUCKET_ROWS = 256


def scored_rows(mask: Optional[torch.Tensor], nseq: int, seqlen: int) -> int:
    """How many rows of a (nseq, seqlen) batch the Stage-2 head scores, from a HOST mask: row (b, t) is scored iff
    t < seqlen - 1 and mask[b, t + 1] != 0 (NaN counts), the rule of pgica_prep_rows.  mask None: every such row."""
    if seqlen < 2:
        return 0
    if mask is None:
        return nseq * (seqlen - 1)
    if mask.is_cuda:
        raise ValueError("scored_rows needs the mask in host memory (reading a device mask would synchronise)")
    if mask.dtype not in (torch.int64, torch.float32, torch.bool, torch.uint8, torch.int32):
        mask = mask.float()  # the dtype functional.mask_kind hands to the kernel
    return int((mask.reshape(nseq, seqlen)[:, 1:] != 0).sum())


def bucket_rows(n: int, granularity: int = BUCKET_ROWS) -> int:
    """Launch size for n scored rows: n rounded up to the granularity (at least one bucket)."""
    return max(1, -(-int(n) // granularity)) * granularity


class GraphedCompactDPOStep:
    """`GraphedDPOStep` on the scored rows only: the tensor work scales with the rows the masks score, not with 2*B*T.

    Each step's launches are sized by a row bucket (the scored rows of the host-side mask, rounded up to BUCKET_ROWS =
    256) and replayed from a forward / backward pair of CUDA graphs captured the first time that bucket is used; the
    exact row count is computed and consumed on the device (functional.lmhead_compact_fwd_bucketed / _bwd_bucketed).
    The inputs are pre-stacked like `GraphedDPOStep`'s (rows [0, B) chosen, [B, 2B) rejected); labels and masks go to
    `copy_inputs` as host (pinned) tensors, since the bucket is chosen from them.

        step = GraphedCompactDPOStep(head, weight, ref_weight, hidden_like, labels_like, mask_like, ref_hidden_like)
        step.copy_inputs(hidden, labels_pinned, mask_pinned, ref_hidden)
        step.launch()
        value = step.loss_value()       # raises if the device found more scored rows than the bucket holds
        step.dweight, step.dhidden      # same tensors whichever bucket ran

    dweight, dhidden, loss and metrics are allocated once, outside the graphs, and every replay writes them in full.
    Memory: each bucket of r rows used adds a private pool of about r * d * 8 bytes (bf16 policy and reference rows,
    fp32 dhidden rows) plus the GEMM workspaces and a few 4-byte arrays of 2*B*T; the static outputs are shared.  An
    fp32 `weight` is cast to a static bf16 copy inside the forward graph, so optimiser updates between replays are
    seen; `ref_weight` is frozen and cast once."""

    def __init__(self, head, weight: torch.Tensor, ref_weight: Optional[torch.Tensor], hidden: torch.Tensor,
                 labels: torch.Tensor, mask: Optional[torch.Tensor], ref_hidden: Optional[torch.Tensor] = None,
                 n_global: Optional[int] = None, warmup: int = 2):
        from . import ops
        if not hidden.is_cuda:
            raise RuntimeError("GraphedCompactDPOStep needs CUDA tensors (there is no CPU path)")
        if hidden.dim() != 3 or hidden.shape[0] % 2 or hidden.shape[0] == 0:
            raise ValueError("GraphedCompactDPOStep: hidden must be (2B, T, d), chosen rows first")
        if weight.dtype not in (torch.float32, torch.bfloat16) or not weight.is_contiguous():
            raise ValueError("GraphedCompactDPOStep: weight must be a contiguous fp32 or bf16 tensor")
        dev = hidden.device
        self.head = head
        self.weight = weight.detach()
        self.use_ref = ref_weight is not None and not head.loss.reference_free
        if self.use_ref and ref_hidden is None:
            raise ValueError("GraphedCompactDPOStep: ref_weight given without ref_hidden")
        self.ref_weight_bf16 = ops.cached_bf16(ref_weight.detach()) if self.use_ref else None
        self.n_global = n_global
        self.warmup = warmup
        self.B = hidden.shape[0] // 2
        nseq, T, d = hidden.shape
        self.hidden = hidden.detach().clone()
        self.labels = labels.to(dev).clone()
        self.mask = None if mask is None else mask.to(dev).clone()
        self.ref_hidden = ref_hidden.detach().to(dev).clone() if self.use_ref else None
        self.weight_bf16 = self.weight if weight.dtype == torch.bfloat16 else \
            torch.empty(weight.shape, dtype=torch.bfloat16, device=dev)
        grad_dtype = lambda t: torch.bfloat16 if t.dtype == torch.bfloat16 else torch.float32
        self.dhidden = torch.zeros(nseq, T, d, dtype=grad_dtype(hidden), device=dev)
        self.dweight = torch.zeros(weight.shape, dtype=grad_dtype(weight), device=dev)
        self.loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.metrics = torch.zeros(5, dtype=torch.float32, device=dev)
        self._one = torch.ones(1, dtype=torch.float32, device=dev)
        self.loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
        self.overflow_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.forward_done = torch.cuda.Event()
        self.graphs = {}  # rows_launch -> (forward graph, backward graph, tensors the graphs own)
        self._mask_host = None if mask is None else mask.detach().cpu()
        self.rows_launch = bucket_rows(scored_rows(self._mask_host, nseq, T))

    def _forward(self, rows):
        from . import _lib
        from . import functional as F
        if self.weight.dtype != torch.bfloat16:
            _lib.check(_lib.load().pgica_cast_f32_to_bf16(F._p(self.weight), self.weight.numel(),
                                                          F._p(self.weight_bf16), F._stream()))
        B, ln = self.B, self.head.length_normalize
        halves = lambda t: None if t is None else [t[:B], t[B:]]
        seqs, ref_seqs, ctx = F.lmhead_compact_fwd_bucketed(
            halves(self.hidden), self.weight_bf16, halves(self.labels), halves(self.mask) or [None, None], rows, ln,
            halves(self.ref_hidden), self.ref_weight_bf16)
        rc, rr = ref_seqs if ref_seqs is not None else (None, None)
        dpo = self.head.loss
        loss, metrics, dpc = F.dpo_loss_fwd(seqs[0], seqs[1], rc, rr, dpo.beta, dpo.label_smoothing,
                                            self.n_global or B)
        self.loss.copy_(loss)
        self.metrics.copy_(metrics)
        self.loss_host.copy_(loss, non_blocking=True)
        self.overflow_host.copy_(ctx.info[-1:], non_blocking=True)
        return ctx, dpc

    def _backward(self, ctx, dpc):
        from . import functional as F
        B = self.B
        grad_seq = F.dpo_grad_seq(dpc, self._one)  # d loss / d (chosen ++ rejected) sequence log-probs
        F.lmhead_compact_bwd_bucketed(ctx, self.weight_bf16, [grad_seq[:B], grad_seq[B:]],
                                      dhidden_outs=[self.dhidden[:B], self.dhidden[B:]], dweight_out=self.dweight)

    def _graphs(self, rows):
        g = self.graphs.get(rows)
        if g is not None:
            return g
        side = torch.cuda.Stream(device=self.hidden.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(self.warmup, 1)):  # first-use work (attributes, occupancy queries, allocator growth)
                self._backward(*self._forward(rows))
        torch.cuda.current_stream().wait_stream(side)
        fwd, bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.no_grad():
            with torch.cuda.graph(fwd):
                ctx, dpc = self._forward(rows)
            with torch.cuda.graph(bwd, pool=fwd.pool()):
                self._backward(ctx, dpc)
        g = self.graphs[rows] = (fwd, bwd, (ctx, dpc))
        return g

    def copy_inputs(self, hidden, labels=None, mask=None, ref_hidden=None):
        """Asynchronous copies into the static input buffers; labels and mask come from host (pinned) memory, and the
        row bucket of the next launch() is chosen from the mask on the host."""
        with torch.no_grad():
            self.hidden.copy_(hidden, non_blocking=True)
            if labels is not None:
                self.labels.copy_(labels, non_blocking=True)
            if mask is not None and self.mask is not None:
                if mask.is_cuda:
                    raise ValueError("GraphedCompactDPOStep.copy_inputs: the mask must be a host tensor")
                self._mask_host = mask
                self.mask.copy_(mask, non_blocking=True)
            if ref_hidden is not None and self.ref_hidden is not None:
                self.ref_hidden.copy_(ref_hidden, non_blocking=True)
        self.rows_launch = bucket_rows(scored_rows(self._mask_host, self.hidden.shape[0], self.hidden.shape[1]))

    def launch(self):
        """Enqueue the step on the current stream: forward (+ loss to pinned memory), then backward.  The first launch
        of a bucket captures its graphs (and synchronises the device once)."""
        fwd, bwd, _ = self._graphs(self.rows_launch)
        fwd.replay()
        self.forward_done.record()
        bwd.replay()

    def loss_value(self) -> float:
        """The step's loss as a Python float; waits for the forward graph only.  Raises when the device counted more
        scored rows than the bucket holds (the masks on the device disagree with the host's)."""
        self.forward_done.synchronize()
        if int(self.overflow_host[0]) != 0:
            raise RuntimeError("GraphedCompactDPOStep: the device masks score more rows than the %d-row bucket chosen "
                               "from the host mask; loss and gradients of this step are invalid" % self.rows_launch)
        return self.loss_host.item()

    def replay(self) -> torch.Tensor:
        """launch() and return the loss as a device tensor (no host synchronisation)."""
        self.launch()
        return self.loss


class GraphedContrastiveStep:
    """CUDA-graph capture of a contrastive-loss step (forward + backward of `loss_module(a, b)`), for the small batches
    the Stage-1 trainer uses: through the eager module API the step costs ~230 us of host time (custom-op dispatch,
    casts, autograd) around ~10 us of device time; replayed it is one `cudaGraphLaunch`.

        step = GraphedContrastiveStep(pg.ContrastiveLoss(temperature=0.07), image_embeddings_like, text_embeddings_like)
        step.copy_inputs(image_embeddings, text_embeddings)
        loss = step.replay()                 # device tensor; step.da / step.db hold the gradients
    """

    def __init__(self, loss_module, a: torch.Tensor, b: torch.Tensor, warmup: int = 2):
        if not a.is_cuda:
            raise RuntimeError("GraphedContrastiveStep needs CUDA tensors (there is no CPU path)")
        self.loss_module = loss_module
        self.a = a.detach().clone().requires_grad_(True)
        self.b = b.detach().clone().requires_grad_(True)
        side = torch.cuda.Stream(device=a.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                torch.autograd.grad(self.loss_module(self.a, self.b), (self.a, self.b))
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self.loss_module(self.a, self.b)
            self.da, self.db = torch.autograd.grad(self.loss, (self.a, self.b))

    def copy_inputs(self, a, b):
        with torch.no_grad():
            self.a.copy_(a, non_blocking=True)
            self.b.copy_(b, non_blocking=True)

    def replay(self) -> torch.Tensor:
        self.graph.replay()
        return self.loss
