"""`FusedAdamW`: torch.optim.AdamW whose update runs as one sm_100a kernel per parameter group (csrc/adamw.cu), with the
trainer's NaN-safe global-norm clip (pkg/training/trainer.py:494-520, 619-633) folded into the same pass.

    opt = FusedAdamW(model.parameters(), lr=5e-5, weight_decay=0.01)
    ...
    loss.backward()
    total_norm, is_finite = opt.clip_and_step(max_norm=1.0)    # instead of clip_grad_norm_(params, 1.0); opt.step()
    opt.zero_grad(set_to_none=True)

Param groups, LR schedulers, zero_grad, step hooks and the state_dict format are torch.optim.AdamW's: a checkpoint of
either optimizer loads into the other.
"""
import torch

from . import functional as F

__all__ = ["FusedAdamW"]


class FusedAdamW(torch.optim.AdamW):
    """AdamW (decoupled weight decay) on fp32 parameters, updated on the GPU by the library's multi-tensor kernel.

    The arithmetic per element is that of torch's single-tensor AdamW; the bias corrections come from the step counters
    in `state[p]['step']`, which stay on the device.  `step()` is plain AdamW; `clip_and_step(max_norm)` also clips by
    the global L2 norm of all gradients and skips a step whose norm is not finite — with no host synchronisation.
    Not supported (ValueError): amsgrad, maximize, capturable, differentiable, foreach=True, fused=True, Tensor lr or
    betas, parameters that are not fp32 or are sparse."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, *,
                 maximize=False, foreach=None, capturable=False, differentiable=False, fused=None):
        for name, value in (("amsgrad", amsgrad), ("maximize", maximize), ("capturable", capturable),
                            ("differentiable", differentiable), ("foreach", foreach), ("fused", fused)):
            if value:
                raise ValueError(f"FusedAdamW: {name}=True is not supported")
        _check_scalars(lr, betas)
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        group = self.param_groups[-1]
        for name in ("amsgrad", "maximize", "capturable", "differentiable", "foreach", "fused"):
            if group.get(name):
                raise ValueError(f"FusedAdamW: {name}=True is not supported")
        _check_scalars(group["lr"], group["betas"])
        for p in group["params"]:
            if p.dtype != torch.float32:
                raise ValueError(f"FusedAdamW: parameters must be fp32 (got {p.dtype})")
            if p.layout != torch.strided:
                raise ValueError("FusedAdamW: sparse parameters are not supported")

    @torch.no_grad()
    def step(self, closure=None, *, grad_stats=None):
        """One AdamW step over every parameter with a gradient: one kernel launch per parameter group (and device).
        `grad_stats`: the (3,) device tensor of functional.grad_norm_clip(..., clip=False); the update then uses the
        clipped gradients and is skipped on the device when the norm is not finite (see clip_and_step)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            by_device = {}
            for p in group["params"]:
                if p.grad is None:
                    continue
                if p.grad.is_sparse:
                    raise ValueError("FusedAdamW: sparse gradients are not supported")
                state = self.state[p]
                if len(state) == 0:
                    state["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
                    state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                elif state["step"].device != p.device or state["step"].dtype != torch.float32:
                    # a torch.optim.AdamW checkpoint keeps its step counters on the CPU: moved once, then they stay
                    state["step"] = state["step"].to(device=p.device, dtype=torch.float32)
                lists = by_device.setdefault(p.device, ([], [], [], [], []))
                for lst, t in zip(lists, (p, p.grad, state["exp_avg"], state["exp_avg_sq"], state["step"])):
                    lst.append(t)
            beta1, beta2 = group["betas"]
            for params, grads, exp_avgs, exp_avg_sqs, steps in by_device.values():
                stats = None if grad_stats is None else grad_stats.to(params[0].device)
                F.adamw_step(params, grads, exp_avgs, exp_avg_sqs, steps, group["lr"], beta1, beta2, group["eps"],
                             group["weight_decay"], grad_stats=stats)
                # the kernel writes through raw pointers: move `_version` as an in-place op would, so that caches keyed
                # on it (ops.cached_bf16) see the new weights
                torch.autograd.graph.increment_version(params)
        return loss

    def clip_and_step(self, max_norm):
        """`clip_grad_norm_(all parameters, max_norm)` followed by `step()`, with the clip folded into the update:
        one norm pass over every gradient of every group (functional.grad_norm_clip, norm only) and one update pass that
        multiplies each gradient by the clip coefficient as it reads it.  Returns (total_norm, is_finite), 0-dim device
        tensors; nothing is read on the host.  Two differences from clip_grad_norm_ + step():
          - p.grad keeps its unclipped values (the clipped gradient is never stored);
          - a NaN or Inf anywhere in the gradients skips the whole update on the device — weights, exp_avg, exp_avg_sq and
            step counters are left exactly as they were — where clip_grad_norm_ would scale every gradient by NaN and the
            step would write NaN into the weights."""
        grads = [p.grad for group in self.param_groups for p in group["params"]
                 if p.grad is not None and p.grad.numel() > 0]
        if not grads:
            self.step()
            return torch.zeros(()), torch.ones((), dtype=torch.bool)
        stats = F.grad_norm_clip(grads, max_norm, clip=False)
        self.step(grad_stats=stats)
        return stats[0], stats[2] != 0


def _check_scalars(lr, betas):
    if isinstance(lr, torch.Tensor):
        raise ValueError("FusedAdamW: a Tensor lr is not supported; pass a float")
    if any(isinstance(b, torch.Tensor) for b in betas):
        raise ValueError("FusedAdamW: Tensor betas are not supported; pass floats")
