#!/usr/bin/env python
"""Benchmark of the loss-head hot path (BASELINE.json metric: DPO pair-tokens/s fwd+bwd; NT-Xent pairs/s as extras).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload at every N (weak scaling, one process per GPU): BASELINE config 2 — Stage-2 DPO head, GPT-2 Medium LM head
(d=1024, V=50257), 16 preference pairs per GPU, seq 128, beta=0.1, random-init weights, synthetic hidden states.
One step = policy forward + backward (dH, dW) + frozen-reference forward + DPO loss (+ dW all-reduce when N>1).
A pair-token is one scored position of one (chosen, rejected) pair: B*(T-1) = 2032 per GPU per step.

`value`   inputs resident in HBM, CUDA events around K steps, max over ranks.
`e2e`     the same step through the public module API (FusedDPOHead.forward_stacked + backward), inputs copied
          from pinned host memory every step, loss read back every step.
`roofline` the dominant kernel of the step against the measured bf16 tensor-core peak (MEASURED_PEAKS.json).
`cpu_baseline` the reference's CPU path (oracle/torch_port.py) timed on this box's host cores, bounded sample.
`--impl reference` times that CPU path alone, on all host threads, in the same JSON shape.
`--dump-outputs DIR` writes what the last timed resident step returned (rank 0) to DIR/<name>.npy, float32; the inputs
          are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(pairs=16, seq_len=128, d=1024, vocab=50257, beta=0.1)
METRIC = "dpo_pair_tokens_per_s"
UNIT = "pair-tokens/s"
WORKLOAD = ("cfg2: Stage-2 DPO loss head, GPT-2 Medium LM head d=1024 V=50257, chosen/rejected seq 128, 16 pairs per "
            "GPU, beta=0.1, policy fwd+bwd + frozen-reference fwd, random-init, all-ones masks")
FLOP_PER_PAIR_TOKEN = 16 * CFG["d"] * CFG["vocab"]  # BASELINE.md §3: policy fwd 4dV + ref fwd 4dV + policy bwd 8dV


def ncu_traffic(kernel_prefix):
    """DRAM bytes (read + write) per launch of a kernel, from the committed `ncu --set full` summary
    profiles/ncu_traffic.json (written by tools/ncu_summary.py from the capture of this very workload).  None when no
    capture of that kernel is on file: the bench never invents the number."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        table = json.load(open(path))
    except Exception:
        return None
    for name, rec in table.items():
        if name.startswith(kernel_prefix):
            return rec.get("dram_bytes_per_launch")
    return None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner, torchrun its OMP notice) write to
# file descriptor 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON line goes to a
# private duplicate of the original stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    hbm=p["hbm_gbs"], source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from a thread DURING the timed region (about one sample per
    millisecond; `nvidia-smi -lms` needs longer to start than a 100 ms timed region lasts)."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        import threading
        self.samples, self.masks, self.power = [], [], []
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        except Exception as e:  # no NVML: report nulls rather than fail the bench
            log("clock sampler unavailable:", repr(e))

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.masks.append(int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.001)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._t is None:
            return out
        self._stop.set()
        self._t.join(timeout=2)
        if self.samples:
            out["sm_mhz"] = statistics.median(self.samples)
            out["sm_min_mhz"] = min(self.samples)
            out["samples"] = len(self.samples)
        if self.power:
            out["power_w_max"] = max(self.power)
        for name, bit in self.REASONS:
            if any(m & bit for m in self.masks):
                out["reasons"].append(name)
        return out


# ----------------------------------------------------------------------------------------------- CPU reference
def cpu_reference_step_inputs(pairs, seed=1234):
    import torch
    T, d, V = CFG["seq_len"], CFG["d"], CFG["vocab"]
    g = torch.Generator().manual_seed(seed)
    W = torch.randn(V, d, generator=g) * 0.02
    Wr = torch.randn(V, d, generator=g) * 0.02
    hs = [torch.randn(pairs, T, d, generator=g) for _ in range(4)]
    yc, yr = torch.randint(0, V, (pairs, T), generator=g), torch.randint(0, V, (pairs, T), generator=g)
    m = torch.ones(pairs, T, dtype=torch.long)
    return W, Wr, hs, yc, yr, m


def reference_cpu_step_fn():
    """One Stage-2 head evaluation on the host cores, written with the reference's OWN modules when its package can be
    imported (baseline/_ref on the GPU box, /root/reference in the build container: components.py is loaded by file
    path, it needs torch only) -> kind "reference"; otherwise the restatement in oracle/torch_port.py -> kind "port"."""
    import torch

    from oracle import ref_model
    from oracle import torch_port as tp
    src = ref_model.reference_src()
    if src is not None:
        import importlib.util
        path = os.path.join(src, "preference_guided_image_captioning_alignment", "models", "components.py")
        spec = importlib.util.spec_from_file_location("_pgica_ref_components_bench", path)
        comp = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(comp)
        dpo = comp.DPOPreferenceLoss(beta=CFG["beta"])
        csl = comp.compute_sequence_logprobs

        def step(hc, hr, W, yc, yr, m, rhc, rhr, Wr):
            lin = torch.nn.functional.linear  # GPT2LMHeadModel.lm_head: nn.Linear without bias (modeling_gpt2.py:651,706)
            pc, pr = csl(lin(hc, W), yc, m), csl(lin(hr, W), yr, m)
            with torch.no_grad():
                rc, rr = csl(lin(rhc, Wr), yc, m), csl(lin(rhr, Wr), yr, m)
            loss, metrics = dpo(pc, pr, rc, rr)
            loss.backward()
            return loss.detach()
        return step, "reference"

    def step(hc, hr, W, yc, yr, m, rhc, rhr, Wr):
        return tp.dpo_head_step(hc, hr, W, yc, yr, m, m, rhc, rhr, Wr, CFG["beta"])[0]
    return step, "port"


def time_cpu_reference(pairs, steps, warmup):
    """The reference's CPU path (fp32 torch ops on all host threads): policy fwd+bwd + frozen-reference fwd + DPO loss
    on `pairs` preference pairs.  -> (pair-tokens/s from the MEDIAN step, median s/step, threads, kind, total s)"""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    W, Wr, hs, yc, yr, m = cpu_reference_step_inputs(pairs)
    W.requires_grad_(True)
    hs[0].requires_grad_(True)
    hs[1].requires_grad_(True)
    fn, kind = reference_cpu_step_fn()

    def step():
        W.grad = hs[0].grad = hs[1].grad = None
        return fn(hs[0], hs[1], W, yc, yr, m, hs[2], hs[3], Wr)

    for _ in range(warmup):
        step()
    times = []
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    total = time.perf_counter() - t_all
    med = statistics.median(times)
    tokens = pairs * (CFG["seq_len"] - 1)
    return tokens / med, med, torch.get_num_threads(), kind, total


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args, rank):
    """`--impl reference`: the reference's CPU implementation of the SAME config (all 16 pairs per step, the requested
    number of steps), every step measured."""
    if rank != 0:
        return
    pairs = CFG["pairs"]
    steps, warmup = max(args.steps, 1), max(min(args.warmup, 2), 1)
    value, sec, threads, kind, total = time_cpu_reference(pairs, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "pairs_per_gpu": pairs, "seq_len": CFG["seq_len"], "d": CFG["d"],
                   "vocab": CFG["vocab"], "parallelism": f"dp{args.gpus}",
                   "note": f"CPU arm: {warmup} warm-up (capped at 2: a step takes ~1 s) + {steps} measured steps, "
                           f"median step; timed region {total:.1f} s"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"all {pairs} pairs per step, {steps} steps (median), fp32 torch ops of the "
                                   f"{'reference modules' if kind == 'reference' else 'restated reference'}, "
                                   f"{cpu_model_name()}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------- our arm
DUMP_DW_ROW_STRIDE = 8  # dW is V x d fp32 (206 MB): every 8th vocabulary row keeps the dump within 64 MB


def dump_outputs(path, outputs):
    """What one resident step hands back, as float32 .npy files under `path`: the sequence log-probs of both forwards,
    the DPO loss and metrics, dH in full and dW sampled every DUMP_DW_ROW_STRIDE-th row (rows 0, 8, 16, ...)."""
    import numpy as np
    seq_p, seq_r, loss, metrics, dh, dw = outputs
    arrays = {"policy_seq_logprobs": seq_p, "reference_seq_logprobs": seq_r, "loss": loss, "metrics": metrics,
              "dhidden": dh, f"dweight_rows_stride{DUMP_DW_ROW_STRIDE}": dw[::DUMP_DW_ROW_STRIDE]}
    arrays = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"output dump of {total} bytes exceeds 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log(f"dumped {len(arrays)} outputs of the last timed step ({total / 2 ** 20:.1f} MB) to {path}")


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    _lib.check(lib.pgica_device_check())
    B, T, d, V, beta = CFG["pairs"], CFG["seq_len"], CFG["d"], CFG["vocab"], CFG["beta"]
    n_global = B * world
    gen = torch.Generator().manual_seed(1234 + rank)
    gw = torch.Generator().manual_seed(1234)  # weights are replicated
    W = (torch.randn(V, d, generator=gw) * 0.02).to(torch.bfloat16).to(dev)
    Wr = (torch.randn(V, d, generator=gw) * 0.02).to(torch.bfloat16).to(dev)
    H_host = torch.randn(2 * B, T, d, generator=gen).to(torch.bfloat16).pin_memory()
    Hr_host = torch.randn(2 * B, T, d, generator=gen).to(torch.bfloat16).pin_memory()
    y_host = torch.randint(0, V, (2 * B, T), generator=gen).pin_memory()
    m_host = torch.ones(2 * B, T, dtype=torch.long).pin_memory()
    H, Hr, y, m = H_host.to(dev), Hr_host.to(dev), y_host.to(dev), m_host.to(dev)
    one = torch.ones((), device=dev)
    fused = _lib.get_option("sgg_fused") != 0  # dH and dW from one recomputation (sgg_f.cu) vs two launches

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: how the LM-head weight gradient is summed over the ranks.
    #   overlap (default)  distributed.OverlappedDWAllReduce: the dual backward kernel publishes per-segment progress,
    #                      a co-resident peer-memory all-reduce kernel (csrc/peer_ar.cu) sums finished segments over
    #                      NVLink while the rest of the vocabulary is still being computed; the packed loss / metric
    #                      scalars ride in the padding rows of the same buffer
    #   nccl               plain NCCL fp32 all-reduce after the kernel + a second small all-reduce for the scalars
    ar_mode = os.environ.get("PGICA_DW_ALLREDUCE", "overlap") if world > 1 else "none"
    overlap = None
    if world > 1 and ar_mode == "overlap" and fused:
        from preference_guided_image_captioning_alignment_b200 import distributed as D
        overlap = D.OverlappedDWAllReduce(V, d, dev, segments=int(os.environ.get("PGICA_DW_SEGMENTS", "8")),
                                          max_ctas=int(os.environ.get("PGICA_DW_AR_CTAS", "-1")),
                                          multicast={"0": False, "1": True}.get(os.environ.get("PGICA_DW_MULTICAST", ""), None))
    elif world > 1:
        ar_mode = "nccl"

    # ------------------------------------------------------------------ resident step (functional API + events)
    def resident_step(ev=None):
        def mark(i):
            if ev is not None:
                ev[i].record()
        mark(0)
        seq_p, lse_p, _, rl, rw, _ = F.lmhead_logprob_fwd(H, W, y, m, False)
        mark(1)
        seq_r = F.lmhead_logprob_fwd(Hr, Wr, y, m, False)[0]
        mark(2)
        loss, metrics, dpc = F.dpo_loss_fwd(seq_p[:B], seq_p[B:], seq_r[:B], seq_r[B:], beta, 0.0, n_global)
        gseq = F.dpo_grad_seq(dpc, one)
        mark(3)
        if overlap is not None:
            packed = torch.cat([loss.reshape(1), metrics])
            dh, dw, done, packed = overlap.backward(H, W, rl, rw, lse_p, gseq, False, scalars=packed)
            mark(4)  # end of the backward kernel on the main stream
            mark(5)
            torch.cuda.current_stream().wait_event(done)  # dW (and the scalars) summed over the ranks
            mark(6)
            return seq_p, seq_r, packed[0], packed[1:], dh, dw
        if fused:
            dh, dw = F.lmhead_logprob_bwd(H, W, rl, rw, lse_p, gseq, False)
            mark(4)
            mark(5)
        else:
            _, dw = F.lmhead_logprob_bwd(H, W, rl, rw, lse_p, gseq, False, need_dhidden=False)
            mark(4)
            dh, _ = F.lmhead_logprob_bwd(H, W, rl, rw, lse_p, gseq, False, need_dweight=False)
            mark(5)
        if world > 1:
            dist.all_reduce(dw)
            packed = torch.cat([loss.reshape(1), metrics])
            dist.all_reduce(packed)
            mark(6)
            loss, metrics = packed[0], packed[1:]
        return seq_p, seq_r, loss, metrics, dh, dw

    for _ in range(max(args.warmup, 3)):
        resident_step()
    barrier()
    n_marks = 7 if world > 1 else 6
    events = [[torch.cuda.Event(enable_timing=True) for _ in range(n_marks)] for _ in range(args.steps)]
    launches0 = lib.pgica_kernel_launches()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin.record()
    for k in range(args.steps - 1):
        resident_step(events[k])
    last = resident_step(events[-1])
    t_end.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    launches = lib.pgica_kernel_launches() - launches0
    elapsed_ms = t_begin.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    # order of marks: 0 start,1 after fwd_policy,2 after fwd_ref,3 after dpo,4 after dW (or the fused backward),
    # 5 after dH,(6 after all-reduce)
    names_in_order = ["fwd_policy", "fwd_reference", "dpo_scalar", "bwd_dH_dW" if fused else "bwd_dW", "bwd_dH"] + \
        (["allreduce_dW"] if world > 1 else [])
    phase_ms = {n: statistics.mean(events[k][i].elapsed_time(events[k][i + 1]) for k in range(args.steps))
                for i, n in enumerate(names_in_order)}
    if fused:
        del phase_ms["bwd_dH"]
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = t.item()
    pair_tokens_step = B * (T - 1)
    value = pair_tokens_step * world * args.steps / (elapsed_ms * 1e-3)
    if os.environ.get("PGICA_BENCH_LEAN"):  # tuning runs: the resident step only (NOT the contract line)
        if rank == 0:
            emit({"lean": True, "metric": METRIC, "value": value, "n_gpus": world, "ms_per_step": elapsed_ms / args.steps,
                  "phase_ms": phase_ms, "dw_allreduce": ar_mode,
                  "segments": overlap.nseg if overlap is not None else None,
                  "ar_ctas": overlap.max_ctas if overlap is not None else None,
                  "multicast": bool(overlap.multicast_ptr) if overlap is not None else None})
        return

    # ------------------------------------------------------------------ end-to-end step (public module API)
    # FusedDPOHead.forward_stacked and its backward, recorded once per input-buffer set into CUDA graphs
    # (pg.GraphedDPOStep) and replayed: issued launch by launch from Python the step is host-bound.  Two buffer sets:
    # while step k computes on one, the inputs of step k+1 are copied from pinned host memory into the other on a
    # copy stream (every step still pays exactly one host->device copy of its inputs inside the timed region, and one
    # device->host read of its loss).  PGICA_BENCH_E2E_GRAPH=0 times the eager module calls instead.
    head = pg.FusedDPOHead(beta=beta)
    # fp32 master copy of the tied weight, as in the reference model: the op keeps a bf16 operand copy that is recast
    # only when the Parameter changes (ops.cached_bf16), and hands back an fp32 dW — the same gradient dtype, and at
    # N > 1 the same all-reduce (fp32 dW + the packed scalars), as the resident arm above
    Wp = W.float().requires_grad_(True)
    h2d = sum(t.numel() * t.element_size() for t in (H_host, Hr_host, y_host, m_host))
    use_graph = os.environ.get("PGICA_BENCH_E2E_GRAPH", "1") != "0" and overlap is None
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"k": 0}
    if use_graph:
        steps_g = [pg.GraphedDPOStep(head, Wp, Wr, H, y, m, Hr, n_global) for _ in range(2)]
        bufs = [(g.hidden, g.ref_hidden, g.labels, g.mask) for g in steps_g]
    else:
        bufs = [tuple(torch.empty_like(t) for t in (H, Hr, y, m)) for _ in range(2)]

    debug_nocopy = bool(os.environ.get("PGICA_BENCH_DEBUG_NOCOPY"))  # diagnosis only: invalidates the e2e number

    def issue_copy(slot):
        if debug_nocopy:
            copied[slot].record()
            return
        copy_stream.wait_event(consumed[slot])  # the step that last used this buffer set has finished
        with torch.cuda.stream(copy_stream), torch.no_grad():
            for dst, src in zip(bufs[slot], (H_host, Hr_host, y_host, m_host)):
                dst.copy_(src, non_blocking=True)
            copied[slot].record()

    for ev in consumed:
        ev.record()
    issue_copy(0)

    # N > 1 with the overlapped all-reduce: the step is issued through the functional wrappers + the reducer (the public
    # multi-GPU entry point, distributed.OverlappedDWAllReduce.backward), same copies in, same loss read out.  The loss
    # goes to pinned memory right after the forward; the host reads it while the backward + all-reduce are running.
    loss_pinned = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    fwd_done = [torch.cuda.Event() for _ in range(2)]

    def e2e_step_overlapped():
        slot = state["k"] & 1
        state["k"] += 1
        issue_copy(slot ^ 1)
        cur = torch.cuda.current_stream()
        cur.wait_event(copied[slot])
        Hd, Hrd, yd, md = bufs[slot]
        Hd = Hd.detach()
        seq_p, lse_p, _, rl, rw, _ = F.lmhead_logprob_fwd(Hd, W, yd, md, False)
        seq_r = F.lmhead_logprob_fwd(Hrd, Wr, yd, md, False)[0]
        loss, metrics, dpc = F.dpo_loss_fwd(seq_p[:B], seq_p[B:], seq_r[:B], seq_r[B:], beta, 0.0, n_global)
        loss_pinned[slot].copy_(loss, non_blocking=True)
        fwd_done[slot].record()
        gseq = F.dpo_grad_seq(dpc, one)
        dh, dw, done, packed = overlap.backward(Hd, W, rl, rw, lse_p, gseq, False,
                                                scalars=torch.cat([loss.reshape(1), metrics]))
        cur.wait_event(done)
        state["packed"] = packed
        consumed[slot].record()
        fwd_done[slot].synchronize()
        return loss_pinned[slot].item()

    def e2e_step():
        if overlap is not None:
            return e2e_step_overlapped()
        slot = state["k"] & 1
        state["k"] += 1
        issue_copy(slot ^ 1)  # prefetch the next step's inputs
        torch.cuda.current_stream().wait_event(copied[slot])
        if use_graph:
            steps_g[slot].launch()
            grad_w = steps_g[slot].dweight
        else:
            Hd, Hrd, yd, md = bufs[slot]
            hin = Hd.requires_grad_(True)
            Wp.grad = None
            loss, metrics = head.forward_stacked(hin, Wp, yd, md, Hrd, Wr, n_global)
            loss.backward()
            hin.requires_grad_(False)
            grad_w = Wp.grad
        if world > 1:
            dist.all_reduce(grad_w)  # the module API hands back an ordinary autograd gradient: NCCL all-reduce (fp32)
            g = steps_g[slot] if use_graph else None
            state["packed"] = torch.cat([(g.loss if g else loss).detach().reshape(1), (g.metrics if g else metrics)])
            dist.all_reduce(state["packed"])
        consumed[slot].record()
        # device -> host read of the step's result; the graphed step copies the loss to pinned memory at the end of its
        # forward graph, so the host reads it while the backward is still running
        return steps_g[slot].loss_value() if use_graph else loss.item()

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last_loss = e2e_step()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = t.item()
    e2e_value = pair_tokens_step * world * args.steps / (e2e_ms * 1e-3)

    # ------------------------------------------------------------------ NT-Xent with global negatives (cfg3 scheme)
    dist_ntxent = None
    if world > 1:
        from preference_guided_image_captioning_alignment_b200 import distributed as D
        bl = 4096  # rows per rank (cfg3: 32768 over 8 GPUs)
        ga = torch.Generator().manual_seed(77 + rank)
        a_l = torch.nn.functional.normalize(torch.randn(bl, 512, generator=ga), dim=-1).to(dev).requires_grad_(True)
        b_l = torch.nn.functional.normalize(torch.randn(bl, 512, generator=ga), dim=-1).to(dev).requires_grad_(True)

        def nt_step():
            a_l.grad = b_l.grad = None
            loss = D.global_ntxent(a_l, b_l, 0.5, assume_normalized=True)  # the rows are unit-norm by construction
            loss.backward()
            return loss

        for _ in range(3):
            nt_step()
        barrier()
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for _ in range(10):
            nt_loss = nt_step()
        n1.record()
        barrier()
        t = torch.tensor([n0.elapsed_time(n1) / 10], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        Bg = bl * world

        # phase split of the same step, issued piece by piece (same building blocks as distributed._GlobalNTXent)
        def nt_phases(ev):
            off = rank * bl
            ev[0].record()
            a_op, b_op = F.as_bf16(a_l.detach()), F.as_bf16(b_l.detach())
            b_all = D.all_gather_rows(b_op)
            ev[1].record()
            lse_row, diag, lse_col_part = F.ntxent_fwd(a_op, b_all, 2.0, off, bounded=True)
            ev[2].record()
            parts = D.all_gather_rows(lse_col_part.reshape(1, Bg))
            lse_col = F.lse_combine(parts)
            loss = F.ntxent_loss(lse_row, diag, lse_col[off:off + bl].contiguous(), 1.0 / Bg)
            dist.all_reduce(loss)
            ev[3].record()
            da, db_part = F.ntxent_bwd(a_op, b_all, 2.0, off, lse_row, lse_col, one, 1.0 / (2.0 * Bg), bounded=True)
            ev[4].record()
            D.reduce_scatter_rows(db_part)
            ev[5].record()

        names = ["cast + all-gather of text rows (bf16)", "forward: row LSE / diagonal / column-LSE partials",
                 "column-LSE all-gather + merge + loss all-reduce", "backward: dA and dB partial (recompute)",
                 "reduce-scatter of dB (fp32)"]
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(8)]
        for e in evs[:3]:
            nt_phases(e)
        barrier()
        for e in evs[3:]:
            nt_phases(e)
        barrier()
        ph = torch.tensor([sum(e[i].elapsed_time(e[i + 1]) for e in evs[3:]) / 5 for i in range(5)], device=dev)
        dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        dist_ntxent = {"global_batch": Bg, "rows_per_gpu": bl, "ms_per_step": t.item(),
                       "pairs_per_s": Bg / (t.item() * 1e-3), "algorithmic_tflops": 6.0 * Bg * Bg * 512 / t.item() / 1e9,
                       "algorithmic_tflops_per_gpu": 6.0 * bl * Bg * 512 / t.item() / 1e9,
                       "frac_of_measured_bf16_peak_per_gpu": 6.0 * bl * Bg * 512 / t.item() / 1e9 / peaks()["burst"],
                       "loss": nt_loss.item(),
                       "phase_ms_max_over_ranks": dict(zip(names, [round(v, 4) for v in ph.tolist()])),
                       "collectives": "all-gather of text rows, all-gather of column-LSE partials, reduce-scatter of dB"}
    # ------------------------------------------------------------------ BASELINE config 4, this GPU's share
    cfg4 = cfg4_extra(torch, dist, F, dev, rank, world, W, Wr, barrier)
    gradclip = gradclip_extra(torch, F, dev) if rank == 0 else None
    if rank != 0:
        return
    pk = peaks()
    rows = 2 * B * T  # rows the GEMMs actually run over (the unscored last position included)
    gemm = 2.0 * rows * d * V  # one GEMM-unit: rows x V x d
    flops = {"fwd_policy": gemm, "fwd_reference": gemm}
    flops.update({"bwd_dH_dW": 2 * gemm} if fused else {"bwd_dH": gemm, "bwd_dW": gemm})
    kernels = {n: {"ms": phase_ms[n], "tflops": flops[n] / phase_ms[n] / 1e9, "algorithmic_flops": flops[n]}
               for n in flops}
    dom = max(flops, key=lambda n: phase_ms[n])
    kname = {"fwd_policy": "gemm_lse_kernel", "fwd_reference": "gemm_lse_kernel", "bwd_dH": "sggx_kernel<4,row>",
             "bwd_dW": "sggx_kernel<4,col>", "bwd_dH_dW": "sggf_kernel<row> (dual: dH and dW from one recomputation)"}
    # DRAM bytes per launch of that kernel from the committed `ncu --set full` capture of this workload
    short = {"fwd_policy": "gemm_lse_kernel", "fwd_reference": "gemm_lse_kernel", "bwd_dH": "sggx_kernel",
             "bwd_dW": "sggx_kernel", "bwd_dH_dW": "sggf_kernel"}
    traffic = {n: ncu_traffic(short[n]) for n in short}
    roofline = {"bound": "tensor", "kernel": kname[dom],
                "phase": dom, "achieved": kernels[dom]["tflops"], "peak": pk["burst"], "unit": "TFLOP/s",
                "frac": kernels[dom]["tflops"] / pk["burst"], "peak_source": pk["source"] + " bf16 dense, burst",
                "traffic": traffic[dom],
                "executed_tflops": kernels[dom]["tflops"] * (1.5 if dom == "bwd_dH_dW" else 2.0 if dom.startswith("bwd") else 1.0),
                "step_achieved": FLOP_PER_PAIR_TOKEN * pair_tokens_step / (elapsed_ms / args.steps) / 1e9,
                "step_frac": FLOP_PER_PAIR_TOKEN * pair_tokens_step / (elapsed_ms / args.steps) / 1e9 / pk["burst"]}
    cpu_val, cpu_sec, cpu_threads, cpu_kind, cpu_total = time_cpu_reference(CFG["pairs"], 5, 1)
    extras = ntxent_extras(torch, F, dev)
    if dist_ntxent is not None:
        extras["global_negatives"] = dist_ntxent
    compaction = torch_eager = cfg5 = None
    if world == 1:
        compaction = compaction_extra(torch, pg, dev, W.float())
        torch_eager = torch_eager_extra(torch, dev)
        cfg5 = cfg5_extra()
    also = {"cfg3_ntxent_global_negatives": dist_ntxent, "cfg4_dpo_seq512": cfg4,
            "cfg5_stage2_step": None if cfg5 is None else {k: cfg5.get(k) for k in ("speedup", "first_loss_rel_diff", "unavailable", "error", "skipped") if k in cfg5},
            "cfg2_valid_row_compaction": None if compaction is None else
            {"rows": compaction["rows"], "speedup_at_10_20_tokens": compaction["speedup"],
             "ms_vs_scored_rows": [[r["scored_rows"], round(r["c_abi_ms_per_step"], 4)] for r in compaction["sweep"]]},
            "ntxent_single_gpu": extras}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "pairs_per_gpu": B, "global_pairs": n_global, "seq_len": T, "d": d, "vocab": V,
                   "parallelism": f"dp{world}", "pair_tokens_per_step_per_gpu": pair_tokens_step,
                   "backward": "dual kernel: dH and dW from one recomputation of the logits" if fused
                               else "one launch per product",
                   "dw_allreduce": ("none" if world == 1 else
                                    f"progress-gated peer-memory all-reduce kernel beside the backward kernel, fp32, "
                                    f"{overlap.nseg} vocabulary segments, {overlap.max_ctas} CTAs, "
                                    f"{'summed in the NVSwitch (multimem.ld_reduce)' if overlap.multicast_ptr else 'unicast peer loads'}"
                                    f"; loss/metric scalars in the same buffer"
                                    if overlap is not None else "nccl fp32 all-reduce after the backward + nccl scalars"),
                   "also_measured": also,
                   "l2": "inputs larger than L2: the step streams 2x103 MB of bf16 LM-head weights and writes a "
                         "206 MB fp32 dW (L2 = 126 MB)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps,
                "last_loss": last_loss if world == 1 else float(state["packed"][0].item()),
                "last_loss_read_in_step": last_loss,  # what the step's D2H read returned (this rank's share when N > 1)
                "api": "functional.lmhead_logprob_fwd / dpo_loss_fwd + distributed.OverlappedDWAllReduce.backward (dW and the "
                       "scalars summed over the ranks by the co-resident peer-memory all-reduce), loss read from pinned "
                       "memory after the forward" if overlap is not None else
                       "GraphedDPOStep.launch + loss_value (CUDA graphs of FusedDPOHead.forward_stacked and its backward)" if use_graph
                       else "FusedDPOHead.forward_stacked + backward, eager"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "kernels": kernels,
        "phase_ms": phase_ms,
        "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": cpu_threads, "kind": cpu_kind,
                         "sample": f"5 steps (median, {cpu_sec * 1e3:.0f} ms) of all 16 pairs after 1 warm-up, fp32 "
                                   f"torch ops of the {'reference modules' if cpu_kind == 'reference' else 'restated reference'}"
                                   f", {cpu_total:.1f} s of CPU time, {cpu_model_name()}"},
        "ntxent": extras,
        "global_negatives": dist_ntxent,
        "cfg4": cfg4,
        "cfg5": cfg5,
        "valid_row_compaction": compaction,
        "torch_eager_same_gpu": torch_eager,
        "grad_norm_clip": gradclip,
    }
    emit(line)


def cfg4_extra(torch, dist, F, dev, rank, world, W, Wr, barrier):
    """BASELINE config 4 (seq 512, 256 preference pairs over 8 GPUs = 32 pairs per GPU, policy + frozen reference):
    the same resident step as the headline, 32 pairs per GPU at every N, dW all-reduced with NCCL when N > 1."""
    B, T, d, V, beta = 32, 512, CFG["d"], CFG["vocab"], CFG["beta"]
    gen = torch.Generator().manual_seed(4321 + rank)
    H = torch.randn(2 * B, T, d, generator=gen).to(torch.bfloat16).to(dev)
    Hr = torch.randn(2 * B, T, d, generator=gen).to(torch.bfloat16).to(dev)
    y = torch.randint(0, V, (2 * B, T), generator=gen).to(dev)
    m = torch.ones(2 * B, T, dtype=torch.long, device=dev)
    one = torch.ones((), device=dev)

    def step():
        seq_p, lse_p, _, rl, rw, _ = F.lmhead_logprob_fwd(H, W, y, m, False)
        seq_r = F.lmhead_logprob_fwd(Hr, Wr, y, m, False)[0]
        loss, metrics, dpc = F.dpo_loss_fwd(seq_p[:B], seq_p[B:], seq_r[:B], seq_r[B:], beta, 0.0, B * world)
        gseq = F.dpo_grad_seq(dpc, one)
        dh, dw = F.lmhead_logprob_bwd(H, W, rl, rw, lse_p, gseq, False)
        if world > 1:
            dist.all_reduce(dw)
            dist.all_reduce(torch.cat([loss.reshape(1), metrics]))
        return loss

    for _ in range(3):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / iters
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    tokens = B * (T - 1) * world
    return {"workload": f"cfg4: seq 512, {B} pairs per GPU ({B * world} global), policy fwd+bwd + reference fwd"
                        + (", NCCL fp32 all-reduce of dW" if world > 1 else ""),
            "ms_per_step": ms, "pair_tokens_per_s": tokens / (ms * 1e-3),
            "algorithmic_tflops_per_gpu": 16.0 * d * V * B * (T - 1) / ms / 1e9}


def compaction_extra(torch, pg, dev, W32):
    """Valid-row compaction on cfg2's shape with the reference's real padding statistics (SURVEY Appendix A): 16 pairs,
    seq 128, right-padded captions (pkg/data/preprocessing.py:223-231 pads to 128; real captions are 10-20 tokens).
    The trainer-facing path — PreferenceLoss on LazyLogits, fp32 hidden states and fp32 tied weight — forward + backward;
    only scored positions count as pair-tokens.  Three paddings show how the time follows the scored rows; next to the
    shortest one the same batch through the full-row op (every row, masked or not)."""
    from preference_guided_image_captioning_alignment_b200 import functional as F
    from preference_guided_image_captioning_alignment_b200 import ops
    from preference_guided_image_captioning_alignment_b200.losses import LazyLogits
    B, T, d, V = CFG["pairs"], CFG["seq_len"], CFG["d"], CFG["vocab"]
    g = torch.Generator().manual_seed(99)
    hw = torch.randn(B, T, d, generator=g).to(dev).requires_grad_(True)
    hl = torch.randn(B, T, d, generator=g).to(dev).requires_grad_(True)
    W = W32.detach().clone().requires_grad_(True)
    Wb = ops.cached_bf16(W)
    yw, yl = (torch.randint(0, V, (B, T), generator=g).to(dev) for _ in range(2))
    pl = pg.PreferenceLoss(CFG["beta"])
    out = {"workload": f"cfg2 shape ({B} pairs, seq {T}, d {d}, V {V}), right-padded captions; PreferenceLoss fwd+bwd on "
                       "LazyLogits, fp32 hidden/weight, reference-free (trainer variant)", "rows": 2 * B * T, "sweep": []}

    def timeit(fn, iters=10, repeats=3):
        # host-latency-bound at few rows (one sync for the row counts, a 206 MB dW allocation per step): the minimum
        # over a few repeats keeps allocator churn left over from the earlier extras out of the number
        best, r = None, None
        for _ in range(repeats):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            best = ms if best is None or ms < best else best
        return best, r

    import gc
    gc.collect()
    torch.cuda.empty_cache()
    for lo, hi in ((10, 20), (40, 60), (T, T)):
        lens = torch.randint(lo, hi + 1, (2, B), generator=g)
        mw, ml = ((torch.arange(T)[None] < lens[i][:, None]).long().to(dev) for i in range(2))
        scored = int(mw[:, 1:].sum() + ml[:, 1:].sum())
        gs = [torch.full((B,), 0.01, device=dev), torch.full((B,), -0.01, device=dev)]

        def module_step():
            W.grad = hw.grad = hl.grad = None
            loss = pl(LazyLogits(hw, W), LazyLogits(hl, W), yw, yl, mw, ml)
            loss.backward()
            return loss

        def kernels_only():  # the C-ABI calls of the same step without autograd / module overhead
            seqs, ctx = F.lmhead_compact_fwd([hw.detach(), hl.detach()], Wb, [yw, yl], [mw, ml], True)
            return F.lmhead_compact_bwd(ctx, Wb, gs)

        ms_mod, loss = timeit(module_step)
        ms_ker, _ = timeit(kernels_only)
        rec = {"caption_tokens": [lo, hi], "scored_rows": scored, "module_ms_per_step": ms_mod,
               "c_abi_ms_per_step": ms_ker, "valid_pair_tokens_per_s": 0.5 * scored / (ms_mod * 1e-3), "loss": loss.item()}
        if lo == 10:
            def full_step():
                W.grad = hw.grad = hl.grad = None
                lw = ops.lmhead_seq_logprob(hw, W, yw, mw, True)[0]
                ll = ops.lmhead_seq_logprob(hl, W, yl, ml, True)[0]
                loss = ops.dpo_loss(lw, ll, None, None, CFG["beta"], 0.0, B)[0]
                loss.backward()
                return loss
            ms_full, loss_f = timeit(full_step)
            rec["all_rows_module_ms_per_step"] = ms_full
            rec["all_rows_loss"] = loss_f.item()
            out["scored_rows"] = scored
            out["speedup"] = ms_full / ms_mod
        out["sweep"].append(rec)
    return out


def torch_eager_extra(torch, dev):
    """The reference's torch path for cfg2 on the SAME B200 (what a user of the reference gets on this GPU without this
    library): F.linear + compute_sequence_logprobs x4 + DPOPreferenceLoss + backward, logits materialised; fp32 with
    TF32 off (the parity setting) and bf16 autocast-free (weights and activations cast to bf16)."""
    fn, kind = reference_cpu_step_fn()
    W, Wr, hs, yc, yr, m = cpu_reference_step_inputs(CFG["pairs"])
    out = {"kind": kind}
    torch.backends.cuda.matmul.allow_tf32 = False
    for name, dt in (("fp32_tf32_off", torch.float32), ("bf16", torch.bfloat16)):
        Wd = W.to(dev, dt).requires_grad_(True)
        Wrd = Wr.to(dev, dt)
        h = [x.to(dev, dt) for x in hs]
        h[0].requires_grad_(True)
        h[1].requires_grad_(True)
        ycd, yrd, md = yc.to(dev), yr.to(dev), m.to(dev)

        def step():
            Wd.grad = h[0].grad = h[1].grad = None
            return fn(h[0], h[1], Wd, ycd, yrd, md, h[2], h[3], Wrd)

        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        out[name] = {"ms_per_step": ms, "pair_tokens_per_s": CFG["pairs"] * (CFG["seq_len"] - 1) / (ms * 1e-3),
                     "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
        del Wd, Wrd, h
        torch.cuda.empty_cache()
    return out


def cfg5_extra():
    """BASELINE config 5 (tools/cfg5_step.py): the reference's own Stage-2 micro-step, unpatched vs install()ed."""
    if os.environ.get("PGICA_BENCH_CFG5", "1") == "0":
        return {"skipped": "PGICA_BENCH_CFG5=0"}
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import cfg5_step
        return cfg5_step.run(batch=8, steps=5, warmup=2, log=log)
    except Exception as e:  # an extra must never take the headline down with it
        return {"error": repr(e)[:300]}


def gradclip_extra(torch, F, dev):
    """SURVEY 8(f) row 2: finite check + global norm + clip over GPT-2-Medium-sized fp32 gradients (355 M elements in
    the tensor shapes of the decoder: wte, 24 x {attn, mlp, ln}), HBM roofline: the norm pass reads every gradient
    once, the clip pass reads and writes it."""
    d, V, L = 1024, CFG["vocab"], 24
    shapes = [(V, d), (1024, d)] + [s for _ in range(L) for s in ((d, 3 * d), (3 * d,), (d, d), (d,), (d, 4 * d),
                                                                   (4 * d,), (4 * d, d), (d,), (d,), (d,), (d,), (d,))]
    grads = [torch.randn(*s, device=dev) * 0.02 for s in shapes]
    nbytes = sum(g.numel() * 4 for g in grads)
    out = {"tensors": len(grads), "elements": nbytes // 4, "dtype": "f32"}
    pk = peaks()
    for name, max_norm, passes in (("norm_only", 1e9, 1), ("norm_and_clip", 1.0, 3)):
        # max_norm halves on every call so that every call of the second variant really clips
        for it in range(2):
            F.grad_norm_clip(grads, max_norm * 0.5 ** it)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for it in range(2, 7):
            F.grad_norm_clip(grads, max_norm * 0.5 ** it)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        out[name] = {"ms": ms, "algorithmic_bytes": passes * nbytes, "gb_per_s": passes * nbytes / ms / 1e6,
                     "frac_of_hbm_peak": passes * nbytes / ms / 1e6 / pk["hbm"]}
    return out


def ntxent_extras(torch, F, dev):
    """NT-Xent pairs/s fwd+bwd: cfg1 (B=64, latency-bound) and a 4096 x 4096 single-GPU batch (D=512, tau=0.5)."""
    out = {}
    one = torch.ones((), device=dev)
    for name, B in (("cfg1_B64", 64), ("B4096", 4096), ("B16384", 16384)):
        a = torch.nn.functional.normalize(torch.randn(B, 512, device=dev), dim=-1).to(torch.bfloat16)
        b = torch.nn.functional.normalize(torch.randn(B, 512, device=dev), dim=-1).to(torch.bfloat16)

        small = F.ntxent_small_supported(B, 512)  # B <= 128: loss and both gradients from ONE single-CTA launch

        def step(unit_norm=True):
            if small:
                return F.ntxent_small(a, b, 2.0, True)[0]
            # unit-norm rows (what the reference model feeds its loss): one pass for both log-sum-exps, one exponential
            # per element in the backward; general inputs: two passes, two exponentials
            lr, dg, lc = F.ntxent_fwd(a, b, 2.0, bounded=unit_norm)
            loss = F.ntxent_loss(lr, dg, lc, 1.0 / B)
            F.ntxent_bwd(a, b, 2.0, 0, lr, lc, one, 1.0 / (2 * B), bounded=unit_norm)
            return loss

        def timed(unit_norm):
            for _ in range(3):
                step(unit_norm)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            iters = 20 if B <= 4096 else 5
            e0.record()
            for _ in range(iters):
                step(unit_norm)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters

        ms = timed(True)
        out[name] = {"pairs_per_s": B / (ms * 1e-3), "us_per_step": ms * 1e3,
                     "algorithmic_tflops": 6.0 * B * B * 512 / ms / 1e9,
                     "launches_per_step": 1 if small else None}
        if not small:
            out[name]["inputs"] = "unit-norm rows promised (one-pass forward, one exponential per element backward)"
            out[name]["us_per_step_general_inputs"] = timed(False) * 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
