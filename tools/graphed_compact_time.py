"""Per-step device time (CUDA events) and host enqueue time of the DPO head at cfg2's shape (16 pairs, T = 128,
d = 1024, V = 50257, frozen reference) for three ways of running it, at the reference's caption statistics (470 / 1555 /
4064 scored rows of 4096):

  graphed_all_rows   GraphedDPOStep: CUDA graphs of FusedDPOHead.forward_stacked + backward, GEMMs over every row
  eager_compact      functional.lmhead_compact_fwd / _bwd + DPO scalar head, launched from Python (one host read of
                     the row counts per forward)
  graphed_compact    GraphedCompactDPOStep: graphs per 256-row bucket, row count kept on the device

Each step copies its labels and mask from pinned host memory and reads its loss back, as a training loop does.
Outputs of graphed_compact are checked against eager_compact at every timed size.  Inputs total ~1 GB per step
(weights, hidden states), larger than L2.  One JSON line per (rows, path), plus the card's name and power limit, on
stdout and, with --out, into that file.

    python tools/graphed_compact_time.py [--steps 50] [--warmup 10] [--out profiles/graphed_compact_time.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("graphed_compact_time.py needs a B200")
    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200 import functional as F
    from test_graphed_compact import caption_masks, eager_step

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, T, d, V = 16, 128, 1024, 50257
    gen = torch.Generator().manual_seed(0)
    W = (torch.randn(V, d, generator=gen) * 0.05).bfloat16().to(dev)
    Wr = (torch.randn(V, d, generator=gen) * 0.05).bfloat16().to(dev)
    H = torch.randn(2 * B, T, d, generator=gen).to(dev)
    Hr = torch.randn(2 * B, T, d, generator=gen).to(dev)
    y = torch.randint(0, V, (2 * B, T), generator=gen)
    yp = y.pin_memory()
    yd = y.to(dev)
    head = pg.FusedDPOHead(beta=0.1)
    Wp = W.float().requires_grad_(True)  # fp32 master weight, as bench.py's end-to-end arm
    info = {"card": card(), "shape": [B, T, d, V], "steps": args.steps}
    print(json.dumps(info))
    lines = [info]

    def timed(issue, read):
        for _ in range(args.warmup):
            issue()
            read()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        host = 0.0
        start.record()
        for _ in range(args.steps):
            t0 = time.perf_counter()
            issue()
            host += time.perf_counter() - t0
            read()
        end.record()
        end.synchronize()
        return start.elapsed_time(end) / args.steps, 1e3 * host / args.steps

    for n in (470, 1555, 4064):
        m = caption_masks(2 * B, T, n, seed=n)
        mp, md = m.pin_memory(), m.to(dev)
        full = pg.GraphedDPOStep(head, Wp, Wr, H, yd, md, Hr)

        def issue_full():
            full.copy_inputs(H, yp, mp, Hr)
            full.launch()

        def issue_eager():
            yd.copy_(yp, non_blocking=True)
            md.copy_(mp, non_blocking=True)
            issue_eager.loss = eager_step(F, H, W, yd, md, Hr, Wr, False)["loss"]

        mem0 = torch.cuda.memory_reserved()
        comp = pg.GraphedCompactDPOStep(head, Wp, Wr, H, y, m, Hr)
        comp.copy_inputs(H, yp, mp, Hr)
        comp.launch()
        comp.loss_value()
        torch.cuda.synchronize()
        pool_mb = (torch.cuda.memory_reserved() - mem0) / 2 ** 20

        def issue_comp():
            comp.copy_inputs(H, yp, mp, Hr)
            comp.launch()

        ref = eager_step(F, H, W, yd, md, Hr, Wr, False)
        torch.cuda.synchronize()
        check = {"loss_abs_diff": abs(float(comp.loss) - float(ref["loss"])),
                 "dW_rel": float((comp.dweight - ref["dw"]).norm() / ref["dw"].norm()),
                 "dH_rel": float((comp.dhidden - ref["dh"]).norm() / ref["dh"].norm()),
                 "metrics_max_abs_diff": float((comp.metrics - ref["metrics"]).abs().max())}
        for name, issue, read in (("graphed_all_rows", issue_full, full.loss_value),
                                  ("eager_compact", issue_eager, lambda: float(issue_eager.loss)),
                                  ("graphed_compact", issue_comp, comp.loss_value)):
            dev_ms, host_ms = timed(issue, read)
            line = {"rows": n, "path": name, "ms_per_step": round(dev_ms, 4), "host_enqueue_ms": round(host_ms, 4)}
            if name == "graphed_compact":
                line.update(bucket=comp.rows_launch, new_memory_mb=round(pool_mb, 1), check_vs_eager=check)
            print(json.dumps(line))
            lines.append(line)
        del full, comp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
