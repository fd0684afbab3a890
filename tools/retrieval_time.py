"""Retrieval ranks in both directions: the dense path (compute_similarity(img, txt, 1.0), then both torch comparisons
and sums) against the fused call (scoring.retrieval_ranks_both: two passes over the similarity tiles, no score matrix).

Alternates the two in one process after a warm-up and keeps the minimum window time over --windows windows.  Records,
per shape: time, peak allocated memory of one call, whether both ranks are equal, and achieved TFLOP/s (2 Ni Nt K with
K = D for bf16 inputs and 3 D for fp32 inputs, which go in as the two-term bf16 split).  Inputs are unit-norm random
rows, each caption a noisy copy of its image's embedding.

    python tools/retrieval_time.py [--out retrieval_time.json] [--windows 5] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import preference_guided_image_captioning_alignment_b200 as pg  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": out[0], "power_limit": out[1], "max_sm_clock": out[2]}
    except Exception:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "?", "max_sm_clock": "?"}


def dense_ranks(img, txt, owner):
    S = pg.compute_similarity(img, txt, 1.0)
    Ni, Nt = S.shape
    if owner is None:
        d = S.diagonal()  # square galleries only: caption i belongs to image i
        return (S > d[:, None]).sum(dim=1), (S > d[None, :]).sum(dim=0)
    q = S[owner, torch.arange(Nt, device=S.device)]
    p = torch.full((Ni,), float("-inf"), device=S.device).scatter_reduce(0, owner, q, "amax")
    return (S > p[:, None]).sum(dim=1), (S > q[None, :]).sum(dim=0)


def timed(fn, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3


def peak_mb(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2**20, out


def case(Ni, Nt, D, dtype, per_image, windows, gen):
    dev = torch.device("cuda", 0)
    img = torch.nn.functional.normalize(torch.randn(Ni, D, generator=gen), dim=-1)
    if per_image:
        owner = (torch.arange(Nt) // per_image)[torch.randperm(Nt, generator=gen)]
        txt = torch.nn.functional.normalize(img[owner] + torch.randn(Nt, D, generator=gen), dim=-1)
        owner = owner.to(dev)
    else:
        owner = None
        txt = torch.nn.functional.normalize(img + torch.randn(Nt, D, generator=gen), dim=-1)
    img, txt = img.to(dtype).to(dev), txt.to(dtype).to(dev)
    dense = lambda: dense_ranks(img, txt, owner)
    fused = lambda: pg.retrieval_ranks_both(img, txt, owner)
    mem_dense, ref = peak_mb(dense)
    mem_fused, got = peak_mb(fused)
    equal = torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
    del ref, got
    torch.cuda.empty_cache()
    iters = max(1, int(2**33 // (Ni * Nt)))  # about the same number of scores per window at every size
    times = {"dense": [], "fused": []}
    for _ in range(windows):
        times["dense"].append(timed(dense, iters))
        torch.cuda.empty_cache()
        times["fused"].append(timed(fused, iters))
    K = D if dtype == torch.bfloat16 else 3 * D
    flop = 2.0 * Ni * Nt * K
    res = {"Ni": Ni, "Nt": Nt, "D": D, "K": K, "dtype": str(dtype).replace("torch.", ""),
           "captions_per_image": per_image or 1, "owner_order": "shuffled" if per_image else "default",
           "iters_per_window": iters, "ms_min": {k: min(v) for k, v in times.items()},
           "ms_all": times, "peak_alloc_mb": {"dense": round(mem_dense, 1), "fused": round(mem_fused, 1)},
           "ranks_equal": bool(equal)}
    res["tflops"] = {k: flop / (res["ms_min"][k] * 1e-3) / 1e12 for k in times}
    res["speedup"] = res["ms_min"]["dense"] / res["ms_min"]["fused"]
    print(json.dumps({k: res[k] for k in ("Ni", "Nt", "dtype", "ms_min", "peak_alloc_mb", "ranks_equal", "tflops",
                                          "speedup")}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="retrieval_time.json", help="where the JSON result goes")
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="small shapes only (a check that the script runs)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "retrieval_time.py measures on the GPU; there is nothing to time without one"
    gen = torch.Generator().manual_seed(0)
    sizes = (1024, 2048) if args.quick else (4096, 16384, 32768, 65536)
    results = []
    for n in sizes:
        for dtype in (torch.bfloat16, torch.float32):
            results.append(case(n, n, 512, dtype, 0, args.windows, gen))
    gallery = (1024, 5120) if args.quick else (8192, 40960)
    for dtype in (torch.bfloat16, torch.float32):
        results.append(case(gallery[0], gallery[1], 512, dtype, 5, args.windows, gen))
    out = {"gpu": card(), "windows": args.windows, "timing": "host clock around iters calls ending in a device "
           "synchronise; minimum over windows, dense and fused alternating", "cases": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
