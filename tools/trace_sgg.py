"""Cycle accounting of the cluster softmax-gradient GEMM (diagnostics build, -DPGICA_TRACE).

    python tools/trace_sgg.py build      # here (no GPU): compile libpgica_trace.so
    python tools/trace_sgg.py run        # on the B200: cfg2 dH / dW shapes, prints per-role wait breakdowns
"""
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "preference_guided_image_captioning_alignment_b200")
TRACE_LIB = os.path.join(PKG, "libpgica_trace.so")

# layout written by sgg_x.cu (exchange through L2)
NAMES = ["prod_other", "prod_wait_empty_mma1", "prod_wait_empty_mma2", "prod_wait_gready",
         "mma_issue", "mma_wait_zempty_outfree", "mma_wait_full1", "mma_wait_gtile", "mma_wait_full2",
         "epi_other", "epi_wait_zfull", "epi_compute", "epi_wait_stfree", "epi_stage_write", "epi_wait_outfull",
         "epi_unused6", "epi_unused7", "epi_unused8",
         "xw_other", "xw_wait_stfull", "xw_wait_gdone", "xw_store_fence_arrive"]


def build():
    from preference_guided_image_captioning_alignment_b200 import _build
    srcs = _build._sources()
    cmd = [_build.nvcc_path()] + _build.NVCC_FLAGS + ["-DPGICA_TRACE", "-shared", "-o", TRACE_LIB] + srcs
    subprocess.check_call(cmd)
    print(TRACE_LIB)


def run():
    os.environ["PGICA_LIB_PATH"] = TRACE_LIB
    import torch
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F
    lib = _lib.load()
    setter = lib.pgica_debug_set_sggx_trace
    setter.argtypes = [ctypes.c_void_p]
    names = NAMES
    dev = "cuda"
    torch.manual_seed(0)
    for mode, mx, my in (("row", 4064, 50257), ("col", 50257, 4064)):
        k = 1024
        x = (torch.randn(mx, k, device=dev) * (0.5 if mode == "row" else 0.02)).to(torch.bfloat16)
        y = (torch.randn(my, k, device=dev) * (0.02 if mode == "row" else 0.5)).to(torch.bfloat16)
        lse = torch.full((mx if mode == "row" else my,), 11.0, device=dev)
        coef = torch.randn_like(lse)
        tgt = torch.randint(0, my if mode == "row" else mx, lse.shape, device=dev, dtype=torch.int32)
        st = (lse, coef, tgt)
        grid = ((mx + 127) // 128) * 4
        buf = torch.zeros(max(grid, 1024), 24, dtype=torch.int64, device=dev)
        kw = dict(row=st) if mode == "row" else dict(col=st)
        for _ in range(2):
            F.softmax_grad_gemm(x, y, 1.0, **kw)
        assert setter(buf.data_ptr()) == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        F.softmax_grad_gemm(x, y, 1.0, **kw)
        e1.record()
        torch.cuda.synchronize()
        setter(None)
        t = buf.cpu().double()
        t = t[t.sum(1) > 0]  # CTAs that ran (the persistent kernel launches fewer than `grid`)
        grid = t.shape[0]
        tot_mma = t[:, 4:9].sum(1)
        res = {"mode": mode, "grid": grid, "ms": e0.elapsed_time(e1),
               "mma_total_cycles_mean": tot_mma.mean().item(), "mma_total_cycles_max": tot_mma.max().item()}
        for i, n in enumerate(names):
            res[n] = round(t[:, i].mean().item())
        # per cluster rank (q = blockIdx % 4)
        for q in range(4):
            sel = t[q::4]
            res[f"q{q}"] = {n: round(sel[:, i].mean().item()) for i, n in enumerate(names)}
        print(json.dumps(res))


if __name__ == "__main__":
    {"build": build, "run": run}[sys.argv[1]]()
