"""CPU tests (no GPU, no compute calls): the C-ABI library builds, loads and exports every symbol that
include/pgica.h declares; host-side argument validation; the Python mirror of the reference interface."""
import ctypes
import os
import re
import subprocess
import sys
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from preference_guided_image_captioning_alignment_b200 import _build, _lib
    _build.build()
    return _lib.load()


def test_header_symbols_exported(lib):
    from preference_guided_image_captioning_alignment_b200 import _lib
    protos = _lib.parse_header()
    text = open(_lib.HEADER_PATH).read() + open(_lib.DEBUG_HEADER_PATH).read()
    declared = set(re.findall(r"\b(pgica_\w+)\s*\(", text))
    assert declared == set(protos), "header parser missed a prototype"
    assert len(declared) >= 50
    # bring-up / test hooks live in pgica_debug.h, not in the product header
    product = set(re.findall(r"\b(pgica_\w+)\s*\(", open(_lib.HEADER_PATH).read()))
    assert not {n for n in product if "debug" in n or "probe" in n}
    assert {"pgica_set_option", "pgica_get_option", "pgica_compact_rows", "pgica_lmhead_rows_bwd"} <= product
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (pgica_\w+)", out))
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.pgica_abi_version() == 1


def test_every_entry_point_cites_the_reference():
    text = open(os.path.join(ROOT, "include", "pgica.h")).read()
    for needle in ("pkg/models/components.py:321-362", "pkg/models/model.py:1052-1085", "pkg/models/components.py:192-249",
                   "pkg/models/model.py:970-1000", "pkg/models/components.py:117-145", "modeling_gpt2.py:706"):
        assert needle in text


def test_library_is_sm100a_only(lib):
    from preference_guided_image_captioning_alignment_b200 import _build, _lib
    # the cuobjdump of the toolkit that built the library: CUDA's bin directory need not be on PATH
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(_build.nvcc_path())), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_host_side_validation_without_gpu(lib):
    need = ctypes.c_size_t(0)
    assert lib.pgica_gemm_lse_workspace_bytes(4064, 50257, 1024, ctypes.byref(need)) == 0
    assert 0 < need.value < (1 << 28)
    assert lib.pgica_gemm_lse_workspace_bytes(128, 256, 1001, ctypes.byref(need)) == -1
    assert b"multiple of 8" in lib.pgica_last_error()
    assert lib.pgica_gemm_lse_workspace_bytes(0, 256, 64, ctypes.byref(need)) == -1
    assert lib.pgica_lmhead_logprob_workspace_bytes(32, 128, 1024, 50257, ctypes.byref(need)) == 0
    assert need.value >= 32 * 128 * 4
    assert lib.pgica_ntxent_workspace_bytes(4096, 32768, 512, ctypes.byref(need)) == 0
    if not torch.cuda.is_available():
        # the product path fails loudly without a B200; it never computes on the host
        assert lib.pgica_device_check() != 0
        assert lib.pgica_last_error()
        assert lib.pgica_gemm_lse(None, None, 128, 128, 64, 1.0, None, 0, None, None, None, 0, None) != 0


def test_no_cpu_fallback_in_python_layer():
    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200._lib import PgicaError
    a, b = torch.randn(4, 64), torch.randn(4, 64)
    with pytest.raises(PgicaError):
        pg.ContrastiveLoss(0.07)(a, b)
    with pytest.raises(PgicaError):
        pg.PreferenceLoss(0.1)(torch.randn(2, 5, 11), torch.randn(2, 5, 11), torch.zeros(2, 5, dtype=torch.long),
                               torch.zeros(2, 5, dtype=torch.long), torch.ones(2, 5), torch.ones(2, 5))
    with pytest.raises(PgicaError):
        pg.DPOPreferenceLoss()(torch.zeros(3), torch.zeros(3))
    # nothing in the product package imports the oracle
    pkg_dir = os.path.dirname(pg.__file__)
    for f in os.listdir(pkg_dir):
        if f.endswith(".py"):
            src = open(os.path.join(pkg_dir, f)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b|import_module\([\"']oracle", src, flags=re.M), f


def test_module_interface_mirrors_reference():
    import inspect

    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200 import components, losses
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(losses.ContrastiveLoss.__init__) == ["self", "temperature"]
    assert sig(losses.ContrastiveLoss.forward) == ["self", "image_embeddings", "text_embeddings"]
    assert inspect.signature(losses.ContrastiveLoss.__init__).parameters["temperature"].default == 0.07
    assert sig(losses.PreferenceLoss.forward) == ["self", "preferred_logits", "rejected_logits", "preferred_labels",
                                                  "rejected_labels", "preferred_mask", "rejected_mask"]
    assert sig(losses.PreferenceLoss._compute_log_probs) == ["self", "logits", "labels", "mask"]
    assert sig(components.ContrastiveLoss.__init__) == ["self", "temperature", "reduction"]
    assert sig(components.ContrastiveLoss.forward) == ["self", "vision_embeds", "text_embeds"]
    assert sig(components.DPOPreferenceLoss.__init__) == ["self", "beta", "reference_free", "label_smoothing"]
    assert sig(components.DPOPreferenceLoss.forward) == ["self", "policy_chosen_logprobs", "policy_rejected_logprobs",
                                                         "reference_chosen_logprobs", "reference_rejected_logprobs"]
    assert sig(components.compute_sequence_logprobs) == ["logits", "labels", "attention_mask"]
    assert sig(components.TemperatureScaledSimilarity.__init__) == ["self", "temperature", "learnable", "min_temp",
                                                                    "max_temp"]
    # state: trainer-variant losses hold plain floats; the similarity module owns a `temperature` buffer
    assert list(pg.ContrastiveLoss(0.3).state_dict()) == [] and pg.ContrastiveLoss(0.3).temperature == 0.3
    assert list(pg.PreferenceLoss(0.2).state_dict()) == [] and pg.PreferenceLoss(0.2).beta == 0.2
    assert list(components.ContrastiveLoss(0.5).state_dict()) == ["similarity.temperature"]
    sim = components.TemperatureScaledSimilarity(0.07)
    assert sim.effective_temperature() == pytest.approx(0.1)       # clamp, components.py:78
    assert components.TemperatureScaledSimilarity(5.0).effective_temperature() == 2.0
    assert isinstance(components.TemperatureScaledSimilarity(0.5, learnable=True).temperature, torch.nn.Parameter)


def test_mask_kind_and_lazy_logits():
    from preference_guided_image_captioning_alignment_b200 import functional as F
    from preference_guided_image_captioning_alignment_b200.losses import LazyLogits
    assert F.mask_kind(None) == (0, None)
    assert F.mask_kind(torch.ones(2, 3, dtype=torch.long))[0] == F.MASK_I64
    assert F.mask_kind(torch.ones(2, 3))[0] == F.MASK_F32
    assert F.mask_kind(torch.ones(2, 3, dtype=torch.bool))[0] == F.MASK_U8
    assert F.mask_kind(torch.ones(2, 3, dtype=torch.int32))[0] == F.MASK_I32
    assert F.mask_kind(torch.ones(2, 3, dtype=torch.float64))[0] == F.MASK_F32
    h, w = torch.randn(2, 5, 8), torch.randn(11, 8)
    z = LazyLogits(h, w)
    assert z.shape == (2, 5, 11) and z.size(-1) == 11 and z.dim() == 3
    torch.testing.assert_close(z.materialize(), h @ w.T)


def test_fake_tensor_propagation():
    """The custom ops carry meta kernels (shape/dtype inference without a device)."""
    from torch._subclasses.fake_tensor import FakeTensorMode

    from preference_guided_image_captioning_alignment_b200 import ops
    with FakeTensorMode():
        a, b = torch.empty(64, 512), torch.empty(64, 512)
        loss, lr, lc = ops.ntxent(a, b, 2.0, True)
        assert loss.shape == () and lr.shape == (64,) and lc.shape == (64,)
        h, w = torch.empty(4, 16, 128), torch.empty(1000, 128)
        out = ops.lmhead_seq_logprob(h, w, torch.empty(4, 16, dtype=torch.long), None, True)
        assert out[0].shape == (4,) and out[1].shape == (64,) and out[3].dtype == torch.int32
        loss, met, dpc = ops.dpo_loss(torch.empty(8), torch.empty(8), None, None, 0.1, 0.0, 8)
        assert met.shape == (5,) and dpc.shape == (8,)


def test_install_rebinds_reference_names():
    import importlib

    from preference_guided_image_captioning_alignment_b200 import components, losses
    install = importlib.import_module("preference_guided_image_captioning_alignment_b200.install")
    pkg = types.ModuleType("fake_ref")
    models = types.ModuleType("fake_ref.models")
    model = types.ModuleType("fake_ref.models.model")
    comp = types.ModuleType("fake_ref.models.components")
    training = types.ModuleType("fake_ref.training")
    trainer = types.ModuleType("fake_ref.training.trainer")
    sentinel = object()
    for m in (model, models, trainer):
        m.ContrastiveLoss = sentinel
        m.PreferenceLoss = sentinel
    for n in ("ContrastiveLoss", "DPOPreferenceLoss", "TemperatureScaledSimilarity", "compute_sequence_logprobs"):
        setattr(comp, n, sentinel)
    mods = {"fake_ref": pkg, "fake_ref.models": models, "fake_ref.models.model": model,
            "fake_ref.models.components": comp, "fake_ref.training": training, "fake_ref.training.trainer": trainer}
    sys.modules.update(mods)
    try:
        done = install.install("fake_ref", fuse_lm_head=False)
        assert trainer.ContrastiveLoss is losses.ContrastiveLoss and trainer.PreferenceLoss is losses.PreferenceLoss
        assert model.ContrastiveLoss is losses.ContrastiveLoss and models.PreferenceLoss is losses.PreferenceLoss
        assert comp.DPOPreferenceLoss is components.DPOPreferenceLoss
        assert ("fake_ref.training.trainer", "PreferenceLoss") in done
        install.uninstall()
        assert trainer.ContrastiveLoss is sentinel and comp.compute_sequence_logprobs is sentinel
    finally:
        for k in mods:
            sys.modules.pop(k, None)


def test_shard_pairs():
    from preference_guided_image_captioning_alignment_b200.distributed import shard_pairs
    for n, w in [(256, 8), (16, 1), (10, 4), (3, 8)]:
        spans = [shard_pairs(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1


def test_dual_backward_planner_host_side():
    """pgica_softmax_grad_gemm_dual_plan is host arithmetic: the role split uses every resident CTA pair, respects the
    TMEM capacity of the holders, and keeps X in one chunk when asked to (bf16 / scattered OutY)."""
    import ctypes

    from preference_guided_image_captioning_alignment_b200 import _lib
    lib = _lib.load()
    out = (ctypes.c_int32 * 6)()
    for mx, my, k in ((4096, 50257, 1024), (32768, 50257, 1024), (64, 64, 512), (4096, 4096, 512), (32768, 32768, 512),
                      (4096, 32768, 1536), (300, 1000, 2048)):
        S = k // 512
        rb2, j2 = ((mx + 127) // 128 + 1) // 2, ((my + 127) // 128 + 1) // 2
        for npairs in (74, 66, 8):
            for single in (0, 1):
                assert lib.pgica_softmax_grad_gemm_dual_plan(mx, my, k, npairs, single, out) == 0
                r2, c2, nh, nw, npr, cg = list(out)
                assert cg == 1
                if npairs < 2 * S + 1 or (single and rb2 * S > npairs - S - 1):
                    assert r2 == 0  # no split / not in one chunk: the caller falls back to one launch per product
                    continue
                assert nh == r2 * S and nw == c2 * S and nh + nw + npr == npairs and npr >= 1
                assert 1 <= r2 <= rb2 and 1 <= c2 <= j2
                if single:
                    assert r2 == rb2
    assert lib.pgica_softmax_grad_gemm_dual_plan(4096, 50257, 1000, 74, 0, out) != 0  # k must be a multiple of 512
    # few row blocks + column groups allowed (flags bit 1): several X-holder pairs share the sweep over the vocabulary
    for mx in (218, 470, 900):
        assert lib.pgica_softmax_grad_gemm_dual_plan(mx, 50257, 1024, 74, 2, out) == 0
        r2, c2, nh, nw, npr, cg = list(out)
        rb2 = ((mx + 127) // 128 + 1) // 2
        assert r2 == rb2 and cg > 1 and nh == r2 * 2 * cg and nh + nw + npr == 74 and npr >= 1


@pytest.mark.parametrize("rb2,j2,r2,c2", [(16, 197, 16, 9), (16, 197, 8, 11), (3, 5, 2, 4), (7, 6, 3, 2), (1, 1, 1, 1),
                                           (5, 40, 5, 3), (22, 22, 22, 22), (4, 9, 3, 9)])
@pytest.mark.parametrize("spread", [0, 1])
@pytest.mark.parametrize("groups", [1, 3])
def test_dual_backward_schedule_is_consistent(rb2, j2, r2, c2, spread, groups):
    """The three roles of the dual backward kernel walk ONE schedule (replayed on the host by the enumerators the
    device code runs): every (row pair, column pair) quad is produced exactly once; every X-holder consumes exactly the
    quads of its row pair and every Y-holder exactly those of its column pair, both in increasing production order
    (the kernel's deadlock-freedom argument); accumulation periods start where they must."""
    import ctypes

    import numpy as np

    from preference_guided_image_captioning_alignment_b200 import _lib
    lib = _lib.load()

    if groups > 1 and (r2 < rb2 or groups > j2):
        pytest.skip("column groups need all of x in one chunk and at least one column pair per group")
    sp = spread | (groups << 8)

    def replay(role, idx, width):
        dummy = np.zeros(1, np.int32)
        n = lib.pgica_debug_dual_schedule(rb2, j2, r2, c2, sp, role, idx, ctypes.c_void_p(dummy.ctypes.data), 0)
        assert n >= 0
        buf = np.zeros((max(n, 1), width), dtype=np.int32)
        assert lib.pgica_debug_dual_schedule(rb2, j2, r2, c2, sp, role, idx, ctypes.c_void_p(buf.ctypes.data), n) == n
        return buf[:n]

    quads = replay(0, 0, 3)
    assert len(quads) == rb2 * j2
    assert np.array_equal(quads[:, 0], np.arange(rb2 * j2))                       # q numbers every quad once, in order
    assert len({(r, c) for _, r, c in quads}) == rb2 * j2                          # every (row pair, column pair) once
    where = {(int(r), int(c)): int(q) for q, r, c in quads}
    # X-holders: slot `idx` of a chunk serves row pairs idx, idx + r2, ... ; one accumulation period per chunk.  With
    # column groups slot = (row pair) * groups + g serves only the column pairs cp with cp % groups == g.
    seen_x = set()
    for slot in range(min(r2, rb2) * groups):
        idx, grp = slot // groups, slot % groups
        tiles = replay(1, slot, 6)
        assert len(tiles) > 0
        assert np.all(np.diff(tiles[:, 0]) >= 0)                                   # production order
        assert np.array_equal(tiles[0::2, 1], np.zeros(len(tiles) // 2)) and np.array_equal(tiles[1::2, 1], np.ones(len(tiles) // 2))
        for q, sel, rp, cp, first, period in tiles[0::2]:
            assert where[(rp, cp)] == q and rp % r2 == idx and period == rp // r2 and cp % groups == grp
            assert (int(rp), int(cp)) not in seen_x                                # exactly one group accumulates a quad
            seen_x.add((int(rp), int(cp)))
        starts = tiles[tiles[:, 4] == 1]
        assert len(starts) == len({int(t[5]) for t in tiles}) and np.all(starts[:, 1] == 0)
    assert seen_x == set(where)
    # Y-holders: slot `idx` of a pass serves column pairs idx, idx + c2, ... ; one period per (chunk, pass)
    seen_y = set()
    for idx in range(min(c2, j2)):
        tiles = replay(2, idx, 6)
        assert np.all(np.diff(tiles[:, 0]) >= 0)
        for q, sel, rp, cp, first, period in tiles[0::2]:
            assert where[(rp, cp)] == q and cp % c2 == idx
            seen_y.add((int(rp), int(cp)))
        periods = {}
        for q, sel, rp, cp, first, period in tiles:
            periods.setdefault(int(period), []).append((int(rp // r2), int(cp), int(first)))
        for recs in periods.values():
            assert len({(ch, cp) for ch, cp, _ in recs}) == 1 and recs[0][2] == 1 and sum(f for _, _, f in recs) == 1
    assert seen_y == set(where)


def test_new_entry_points_refuse_cpu_tensors():
    """No CPU fallback anywhere: the dual backward, the graphed step and the gradient-norm module raise on CPU tensors."""
    import torch

    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200 import _lib
    from preference_guided_image_captioning_alignment_b200 import functional as F
    x = torch.randn(128, 512).to(torch.bfloat16)
    with pytest.raises(_lib.PgicaError):
        F.softmax_grad_gemm_dual(x, x, 1.0, row=(torch.zeros(128), torch.ones(128), None))
    p = torch.nn.Parameter(torch.zeros(10))
    p.grad = torch.ones(10)
    with pytest.raises(_lib.PgicaError):
        pg.NaNSafeGradientNorm(max_norm=1.0)([p])
    with pytest.raises(ValueError):
        pg.NaNSafeGradientNorm(norm_type=1.0)
    with pytest.raises(RuntimeError):
        pg.GraphedDPOStep(pg.FusedDPOHead(), torch.zeros(8, 4), None, torch.zeros(2, 3, 4),
                          torch.zeros(2, 3, dtype=torch.long), None)
    assert pg.NaNSafeGradientNorm()([torch.nn.Parameter(torch.zeros(3))])[1] is True  # no gradients: (0, True) like the reference
