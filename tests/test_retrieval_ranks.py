"""Retrieval ranks in both directions (scoring.retrieval_ranks_both / retrieval_recall, pgica_retrieval_ranks).

Definitions (S = image @ text.T in fp32 as compute_similarity computes it, owner = text_to_image):
    p_i           = max of S[i, j] over the captions j with owner[j] == i (NaN if any of them is NaN)
    image_rank[i] = #{j : S[i, j] > p_i},            -1 if image i owns no caption
    q_j           = S[owner[j], j]
    text_rank[j]  = #{i : S[i, j] > q_j},            -1 if owner[j] == -1

The tests not marked `gpu` check the host-side validation and run anywhere."""
import ctypes

import pytest
import torch


def reference_ranks(S, owner):
    """The definitions above in torch, on any (Ni, Nt) score matrix and an int64 owner vector on the same device."""
    Ni, Nt = S.shape
    has = owner >= 0
    cols = torch.arange(Nt, device=S.device)[has]
    own = torch.zeros(Ni, Nt, dtype=torch.bool, device=S.device)
    own[owner[has], cols] = True
    p = torch.where(own, S, torch.tensor(float("-inf"), dtype=S.dtype, device=S.device)).amax(dim=1)
    p = torch.where((own & S.isnan()).any(dim=1), torch.tensor(float("nan"), dtype=S.dtype, device=S.device), p)
    image_rank = (S > p[:, None]).sum(dim=1)
    image_rank[~own.any(dim=1)] = -1
    q = torch.full((Nt,), float("nan"), dtype=S.dtype, device=S.device)
    q[cols] = S[owner[has], cols]
    text_rank = (S > q[None, :]).sum(dim=0)
    text_rank[~has] = -1
    return image_rank, text_rank


def default_owner(Ni, Nt, device="cpu"):
    j = torch.arange(Nt, device=device)
    return torch.where(j < Ni, j, torch.full_like(j, -1))


def shuffled_owner(Ni, Nt, gen):
    """Several captions per image in shuffled order, some captions without an image (-1), some images owning nothing."""
    owned = max(1, Ni - Ni // 5)  # the last fifth of the images own nothing
    owner = torch.randint(0, owned, (Nt,), generator=gen)
    owner[torch.randperm(Nt, generator=gen)[: Nt // 7]] = -1
    return owner


def test_reference_ranks_by_hand():
    S = torch.tensor([[3.0, 1.0, 3.0, float("nan")],
                      [0.0, 2.0, 5.0, 1.0],
                      [1.0, 1.0, 1.0, 1.0]])
    owner = torch.tensor([0, 1, 1, -1])
    ir, tr = reference_ranks(S, owner)
    # image 0: p = 3 (caption 0), nothing above it (ties and NaN do not count); image 1: p = max(2, 5) = 5;
    # image 2 owns nothing
    assert ir.tolist() == [0, 0, -1]
    # caption 0: q = 3, nobody above; caption 1: q = 2, nobody above; caption 2: q = 5, nobody above; caption 3: none
    assert tr.tolist() == [0, 0, 0, -1]
    S[1, 1] = float("nan")
    ir, tr = reference_ranks(S, owner)
    assert ir.tolist() == [0, 0, -1] and tr.tolist() == [0, 0, 0, -1]  # NaN threshold: 0
    S[0, 1] = 9.0
    ir, tr = reference_ranks(S, default_owner(3, 4))
    assert ir.tolist() == [1, 0, 0] and tr.tolist() == [0, 0, 2, -1]


# ------------------------------------------------------------------------------------------------ host-side validation
def test_new_functions_refuse_bad_input_before_launch():
    import preference_guided_image_captioning_alignment_b200 as pg
    from preference_guided_image_captioning_alignment_b200 import _lib
    img, txt = torch.randn(6, 16), torch.randn(9, 16)
    for fn in (pg.retrieval_ranks_both, pg.retrieval_recall, pg.retrieval_ranks):
        with pytest.raises(_lib.PgicaError):
            fn(img, txt)  # CPU tensors: no fallback
    for fn in (pg.retrieval_ranks_both, pg.retrieval_recall):
        with pytest.raises(_lib.PgicaError):
            fn(img, txt, torch.zeros(9, dtype=torch.int64))
        for bad in (torch.full((9,), 6), torch.full((9,), -2), torch.zeros(10, dtype=torch.int64),
                    torch.zeros(9, 1, dtype=torch.int64), torch.zeros(9, dtype=torch.float32), [0] * 9,
                    torch.zeros(9, dtype=torch.int16)):
            with pytest.raises(ValueError):
                fn(img, txt, bad)
        for a, b in ((torch.randn(0, 16), txt), (img, torch.randn(0, 16)), (img, torch.randn(9, 8)), (img[0], txt)):
            with pytest.raises(ValueError):
                fn(a, b)
    with pytest.raises(ValueError):
        pg.retrieval_ranks(torch.randn(0, 16), txt)


def test_c_abi_validation_without_gpu():
    from preference_guided_image_captioning_alignment_b200 import _build, _lib
    _build.build()
    lib = _lib.load()
    need = ctypes.c_size_t(0)
    assert lib.pgica_retrieval_ranks_workspace_bytes(65536, 65536, 512, ctypes.byref(need)) == 0
    assert need.value == 256 * 256 + 4 * 65536 * 2  # the tile mask and 4 bytes per row and column: no rows x cols buffer
    assert lib.pgica_retrieval_ranks_workspace_bytes(8192, 40960, 1536, ctypes.byref(need)) == 0
    assert need.value == 32 * 160 + 4 * (8192 + 40960)
    assert lib.pgica_retrieval_ranks_workspace_bytes(128, 256, 1001, ctypes.byref(need)) == -1
    assert b"multiple of 8" in lib.pgica_last_error()
    assert lib.pgica_retrieval_ranks_workspace_bytes(0, 256, 64, ctypes.byref(need)) == -1
    assert lib.pgica_retrieval_ranks_workspace_bytes(256, 0, 64, ctypes.byref(need)) == -1
    if not torch.cuda.is_available():
        assert lib.pgica_retrieval_ranks(None, None, 128, 128, 64, None, None, None, None, 0, None) != 0


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def pg(cuda_device):
    import preference_guided_image_captioning_alignment_b200 as pkg
    from preference_guided_image_captioning_alignment_b200 import _lib
    assert _lib.load().pgica_device_check() == 0, _lib.load().pgica_last_error()
    return pkg


def int_embeddings(n, d, gen, dup):
    """Small integers (every product and sum exact in fp32 and bf16) with `dup` planted duplicate rows and one zero row:
    exact ties inside rows and columns."""
    x = torch.randint(-3, 4, (n, d), generator=gen).float()
    if n > 1:
        src = torch.randint(0, n, (dup,), generator=gen)
        dst = torch.randint(0, n, (dup,), generator=gen)
        x[dst] = x[src]
        x[torch.randint(0, n, (1,), generator=gen)] = 0.0
    return x


INT_SHAPES = [(1, 1, 8), (5, 7, 16), (129, 391, 32), (391, 129, 32), (300, 270, 64), (257, 513, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("pairing", ["default", "shuffled"])
@pytest.mark.parametrize("Ni,Nt,D", INT_SHAPES)
def test_exact_ranks_integer_inputs(pg, cuda_device, Ni, Nt, D, pairing, dtype):
    gen = torch.Generator().manual_seed(Ni * 7919 + Nt * 31 + D)
    img = int_embeddings(Ni, D, gen, dup=max(1, Ni // 10))
    txt = int_embeddings(Nt, D, gen, dup=max(1, Nt // 10))
    if pairing == "default":
        owner, arg = default_owner(Ni, Nt), None
    else:
        owner = shuffled_owner(Ni, Nt, gen)
        # plant positives that tie with other captions of the same image and with other images
        for j in range(0, Nt, 5):
            if owner[j] >= 0:
                txt[(j + 1) % Nt] = txt[j]
        arg = owner.to(cuda_device)
    ir_ref, tr_ref = reference_ranks(img.double() @ txt.double().T, owner)
    ir, tr = pg.retrieval_ranks_both(img.to(dtype).to(cuda_device), txt.to(dtype).to(cuda_device), arg)
    assert ir.dtype == torch.int64 and tr.dtype == torch.int64 and ir.shape == (Ni,) and tr.shape == (Nt,)
    assert torch.equal(ir.cpu(), ir_ref), (ir.cpu() - ir_ref).abs().max()
    assert torch.equal(tr.cpu(), tr_ref), (tr.cpu() - tr_ref).abs().max()
    if pairing == "shuffled" and Ni > 1:
        assert (ir_ref == -1).any() and (tr_ref == -1).any()
    assert (ir_ref >= 1).any() or Ni * Nt < 40  # ties and misses do occur


def unit(n, d, gen):
    return torch.nn.functional.normalize(torch.randn(n, d, generator=gen), dim=-1)


DENSE_CASES = [(4096, 4096, 512, torch.bfloat16, 1, False), (4096, 4096, 512, torch.float32, 1, False),
               (16384, 16384, 512, torch.bfloat16, 1, False), (1000, 5000, 512, torch.float32, 5, False),
               (1000, 5000, 512, torch.bfloat16, 5, True), (777, 777, 256, torch.float32, 1, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("Ni,Nt,D,dtype,per_image,nan_rows", DENSE_CASES)
def test_bitwise_equal_to_dense_path(pg, cuda_device, Ni, Nt, D, dtype, per_image, nan_rows):
    """Both ranks equal the definitions evaluated in torch on compute_similarity(img, txt, 1.0): the same fp32 scores."""
    gen = torch.Generator().manual_seed(Ni + Nt + D)
    img = unit(Ni, D, gen)
    if per_image == 1:
        owner, arg = default_owner(Ni, Nt), None
        txt = unit(Nt, D, gen)
    else:
        owner = torch.arange(Nt) // per_image
        owner = owner[torch.randperm(Nt, generator=gen)]
        txt = torch.nn.functional.normalize(img[owner] + 0.9 * torch.randn(Nt, D, generator=gen), dim=-1)
        arg = owner.to(cuda_device)
    if nan_rows:
        img[Ni // 3] = float("nan")
        txt[Nt // 2] = float("nan")
    img, txt = img.to(dtype).to(cuda_device), txt.to(dtype).to(cuda_device)
    ir, tr = pg.retrieval_ranks_both(img, txt, arg)
    S = pg.compute_similarity(img, txt, 1.0)
    ir_ref, tr_ref = reference_ranks(S, owner.to(cuda_device))
    del S
    assert torch.equal(ir, ir_ref), int((ir != ir_ref).sum())
    assert torch.equal(tr, tr_ref), int((tr != tr_ref).sum())
    if nan_rows:
        assert ir[Ni // 3].item() == 0 and tr[Nt // 2].item() == 0
    assert torch.equal(pg.retrieval_ranks_both(img, txt, arg)[1], tr)  # deterministic
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_retrieval_ranks_is_the_image_half(pg, cuda_device):
    gen = torch.Generator().manual_seed(11)
    for Ni, Nt in ((300, 300), (700, 250), (100, 1000)):
        img, txt = unit(Ni, 128, gen).to(cuda_device), unit(Nt, 128, gen).to(cuda_device)
        r = pg.retrieval_ranks(img, txt)
        both = pg.retrieval_ranks_both(img, txt)
        assert torch.equal(r, both[0]) and torch.equal(r, pg.retrieval_ranks_both(img, txt)[0])
        assert torch.equal(both[1], pg.retrieval_ranks_both(img, txt)[1])
        if Ni > Nt:
            assert bool((r[Nt:] == -1).all()) and bool((r[:Nt] >= 0).all())


@pytest.mark.gpu
def test_recall_from_ranks(pg, cuda_device):
    gen = torch.Generator().manual_seed(5)
    img = unit(500, 256, gen)
    owner = shuffled_owner(500, 2000, gen)
    txt = torch.nn.functional.normalize(img[owner.clamp(min=0)] + 1.2 * torch.randn(2000, 256, generator=gen), dim=-1)
    args = (img.to(cuda_device), txt.to(cuda_device), owner.to(cuda_device))
    ir, tr = (r.cpu() for r in pg.retrieval_ranks_both(*args))
    rec = pg.retrieval_recall(*args, ks=(1, 5, 10))
    for name, r in (("image_to_text", ir), ("text_to_image", tr)):
        valid = r >= 0
        for k in (1, 5, 10):
            assert isinstance(rec[name][k], float)
            assert rec[name][k] == pytest.approx(((r >= 0) & (r < k)).sum().item() / valid.sum().item(), abs=0)
        assert 0.0 < rec[name][1] <= rec[name][5] <= rec[name][10] <= 1.0


@pytest.mark.gpu
def test_fixed_launch_count_and_no_dense_memory(pg, cuda_device):
    from preference_guided_image_captioning_alignment_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator().manual_seed(3)
    deltas = []
    for n in (64, 1000, 5000, 16384):
        img = unit(n, 512, gen).to(torch.bfloat16).to(cuda_device)
        txt = unit(n, 512, gen).to(torch.bfloat16).to(cuda_device)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        n0 = lib.pgica_kernel_launches()
        pg.retrieval_ranks_both(img, txt)
        deltas.append(lib.pgica_kernel_launches() - n0)
        torch.cuda.synchronize()
        if n == 16384:
            grew = torch.cuda.max_memory_allocated() - base
            assert grew < 64 << 20, grew  # the dense path holds a 1 GiB score matrix here
    assert len(set(deltas)) == 1 and deltas[0] == 4, deltas
