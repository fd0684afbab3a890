// K2/K4: the backward of both loss heads as one "softmax-gradient GEMM":
//
//   Out[i, :] = sum_j G(i, j) * Y[j, :]         G(i, j) = rC[i] * (exp(s*z_ij - rL[i]) - [j == rT[i]])
//                                                       + cC[j] * (exp(s*z_ij - cL[j]) - [i == cT[j]])
//   z_ij = <X[i, :], Y[j, :]>   recomputed tile by tile on the tensor cores; G never leaves the SM.
//
//   DPO dH : X = H (tokens),  Y = W (vocab),  row term only   (rC = -coef, rL = lse, rT = label)
//   DPO dW : X = W (vocab),   Y = H (tokens), column term only
//   NT-Xent dA / dB : X = a / b, Y = b / a, both terms (row and column log-sum-exp)
//
// One CTA owns a 128-row x 256-column block of Out, resident in TMEM (256 columns) for the whole loop over
// the 128-row tiles of Y.  Per tile: MMA1 (128x128xK) -> Z in TMEM (double-buffered) -> epilogue warps turn Z
// into the bf16 G tile in shared memory (K-major, 128-B swizzle) -> MMA2 (128x256x128) accumulates into Out
// with the Y tile read MN-major.  Operands stream through one TMA ring of 32-KB slots.
#include <stdlib.h>

#include "common.h"
#include "sgg_tile.cuh"

namespace pgica {
namespace {

constexpr int kBM = 128;        // rows of X / Out per CTA
constexpr int kBT = 128;        // rows of Y per tile (N of MMA1, K of MMA2)
constexpr int kBD = 256;        // Out columns per CTA (N of MMA2)
constexpr int kBK = 64;         // k-chunk (one 128-B swizzle row)
constexpr int kSlots = 6;       // ring depth (even: a two-slot item never wraps)
constexpr uint32_t kChunkBytes = 128 * kBK * 2;   // 16 KB: a [128][64] bf16 box
constexpr uint32_t kSlotBytes = 2 * kChunkBytes;  // 32 KB
constexpr uint32_t kPBytes = kBM * kBT * 2;       // 32 KB
constexpr int kThreads = 256;

constexpr uint32_t kTmemOut = 0, kTmemZ = 256;  // column offsets: Out [0,256), Z0 [256,384), Z1 [384,512)

struct SggParams {
  int mx, my, k, num_tiles, passes, ldo, out_bf16;
  SoftmaxGradStats st;
  void* out;
};

constexpr size_t kSggSmem = 1024 + kSlots * kSlotBytes + kPBytes + 3 * kBT * 4 + 256;

template <bool kRow, bool kCol>
__global__ void __launch_bounds__(kThreads, 1)
sgg_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_y, const SggParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* ring = smem;
  uint8_t* p_tile = smem + kSlots * kSlotBytes;
  float* s_col = reinterpret_cast<float*>(p_tile + kPBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_col + 3 * kBT);
  uint64_t* empty_bar = full_bar + kSlots;
  uint64_t* zfull_bar = empty_bar + kSlots;   // [2]
  uint64_t* zempty_bar = zfull_bar + 2;       // [2]
  uint64_t* pfull_bar = zempty_bar + 2;
  uint64_t* pfree_bar = pfull_bar + 1;
  uint64_t* out_bar = pfree_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(out_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_blk = blockIdx.x / p.passes;
  const int q = blockIdx.x - m_blk * p.passes;
  const int num_kb = (p.k + kBK - 1) / kBK;
  const bool pad = (num_kb & 1) != 0;
  const int J = p.num_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_y);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kSlots; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&zfull_bar[i], 1);
      mbar_init(&zempty_bar[i], 128);
    }
    mbar_init(pfull_bar, 128);
    mbar_init(pfree_bar, 1);
    mbar_init(out_bar, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // (whole warp walks the schedule so that control flow stays warp-uniform; one elected lane issues the copies)
    int slot = 0;
    uint32_t phase = 0;
    auto advance = [&]() {
      if (++slot == kSlots) {
        slot = 0;
        phase ^= 1;
      }
    };
    auto load_mma1 = [&](int j) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[slot], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full_bar[slot], kSlotBytes);
          uint8_t* dst = ring + slot * kSlotBytes;
          tma_load_2d(dst, &tm_x, &full_bar[slot], kb * kBK, m_blk * kBM);
          tma_load_2d(dst + kChunkBytes, &tm_y, &full_bar[slot], kb * kBK, j * kBT);
        }
        __syncwarp();
        advance();
      }
      if (pad) {  // keep every item an even number of slots
        mbar_wait(&empty_bar[slot], phase ^ 1);
        if (elect_one()) mbar_expect_tx(&full_bar[slot], 0);
        __syncwarp();
        advance();
      }
    };
    auto load_mma2 = [&](int j) {  // Y[j tile, q*256 .. +256) as four [128][64] boxes in two slots
      for (int h = 0; h < 2; ++h) {
        mbar_wait(&empty_bar[slot], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full_bar[slot], kSlotBytes);
          uint8_t* dst = ring + slot * kSlotBytes;
          tma_load_2d(dst, &tm_y, &full_bar[slot], q * kBD + (2 * h) * kBK, j * kBT);
          tma_load_2d(dst + kChunkBytes, &tm_y, &full_bar[slot], q * kBD + (2 * h + 1) * kBK, j * kBT);
        }
        __syncwarp();
        advance();
      }
    };
    for (int j = 0; j < J; ++j) {
      load_mma1(j);
      if (j > 0) load_mma2(j - 1);
    }
    load_mma2(J - 1);
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, one elected lane)
    constexpr uint32_t idesc1 = make_idesc_bf16(kBM, kBT, 0, 0);
    constexpr uint32_t idesc2 = make_idesc_bf16(kBM, kBD, 0, 1);
    const uint64_t desc_k = make_smem_desc(0, 16, 1024);            // K-major operand, start address 0
    const uint64_t desc_mn = make_smem_desc(0, kChunkBytes, 1024);  // MN-major operand (Y tile of MMA2)
    int slot = 0;
    uint32_t phase = 0;
    auto advance = [&]() {
      if (++slot == kSlots) {
        slot = 0;
        phase ^= 1;
      }
    };
    uint32_t pphase = 0;
    const uint32_t p_addr = smem_u32(p_tile);
    auto mma2 = [&](int j) {
      mbar_wait(pfull_bar, pphase);
      pphase ^= 1;
      mbar_wait(&full_bar[slot], phase);
      const int slot2 = slot + 1;  // never wraps: items are even-sized, ring is even
      mbar_wait(&full_bar[slot2], phase);
      tc_fence_after_sync();
      if (elect_one()) {
        const uint32_t y_addr = smem_u32(ring + slot * kSlotBytes);
        const uint64_t dg = desc_k | ((p_addr >> 4) & 0x3FFF);
        const uint64_t dy = desc_mn | ((y_addr >> 4) & 0x3FFF);
#pragma unroll
        for (int ks = 0; ks < kBT / 16; ++ks)
          umma_bf16_ss(tmem_base + kTmemOut, dg + (ks >> 2) * (kChunkBytes >> 4) + (ks & 3) * 2,
                       dy + ks * (16 * 128 >> 4), idesc2, (j | ks) != 0 ? 1u : 0u);
        umma_commit(&empty_bar[slot]);
        umma_commit(&empty_bar[slot2]);
        umma_commit(pfree_bar);
      }
      __syncwarp();
      advance();
      advance();
    };
    int zb = 0;
    uint32_t zphase = 0;
    for (int j = 0; j < J; ++j) {
      mbar_wait(&zempty_bar[zb], zphase ^ 1);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + kTmemZ + zb * kBT;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[slot], phase);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t x_addr = smem_u32(ring + slot * kSlotBytes);
          const uint64_t da = desc_k | ((x_addr >> 4) & 0x3FFF);
          const uint64_t db = desc_k | (((x_addr + kChunkBytes) >> 4) & 0x3FFF);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) umma_bf16_ss(d_tmem, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[slot]);
          if (kb == num_kb - 1) umma_commit(&zfull_bar[zb]);
        }
        __syncwarp();
        advance();
      }
      if (pad) {
        mbar_wait(&full_bar[slot], phase);
        if (elect_one()) mbar_arrive(&empty_bar[slot]);
        __syncwarp();
        advance();
      }
      if (++zb == 2) {
        zb = 0;
        zphase ^= 1;
      }
      if (j > 0) mma2(j - 1);
    }
    mma2(J - 1);
    if (elect_one()) umma_commit(out_bar);
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: Z -> G (bf16, smem)
    const int quarter = warp & 3;
    const int et = threadIdx.x - 128;  // 0..127
    const int row_in_blk = quarter * 32 + lane;
    const int row = m_blk * kBM + row_in_blk;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    float rl, rc;
    int rt;
    load_row_stat<kRow>(p.st, row, row < p.mx, rl, rc, rt);
    auto load_col = [&](int j, float& l, float& cf, int& tg) {
      const int col = j * kBT + et;
      load_col_stat<kCol>(p.st, col, col < p.my, l, cf, tg);
    };
    float nl, nc;
    int nt;
    load_col(0, nl, nc, nt);
    int zb = 0;
    uint32_t zphase = 0, fphase = 0;
    const uint32_t p_addr = smem_u32(p_tile);
    for (int j = 0; j < J; ++j) {
      if (kCol) {
        stage_col_stat<false>(s_col, et, nl, nc, nt, p.st.c);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (j + 1 < J) load_col(j + 1, nl, nc, nt);
      }
      mbar_wait(&zfull_bar[zb], zphase);
      tc_fence_after_sync();
      mbar_wait(pfree_bar, fphase ^ 1);  // MMA2(j-1) has finished reading the G tile
      fphase ^= 1;
      const int rrel = rt - j * kBT;
#pragma unroll 1
      for (int ch = 0; ch < kBT / 32; ++ch) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + lane_addr + kTmemZ + zb * kBT + ch * 32, r);
        tmem_ld_wait();
        float g[32];
        g_chunk<kRow, kCol>(r, p.st.c, rl, rc, 0.f, row, rrel, s_col, ch, g);
        uint32_t gp[16];
        pack_g_chunk(g, gp);
        store_g_chunk(p_addr, row_in_blk, ch, gp);
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      mbar_arrive(pfull_bar);
      mbar_arrive(&zempty_bar[zb]);
      if (++zb == 2) {
        zb = 0;
        zphase ^= 1;
      }
      if (kCol) asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    // ------------------------------------------------------------------ final: Out (TMEM) -> global
    mbar_wait(out_bar, 0);
    tc_fence_after_sync();
    const int ocol0 = q * kBD;
#pragma unroll 1
    for (int ch = 0; ch < kBD / 32; ++ch) {
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + lane_addr + kTmemOut + ch * 32, r);
      tmem_ld_wait();
      const int col = ocol0 + ch * 32;
      if (row < p.mx && col < p.k) store_out_chunk<true>(p.out, p.out_bf16, p.ldo, row, col, p.k, r);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

}  // namespace

int sggx_dispatch(int cluster, const void* x, const void* y, int64_t mx, int64_t my, int64_t k,
                  const SoftmaxGradStats& stats, void* out, int out_is_bf16, void* workspace, size_t workspace_bytes,
                  cudaStream_t st);
size_t sggx_workspace_bytes();

// Cluster size for the shared-recompute kernel (sgg_x.cu): the largest of {4, 2} whose 256-column slices tile k exactly,
// unless option sgg_cluster caps it (1 = the single-CTA kernel in this file).
static int choose_cluster(int64_t k) {
  int want = (int)get_option(kOptSggCluster);
  if (want <= 0) want = 4;
  if (want >= 4 && k % 1024 == 0) return 4;
  if (want >= 2 && k % 512 == 0) return 2;
  return 1;
}
}  // namespace pgica

extern "C" int pgica_softmax_grad_gemm_workspace_bytes(int64_t mx, int64_t my, int64_t k, size_t* bytes_host) {
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  (void)mx;
  (void)my;
  (void)k;
  *bytes_host = pgica::sggx_workspace_bytes();
  return PGICA_OK;
}

extern "C" int pgica_softmax_grad_gemm(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale,
                                       const float* r_lse, const float* r_coef, const int32_t* r_tgt,
                                       const float* c_lse, const float* c_coef, const int32_t* c_tgt, void* out,
                                       int out_is_bf16, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace pgica;
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(x && y && out, "softmax_grad_gemm: null operand");
  PGICA_REQUIRE(mx > 0 && my > 0 && k > 0 && k % 8 == 0, "softmax_grad_gemm: bad shape (mx %lld my %lld k %lld)",
                (long long)mx, (long long)my, (long long)k);
  PGICA_REQUIRE(mx < (1ll << 30) && my < (1ll << 30) && k <= (1 << 20), "softmax_grad_gemm: dimension too large");
  const bool row = r_lse != nullptr, col = c_lse != nullptr;
  PGICA_REQUIRE(row || col, "softmax_grad_gemm: need row statistics, column statistics or both");
  PGICA_REQUIRE(!row || r_coef, "softmax_grad_gemm: r_coef missing");
  PGICA_REQUIRE(!col || c_coef, "softmax_grad_gemm: c_coef missing");
  PGICA_REQUIRE(scale > 0.f, "softmax_grad_gemm: scale must be positive");
  const SoftmaxGradStats stats{scale * kLog2e, r_lse, r_coef, r_tgt, c_lse, c_coef, c_tgt};
  const int cluster = choose_cluster(k);
  if (cluster > 1 && workspace != nullptr && workspace_bytes > 0)
    return sggx_dispatch(cluster, x, y, mx, my, k, stats, out, out_is_bf16, workspace, workspace_bytes,
                         static_cast<cudaStream_t>(stream));
  SggParams p{};
  p.mx = (int)mx;
  p.my = (int)my;
  p.k = (int)k;
  p.num_tiles = (int)ceil_div(my, kBT);
  p.passes = (int)ceil_div(k, kBD);
  p.ldo = (int)k;
  p.out_bf16 = out_is_bf16;
  p.st = stats;
  p.out = out;
  CUtensorMap tm_x, tm_y;
  rc = make_tmap_bf16(&tm_x, x, mx, k, k, 128);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y, y, my, k, k, 128);
  if (rc != PGICA_OK) return rc;
  const int64_t grid = ceil_div(mx, kBM) * p.passes;
  PGICA_REQUIRE(grid < (1ll << 31), "softmax_grad_gemm: grid too large");
  rc = with_terms(row, col, [&](auto r, auto c) {
    auto kern = sgg_kernel<decltype(r)::value, decltype(c)::value>;
    PGICA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSggSmem));
    kern<<<(unsigned)grid, kThreads, kSggSmem, static_cast<cudaStream_t>(stream)>>>(tm_x, tm_y, p);
    return PGICA_OK;
  });
  if (rc != PGICA_OK) return rc;
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}
