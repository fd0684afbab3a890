// Stage-1 head at the batch sizes the reference actually trains with (configs/default.yaml: B = 8; BASELINE config 1:
// B = 64): the WHOLE symmetric NT-Xent — similarity, both log-sum-exps, loss and both gradients — in ONE launch of ONE
// CTA.  At these sizes the head is pure launch latency (12.6 MFLOP at B = 64); the general path needs ~10 launches
// (two GEMM+LSE kernels with their merges, loss, coefficient kernels, the backward) = 85-105 us per step, this kernel
// a handful of microseconds.  B <= 128 rows per side, D <= 512, D % 64 == 0, bf16 operands used as given
// (pkg/models/model.py:970-1000 semantics; the caller normalises).
//
//   phase 1  Z[128 x 128] = A B^T on tcgen05 (operands streamed through a 4-stage TMA ring, accumulator in TMEM)
//   phase 2  thread i takes row i of Z out of TMEM, scales it into the log2 domain and parks it in shared memory;
//            then row i's and (reading down the tile) column i's running max / sum -> lse_row, lse_col, loss
//   phase 3  G = w (softmax_row + softmax_col - 2 I) as a bf16 tile in shared memory (128-byte swizzle)
//   phase 4  dA = G B and dB = G^T A, 128 output columns per pass: G (or the same tile read MN-major for G^T) times
//            the operand rows re-streamed MN-major; results leave through shared memory as coalesced row stores.
// The gradients are those of the loss itself (upstream gradient 1); autograd scales them by the upstream scalar.
#include "common.h"
#include "sgg_tile.cuh"

#include <mutex>

namespace pgica {
namespace {

constexpr int kT = 128;                          // tile edge: rows of A, rows of B
constexpr int kBK = 64;
constexpr uint32_t kChunk = kT * kBK * 2;        // 16 KB: a [128][64] bf16 box
constexpr int kRing = 4;                         // phase-1 stages of (A chunk + B chunk)
constexpr int kPitch = kT + 1;                   // fp32 tile in shared memory, padded against bank conflicts
constexpr int kThreads = 128;
constexpr float kLn2 = 0.6931471805599453f;
// shared memory: [0, 128K) ring in phase 1, then {operand buffers 2 x 32K | G tile 32K | unused}; fp32 tile; vectors
constexpr uint32_t kOffOp = 0, kOffG = 2 * 2 * kChunk, kOffZ = kRing * 2 * kChunk;
constexpr uint32_t kZBytes = kT * kPitch * 4;
constexpr size_t kSmem = 1024 + kOffZ + kZBytes + 4 * kT * 4 + 256;
constexpr uint32_t kTmemZ = 0, kTmemOut = 128;   // TMEM columns: Z [0,128), two output buffers [128,256) [256,384)

struct NtxSmallParams {
  int n, k;          // rows per side, width of the operands / gradients
  int kf;            // depth of the similarity product (k, or 3k for split fp32 operands [hi|lo|hi] x [hi|hi|lo])
  float c;           // inv_tau * log2(e)
  float w;           // gradient weight: inv_tau / (2n) (mean) or inv_tau / 2 (sum)
  float loss_mult;   // 0.5 / n (mean) or 0.5 (sum)
  float* loss;
  float* lse_row;    // natural log
  float* lse_col;
  float* da;         // [n][k] fp32
  float* db;
};

__global__ void __launch_bounds__(kThreads, 1)
ntxent_small_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                    const NtxSmallParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  float* zs = reinterpret_cast<float*>(smem + kOffZ);
  float* s_lr = reinterpret_cast<float*>(smem + kOffZ + kZBytes);
  float* s_lc = s_lr + kT;
  float* s_red = s_lc + kT;  // [kT] scratch for the loss reduction
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_red + 2 * kT);
  uint64_t* empty_bar = full_bar + kRing;
  uint64_t* zfull_bar = empty_bar + kRing;
  uint64_t* opfull_bar = zfull_bar + 1;   // [2]
  uint64_t* outfull_bar = opfull_bar + 2; // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(outfull_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = threadIdx.x;  // this thread's row (and, in the column pass, its column)
  const int nkb = p.kf / kBK;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < kRing; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(zfull_bar, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&opfull_bar[s], 1);
      mbar_init(&outfull_bar[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint64_t desc_k = make_smem_desc(0, 16, 1024);

  // ------------------------------------------------------------------------------------------- phase 1: Z = A B^T
  if (warp == 0) {
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % kRing;
      if (kb >= kRing) mbar_wait(&empty_bar[s], ((kb / kRing) - 1) & 1);
      if (elect_one()) {
        mbar_expect_tx(&full_bar[s], 2 * kChunk);
        tma_load_2d(smem + s * 2 * kChunk, &tm_a, &full_bar[s], kb * kBK, 0);
        tma_load_2d(smem + s * 2 * kChunk + kChunk, &tm_b, &full_bar[s], kb * kBK, 0);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(kT, kT, 0, 0);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % kRing;
      mbar_wait(&full_bar[s], (kb / kRing) & 1);
      tc_fence_after_sync();
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(smem + s * 2 * kChunk);
        const uint64_t da = desc_k | ((a_addr >> 4) & 0x3FFF);
        const uint64_t db = desc_k | (((a_addr + kChunk) >> 4) & 0x3FFF);
#pragma unroll
        for (int ks = 0; ks < kBK / 16; ++ks) umma_bf16_ss(tmem_base + kTmemZ, da + 2 * ks, db + 2 * ks, idesc, (kb | ks) != 0 ? 1u : 0u);
        umma_commit(&empty_bar[s]);
        if (kb == nkb - 1) umma_commit(zfull_bar);
      }
      __syncwarp();
    }
  }
  mbar_wait(zfull_bar, 0);
  tc_fence_after_sync();

  // ------------------------------------------------------------------------------------------- phase 2: statistics
  // row i of t = z * inv_tau * log2(e) into shared memory
#pragma unroll 1
  for (int ch = 0; ch < kT / 32; ++ch) {
    uint32_t r[32];
    tmem_ld_32x32(tmem_base + lane_addr + kTmemZ + ch * 32, r);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) zs[i * kPitch + ch * 32 + j] = __uint_as_float(r[j]) * p.c;
  }
  __syncthreads();
  float lr = 0.f, lc = 0.f, tii = 0.f;
  if (i < p.n) {
    float m = -INFINITY;
    for (int j = 0; j < p.n; ++j) m = fmaxf(m, zs[i * kPitch + j]);
    float s = 0.f;
    for (int j = 0; j < p.n; ++j) s += fast_exp2(zs[i * kPitch + j] - m);
    lr = m + log2f(s);
    m = -INFINITY;
    for (int j = 0; j < p.n; ++j) m = fmaxf(m, zs[j * kPitch + i]);
    s = 0.f;
    for (int j = 0; j < p.n; ++j) s += fast_exp2(zs[j * kPitch + i] - m);
    lc = m + log2f(s);
    tii = zs[i * kPitch + i];
    p.lse_row[i] = lr * kLn2;
    p.lse_col[i] = lc * kLn2;
  }
  s_lr[i] = lr;
  s_lc[i] = lc;
  s_red[i] = i < p.n ? (lr - tii) + (lc - tii) : 0.f;
  __syncthreads();
  if (warp == 0) {
    float v = s_red[lane] + s_red[lane + 32] + s_red[lane + 64] + s_red[lane + 96];
    v = warp_sum(v);
    if (lane == 0) *p.loss = v * kLn2 * p.loss_mult;
  }

  // ------------------------------------------------------------------------------------------- phase 3: G tile (bf16)
  {
    const uint32_t g_local = smem_u32(smem + kOffG);
#pragma unroll 1
    for (int ch = 0; ch < kT / 32; ++ch) {
      uint32_t gp[16];
#pragma unroll
      for (int jj = 0; jj < 32; jj += 2) {
        float g2[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = ch * 32 + jj + u;
          float g = 0.f;
          if (i < p.n && j < p.n) {
            const float t = zs[i * kPitch + j];
            g = p.w * (fast_exp2(t - lr) + fast_exp2(t - s_lc[j]));
            if (j == i) g -= 2.f * p.w;
          }
          g2[u] = g;
        }
        gp[jj >> 1] = pack_bf16x2(g2[0], g2[1]);
      }
      store_g_chunk(g_local, i, ch, gp);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before_sync();
  __syncthreads();  // G complete; the fp32 tile and the phase-1 ring may be reused from here on
  tc_fence_after_sync();

  // ------------------------------------------------------------------------------------------- phase 4: dA = G B, dB = G^T A
  const int halves = p.k / 128;       // passes per output matrix
  const int passes = 2 * halves;
  auto issue_operand = [&](int ps) {  // operand rows (all 128) x 128 columns, as two [128][64] boxes read MN-major
    const bool second = ps >= halves;
    const CUtensorMap* tm = second ? &tm_a : &tm_b;
    const int col0 = (second ? ps - halves : ps) * 128;
    uint8_t* dst = smem + kOffOp + (ps & 1) * 2 * kChunk;
    mbar_expect_tx(&opfull_bar[ps & 1], 2 * kChunk);
    tma_load_2d(dst, tm, &opfull_bar[ps & 1], col0, 0);
    tma_load_2d(dst + kChunk, tm, &opfull_bar[ps & 1], col0 + kBK, 0);
  };
  auto issue_mma = [&](int ps) {
    const bool second = ps >= halves;
    const uint32_t idesc2 = make_idesc_bf16(kT, 128, second ? 1 : 0, 1);
    const uint32_t g_addr = smem_u32(smem + kOffG);
    const uint32_t o_addr = smem_u32(smem + kOffOp + (ps & 1) * 2 * kChunk);
    const uint64_t dg = (second ? make_smem_desc(0, kChunk, 1024) : desc_k) | ((g_addr >> 4) & 0x3FFF);
    const uint64_t dob = make_smem_desc(0, kChunk, 1024) | ((o_addr >> 4) & 0x3FFF);
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t da = second ? dg + ks * (2048 >> 4) : dg + (ks >> 2) * (kChunk >> 4) + (ks & 3) * 2;
      umma_bf16_ss(tmem_base + kTmemOut + (ps & 1) * 128, da, dob + ks * (2048 >> 4), idesc2, ks != 0 ? 1u : 0u);
    }
    umma_commit(&outfull_bar[ps & 1]);
  };
  if (threadIdx.x == 0) {
    issue_operand(0);
    if (passes > 1) issue_operand(1);
  }
  if (warp == 1) {
    mbar_wait(&opfull_bar[0], 0);
    tc_fence_after_sync();
    if (elect_one()) issue_mma(0);
    __syncwarp();
  }
#pragma unroll 1
  for (int ps = 0; ps < passes; ++ps) {
    if (warp == 1 && ps + 1 < passes) {  // the next pass's product runs while this pass's result is written out
      mbar_wait(&opfull_bar[(ps + 1) & 1], ((ps + 1) >> 1) & 1);
      tc_fence_after_sync();
      if (elect_one()) issue_mma(ps + 1);
      __syncwarp();
    }
    mbar_wait(&outfull_bar[ps & 1], (ps >> 1) & 1);
    tc_fence_after_sync();
    // rows of this warp: TMEM -> padded fp32 tile -> coalesced 512-byte row stores
#pragma unroll 1
    for (int ch = 0; ch < 4; ++ch) {
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + lane_addr + kTmemOut + (ps & 1) * 128 + ch * 32, r);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) zs[i * kPitch + ch * 32 + j] = __uint_as_float(r[j]);
    }
    __syncwarp();
    {
      const bool second = ps >= halves;
      float* out = second ? p.db : p.da;
      const int col0 = (second ? ps - halves : ps) * 128;
      for (int rr = 0; rr < 32; ++rr) {
        const int row = warp * 32 + rr;
        if (row >= p.n) break;
        const float* src = zs + row * kPitch + lane * 4;
        float4 v = make_float4(src[0], src[1], src[2], src[3]);
        *reinterpret_cast<float4*>(out + (size_t)row * p.k + col0 + lane * 4) = v;
      }
    }
    tc_fence_before_sync();
    __syncthreads();  // output buffer, staging tile and operand buffer of this pass are free again
    tc_fence_after_sync();
    if (threadIdx.x == 0 && ps + 2 < passes) issue_operand(ps + 2);
  }
  if (warp == 0) tmem_dealloc<512>(tmem_base);
}

}  // namespace
}  // namespace pgica

extern "C" int pgica_ntxent_small_supported(int64_t rows, int64_t dim) {
  return (rows >= 1 && rows <= 128 && dim >= 128 && dim <= 512 && dim % 128 == 0) ? 1 : 0;
}

static int ntxent_small_launch(const void* a, const void* b, int64_t rows, int64_t dim, int64_t depth, float inv_tau,
                               int reduce_mean, float* loss, float* lse_row, float* lse_col, float* da, float* db,
                               void* stream) {
  using namespace pgica;
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(a && b && loss && lse_row && lse_col && da && db, "ntxent_small: null pointer");
  PGICA_REQUIRE(pgica_ntxent_small_supported(rows, dim), "ntxent_small: needs 1 <= rows <= 128 and dim in {128, 256, 384, 512} (got %lld x %lld)",
                (long long)rows, (long long)dim);
  PGICA_REQUIRE(inv_tau > 0.f, "ntxent_small: temperature must be positive");
  PGICA_REQUIRE((reinterpret_cast<uintptr_t>(da) & 15u) == 0 && (reinterpret_cast<uintptr_t>(db) & 15u) == 0,
                "ntxent_small: gradient buffers must be 16-byte aligned");
  NtxSmallParams p{};
  p.n = (int)rows;
  p.k = (int)dim;
  p.kf = (int)depth;
  p.c = inv_tau * kLog2e;
  p.w = reduce_mean ? inv_tau / (2.0f * rows) : inv_tau * 0.5f;
  p.loss_mult = reduce_mean ? 0.5f / rows : 0.5f;
  p.loss = loss;
  p.lse_row = lse_row;
  p.lse_col = lse_col;
  p.da = da;
  p.db = db;
  CUtensorMap tm_a, tm_b;
  rc = make_tmap_bf16(&tm_a, a, rows, depth, depth, kT);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_b, b, rows, depth, depth, kT);
  if (rc != PGICA_OK) return rc;
  static std::once_flag once[64];
  int dev = 0;
  PGICA_CUDA_OK(cudaGetDevice(&dev));
  cudaError_t attr_err = cudaSuccess;
  std::call_once(once[dev & 63], [&] {
    attr_err = cudaFuncSetAttribute(ntxent_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem);
  });
  PGICA_CUDA_OK(attr_err);
  ntxent_small_kernel<<<1, kThreads, kSmem, static_cast<cudaStream_t>(stream)>>>(tm_a, tm_b, p);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

extern "C" int pgica_ntxent_small(const void* a, const void* b, int64_t rows, int64_t dim, float inv_tau,
                                  int reduce_mean, float* loss, float* lse_row, float* lse_col, float* da, float* db,
                                  void* stream) {
  return ntxent_small_launch(a, b, rows, dim, dim, inv_tau, reduce_mean, loss, lse_row, lse_col, da, db, stream);
}

extern "C" int pgica_ntxent_small_split(const void* a_left3, const void* b_right3, int64_t rows, int64_t dim,
                                        float inv_tau, int reduce_mean, float* loss, float* lse_row, float* lse_col,
                                        float* da, float* db, void* stream) {
  return ntxent_small_launch(a_left3, b_right3, rows, dim, 3 * dim, inv_tau, reduce_mean, loss, lse_row, lse_col, da, db,
                             stream);
}
