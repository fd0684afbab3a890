// SURVEY 8(f) rows 3 and 4 — the HBM-bound pieces on either side of the two loss heads.
//
// Row 4, the decoder's cross-attention over ONE key (pkg/models/model.py:528-535, 594-601): nn.MultiheadAttention is
// called with the projected image as its only key / value token, so the softmax over keys is identically 1 and the
// block reduces to
//     y[b, t, :] = LayerNorm( x[b, t, :] + b_o + sum_h w[b, t, h] * U[b, h, :] )        U[b, h, :] = W_o[:, head h] v_h[b]
// with w = 1 in evaluation and w = keep[b, t, h] / (1 - p) under attention dropout (a mask per head and position).
// The query and key projections, the score matrix and the softmax — a (B*T, E) x (E, E) GEMM and a dozen launches in
// the reference — disappear; what is left streams x once and writes y once.
//
// Row 3, the tail of the projection heads feeding the contrastive head (model.py:136-142, 338-344, 826-829):
//     e = LayerNorm(z) (returned: the decoder consumes it),  n = e / max(||e||, eps)  (the NT-Xent operand)
// one launch instead of LayerNorm + norm + clamp + div, and one launch for the backward of both outputs.
#include "common.h"
#include "ptx.cuh"

#include <mutex>

namespace pgica {
namespace {

constexpr int kLnThreads = 256;

__device__ __forceinline__ float block_sum(float v, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_sum(v);
  __syncthreads();  // red may still be read from the previous reduction
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;  // every thread of every warp holds the total
}

// ------------------------------------------------------------------------------------------------ row 4 forward
// One block per (b, t) row; E <= 4 * 4 * 256 (each thread keeps up to 4 float4 of the row in registers).
__global__ void __launch_bounds__(kLnThreads)
xattn_ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ u, const float* __restrict__ w,
                    const float* __restrict__ bo, const float* __restrict__ gamma, const float* __restrict__ beta, int T,
                    int E, int H, float eps, float* __restrict__ y, float* __restrict__ mean, float* __restrict__ rstd) {
  __shared__ float red[32];
  __shared__ float s_w[32];
  const int row = blockIdx.x, b = row / T;
  const int nv = E / 4;
  if (threadIdx.x < H) s_w[threadIdx.x] = w ? w[(size_t)row * H + threadIdx.x] : 1.f;
  __syncthreads();
  float4 pre[4];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = threadIdx.x + i * kLnThreads;
    if (v < nv) {
      float4 a = reinterpret_cast<const float4*>(x + (size_t)row * E)[v];
      if (bo) {
        const float4 c = reinterpret_cast<const float4*>(bo)[v];
        a.x += c.x, a.y += c.y, a.z += c.z, a.w += c.w;
      }
      for (int h = 0; h < H; ++h) {
        const float4 uu = reinterpret_cast<const float4*>(u + ((size_t)b * H + h) * E)[v];
        const float wh = s_w[h];
        a.x = fmaf(wh, uu.x, a.x), a.y = fmaf(wh, uu.y, a.y), a.z = fmaf(wh, uu.z, a.z), a.w = fmaf(wh, uu.w, a.w);
      }
      pre[i] = a;
      sum += a.x + a.y + a.z + a.w;
    }
  }
  const float mu = block_sum(sum, red) / E;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = threadIdx.x + i * kLnThreads;
    if (v < nv) {
      const float4 a = pre[i];
      sq += (a.x - mu) * (a.x - mu) + (a.y - mu) * (a.y - mu) + (a.z - mu) * (a.z - mu) + (a.w - mu) * (a.w - mu);
    }
  }
  const float rs = rsqrtf(block_sum(sq, red) / E + eps);  // biased variance, like nn.LayerNorm
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = threadIdx.x + i * kLnThreads;
    if (v < nv) {
      const float4 a = pre[i], g = reinterpret_cast<const float4*>(gamma)[v], bt = reinterpret_cast<const float4*>(beta)[v];
      float4 o;
      o.x = (a.x - mu) * rs * g.x + bt.x;
      o.y = (a.y - mu) * rs * g.y + bt.y;
      o.z = (a.z - mu) * rs * g.z + bt.z;
      o.w = (a.w - mu) * rs * g.w + bt.w;
      reinterpret_cast<float4*>(y + (size_t)row * E)[v] = o;
    }
  }
  if (threadIdx.x == 0) {
    mean[row] = mu;
    rstd[row] = rs;
  }
}

// ------------------------------------------------------------------------------------------------ row 4 backward
// One block per sequence b (deterministic: the block owns du[b] and its own rows of the per-sequence partials of
// dgamma / dbeta / db_o, which the caller sums over b).  pre is recomputed from x, u, w: nothing row-sized is saved.
__global__ void __launch_bounds__(kLnThreads)
xattn_ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ u,
                    const float* __restrict__ w, const float* __restrict__ bo, const float* __restrict__ gamma,
                    const float* __restrict__ mean, const float* __restrict__ rstd, int T, int E, int H,
                    float* __restrict__ dx, float* __restrict__ du, float* __restrict__ dgamma_part,
                    float* __restrict__ dbeta_part, float* __restrict__ dpre_sum_part) {
  __shared__ float red[32];
  __shared__ float s_w[32];
  const int b = blockIdx.x;
  const int nv = E / 4;
  // this thread's columns: up to 4 float4 -> accumulators for dgamma, dbeta, sum of dpre and du[h] (H <= 8 kept in
  // registers for the first float4 group only would not be general: du is accumulated in global memory instead, each
  // element owned by exactly one thread, so plain read-modify-write is race-free and deterministic)
  float4 acc_g[4], acc_b[4], acc_p[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc_g[i] = acc_b[i] = acc_p[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int h = 0; h < H; ++h)
    for (int v = threadIdx.x; v < nv; v += kLnThreads)
      reinterpret_cast<float4*>(du + ((size_t)b * H + h) * E)[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t = 0; t < T; ++t) {
    const int row = b * T + t;
    __syncthreads();
    if (threadIdx.x < H) s_w[threadIdx.x] = w ? w[(size_t)row * H + threadIdx.x] : 1.f;
    __syncthreads();
    const float mu = mean[row], rs = rstd[row];
    float4 xh[4], gg[4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int v = threadIdx.x + i * kLnThreads;
      if (v < nv) {
        float4 a = reinterpret_cast<const float4*>(x + (size_t)row * E)[v];
        if (bo) {
          const float4 c = reinterpret_cast<const float4*>(bo)[v];
          a.x += c.x, a.y += c.y, a.z += c.z, a.w += c.w;
        }
        for (int h = 0; h < H; ++h) {
          const float4 uu = reinterpret_cast<const float4*>(u + ((size_t)b * H + h) * E)[v];
          const float wh = s_w[h];
          a.x = fmaf(wh, uu.x, a.x), a.y = fmaf(wh, uu.y, a.y), a.z = fmaf(wh, uu.z, a.z), a.w = fmaf(wh, uu.w, a.w);
        }
        const float4 d = reinterpret_cast<const float4*>(dy + (size_t)row * E)[v];
        const float4 g = reinterpret_cast<const float4*>(gamma)[v];
        float4 h4, q;
        h4.x = (a.x - mu) * rs, h4.y = (a.y - mu) * rs, h4.z = (a.z - mu) * rs, h4.w = (a.w - mu) * rs;
        q.x = d.x * g.x, q.y = d.y * g.y, q.z = d.z * g.z, q.w = d.w * g.w;
        xh[i] = h4;
        gg[i] = q;
        acc_g[i].x += d.x * h4.x, acc_g[i].y += d.y * h4.y, acc_g[i].z += d.z * h4.z, acc_g[i].w += d.w * h4.w;
        acc_b[i].x += d.x, acc_b[i].y += d.y, acc_b[i].z += d.z, acc_b[i].w += d.w;
        s1 += q.x + q.y + q.z + q.w;
        s2 += q.x * h4.x + q.y * h4.y + q.z * h4.z + q.w * h4.w;
      }
    }
    const float m1 = block_sum(s1, red) / E;
    const float m2 = block_sum(s2, red) / E;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int v = threadIdx.x + i * kLnThreads;
      if (v < nv) {
        float4 dp;
        dp.x = rs * (gg[i].x - m1 - xh[i].x * m2);
        dp.y = rs * (gg[i].y - m1 - xh[i].y * m2);
        dp.z = rs * (gg[i].z - m1 - xh[i].z * m2);
        dp.w = rs * (gg[i].w - m1 - xh[i].w * m2);
        reinterpret_cast<float4*>(dx + (size_t)row * E)[v] = dp;
        acc_p[i].x += dp.x, acc_p[i].y += dp.y, acc_p[i].z += dp.z, acc_p[i].w += dp.w;
        for (int h = 0; h < H; ++h) {
          const float wh = s_w[h];
          if (wh != 0.f) {
            float4* dst = reinterpret_cast<float4*>(du + ((size_t)b * H + h) * E) + v;
            float4 c = *dst;
            c.x = fmaf(wh, dp.x, c.x), c.y = fmaf(wh, dp.y, c.y), c.z = fmaf(wh, dp.z, c.z), c.w = fmaf(wh, dp.w, c.w);
            *dst = c;
          }
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = threadIdx.x + i * kLnThreads;
    if (v < nv) {
      reinterpret_cast<float4*>(dgamma_part + (size_t)b * E)[v] = acc_g[i];
      reinterpret_cast<float4*>(dbeta_part + (size_t)b * E)[v] = acc_b[i];
      reinterpret_cast<float4*>(dpre_sum_part + (size_t)b * E)[v] = acc_p[i];
    }
  }
}

// ------------------------------------------------------------------------------------------------ row 3
// One warp per row (D <= 1024, D % 4 == 0): e = LayerNorm(z) * gamma + beta, n = e / max(||e||, eps_norm).
__global__ void ln_l2norm_fwd_kernel(const float* __restrict__ z, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, int rows, int D, float eps_ln, float eps_norm,
                                     float* __restrict__ e, float* __restrict__ n, float* __restrict__ stats) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* zr = z + (size_t)r * D;
  float s = 0.f;
  for (int k = lane; k < D; k += 32) s += zr[k];
  const float mu = warp_sum(s) / D;
  float q = 0.f;
  for (int k = lane; k < D; k += 32) q += (zr[k] - mu) * (zr[k] - mu);
  const float rs = rsqrtf(warp_sum(q) / D + eps_ln);
  float ss = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float v = (zr[k] - mu) * rs * gamma[k] + beta[k];
    e[(size_t)r * D + k] = v;
    ss = fmaf(v, v, ss);
  }
  const float inv = 1.f / fmaxf(sqrtf(warp_sum(ss)), eps_norm);
  for (int k = lane; k < D; k += 32) n[(size_t)r * D + k] = e[(size_t)r * D + k] * inv;
  if (lane == 0) {
    stats[3 * r] = mu;
    stats[3 * r + 1] = rs;
    stats[3 * r + 2] = inv;
  }
}

// Backward of both outputs: de_total = de + (dn - nh <nh, dn>) * inv  (nh = e * inv), then the LayerNorm backward.
// A row with ||e|| < eps_norm gets de + dn * inv and no projection: F.normalize's clamp_min passes no gradient to the
// norm there.  The sum of squares is recomputed in the forward's order (same lanes, same fmaf chain, same butterfly),
// so 1 / sqrtf(ss) exceeds the stored inv exactly when the forward clamped.
// dgamma / dbeta partials per block of 8 rows (summed by the caller: deterministic).
__global__ void ln_l2norm_bwd_kernel(const float* __restrict__ z, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const float* __restrict__ stats,
                                     const float* __restrict__ de, const float* __restrict__ dn, int rows, int D,
                                     float* __restrict__ dz, float* __restrict__ dgamma_part,
                                     float* __restrict__ dbeta_part) {
  extern __shared__ float s_part[];  // [2][8][D]
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + wib;
  float* pg = s_part + (size_t)wib * D;
  float* pb = s_part + (size_t)(8 + wib) * D;
  for (int k = lane; k < D; k += 32) pg[k] = pb[k] = 0.f;
  if (r < rows) {
    const float mu = stats[3 * r], rs = stats[3 * r + 1], inv = stats[3 * r + 2];
    const float* zr = z + (size_t)r * D;
    float dot = 0.f, ss = 0.f;
    if (dn)
      for (int k = lane; k < D; k += 32) {
        const float ev = (zr[k] - mu) * rs * gamma[k] + beta[k];
        ss = fmaf(ev, ev, ss);
        dot = fmaf(ev * inv, dn[(size_t)r * D + k], dot);
      }
    dot = warp_sum(dot);
    ss = warp_sum(ss);
    if (1.f / sqrtf(ss) > inv) dot = 0.f;
    float s1 = 0.f, s2 = 0.f;
    for (int k = lane; k < D; k += 32) {
      const float xh = (zr[k] - mu) * rs;
      const float ev = xh * gamma[k] + beta[k];
      float g = de ? de[(size_t)r * D + k] : 0.f;
      if (dn) g += (dn[(size_t)r * D + k] - ev * inv * dot) * inv;
      pg[k] = g * xh;
      pb[k] = g;
      const float gq = g * gamma[k];
      s1 += gq;
      s2 = fmaf(gq, xh, s2);
    }
    s1 = warp_sum(s1) / D;
    s2 = warp_sum(s2) / D;
    for (int k = lane; k < D; k += 32) {
      const float xh = (zr[k] - mu) * rs;
      dz[(size_t)r * D + k] = rs * (pb[k] * gamma[k] - s1 - xh * s2);
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < D; k += blockDim.x) {
    float a = 0.f, c = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      a += s_part[(size_t)i * D + k];
      c += s_part[(size_t)(8 + i) * D + k];
    }
    dgamma_part[(size_t)blockIdx.x * D + k] = a;
    dbeta_part[(size_t)blockIdx.x * D + k] = c;
  }
}

}  // namespace
}  // namespace pgica

extern "C" {

using namespace pgica;

int pgica_xattn_ln_fwd(const float* x, const float* u, const float* w, const float* out_bias, const float* gamma,
                       const float* beta, int64_t batch, int64_t seqlen, int64_t dim, int64_t heads, float eps, float* y,
                       float* mean, float* rstd, void* stream) {
  PGICA_REQUIRE(x && u && gamma && beta && y && mean && rstd, "xattn_ln_fwd: null pointer");
  PGICA_REQUIRE(batch > 0 && seqlen > 0 && dim > 0 && dim % 4 == 0 && dim <= 4096 && heads >= 1 && heads <= 32 &&
                    batch * seqlen < (1ll << 31),
                "xattn_ln_fwd: bad shape (batch %lld seq %lld dim %lld heads %lld; dim %% 4 == 0, dim <= 4096, heads <= 32)",
                (long long)batch, (long long)seqlen, (long long)dim, (long long)heads);
  xattn_ln_fwd_kernel<<<(unsigned)(batch * seqlen), kLnThreads, 0, (cudaStream_t)stream>>>(
      x, u, w, out_bias, gamma, beta, (int)seqlen, (int)dim, (int)heads, eps, y, mean, rstd);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_xattn_ln_bwd(const float* dy, const float* x, const float* u, const float* w, const float* out_bias,
                       const float* gamma, const float* mean, const float* rstd, int64_t batch, int64_t seqlen,
                       int64_t dim, int64_t heads, float* dx, float* du, float* dgamma_part, float* dbeta_part,
                       float* dpre_sum_part, void* stream) {
  PGICA_REQUIRE(dy && x && u && gamma && mean && rstd && dx && du && dgamma_part && dbeta_part && dpre_sum_part,
                "xattn_ln_bwd: null pointer");
  PGICA_REQUIRE(batch > 0 && seqlen > 0 && dim > 0 && dim % 4 == 0 && dim <= 4096 && heads >= 1 && heads <= 32,
                "xattn_ln_bwd: bad shape");
  xattn_ln_bwd_kernel<<<(unsigned)batch, kLnThreads, 0, (cudaStream_t)stream>>>(
      dy, x, u, w, out_bias, gamma, mean, rstd, (int)seqlen, (int)dim, (int)heads, dx, du, dgamma_part, dbeta_part,
      dpre_sum_part);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_ln_l2norm_fwd(const float* z, const float* gamma, const float* beta, int64_t rows, int64_t dim, float eps_ln,
                        float eps_norm, float* e, float* n, float* stats, void* stream) {
  PGICA_REQUIRE(z && gamma && beta && e && n && stats, "ln_l2norm_fwd: null pointer");
  PGICA_REQUIRE(rows > 0 && dim > 0 && dim <= 8192 && rows < (1ll << 31), "ln_l2norm_fwd: bad shape");
  ln_l2norm_fwd_kernel<<<(unsigned)ceil_div(rows, 8), 256, 0, (cudaStream_t)stream>>>(z, gamma, beta, (int)rows, (int)dim,
                                                                                     eps_ln, eps_norm, e, n, stats);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_ln_l2norm_bwd(const float* z, const float* gamma, const float* beta, const float* stats, const float* de,
                        const float* dn, int64_t rows, int64_t dim, float* dz, float* dgamma_part, float* dbeta_part,
                        void* stream) {
  PGICA_REQUIRE(z && gamma && beta && stats && dz && dgamma_part && dbeta_part && (de || dn), "ln_l2norm_bwd: null pointer");
  PGICA_REQUIRE(rows > 0 && dim > 0 && dim <= 2048, "ln_l2norm_bwd: bad shape (dim <= 2048)");
  const size_t smem = (size_t)16 * dim * sizeof(float);
  static std::once_flag once[64];
  int dev = 0;
  PGICA_CUDA_OK(cudaGetDevice(&dev));
  cudaError_t err = cudaSuccess;
  std::call_once(once[dev & 63], [&] {
    err = cudaFuncSetAttribute(ln_l2norm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 2048 * 4);
  });
  PGICA_CUDA_OK(err);
  ln_l2norm_bwd_kernel<<<(unsigned)ceil_div(rows, 8), 256, smem, (cudaStream_t)stream>>>(
      z, gamma, beta, stats, de, dn, (int)rows, (int)dim, dz, dgamma_part, dbeta_part);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

}  // extern "C"
