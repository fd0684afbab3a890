// The HBM-/latency-bound pieces around the two tensor-core kernels: label/mask plumbing, per-sequence
// reductions (warp shuffles), the DPO scalar head, NT-Xent loss assembly, L2 row normalisation and its
// backward, dtype casts, and the streaming log-softmax path for callers that hand in materialised logits.
#include "common.h"
#include "ptx.cuh"

namespace pgica {
namespace {

constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float load_mask(const void* mask, int kind, size_t i) {
  switch (kind) {
    case PGICA_MASK_I64: return static_cast<float>(static_cast<const long long*>(mask)[i]);
    case PGICA_MASK_F32: return static_cast<const float*>(mask)[i];
    case PGICA_MASK_U8: return static_cast<float>(static_cast<const unsigned char*>(mask)[i]);
    case PGICA_MASK_I32: return static_cast<float>(static_cast<const int*>(mask)[i]);
    default: return 1.f;
  }
}

// row r = b*T + t scores position t of sequence b against labels[b][t+1] with weight mask[b][t+1];
// the last position of every sequence has nothing to predict: weight 0, label -1.
__global__ void prep_rows_kernel(const long long* __restrict__ labels, const void* __restrict__ mask, int mask_kind,
                                 int nseq, int T, int vocab, int* __restrict__ row_label,
                                 float* __restrict__ row_weight) {
  const size_t r = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (r >= (size_t)nseq * T) return;
  const int t = (int)(r % T);
  int lab = -1;
  float w = 0.f;
  if (t + 1 < T) {
    const long long y = labels[r + 1];
    w = load_mask(mask, mask_kind, r + 1);
    lab = (y >= 0 && y < vocab) ? (int)y : -1;
    if (lab < 0 && w != 0.f) w = NAN;  // an unmasked label outside the vocabulary poisons the sequence
  }
  row_label[r] = lab;
  row_weight[r] = w;
}

// One warp per sequence: seq_logp[b] = sum_t w * (z_tgt - lse) (optionally / sum_t w); warp-shuffle reduction.
// nll_sum (optional) accumulates sum over ALL scored positions of (lse - z_tgt): the HF causal-LM loss numerator.
__global__ void seq_reduce_kernel(const float* __restrict__ lse, const float* __restrict__ ztgt,
                                  const float* __restrict__ row_weight, int nseq, int T, int length_normalize,
                                  float* __restrict__ seq_logp, float* __restrict__ nll_sum) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= nseq) return;
  float s = 0.f, wsum = 0.f, nll = 0.f;
  for (int t = lane; t + 1 < T; t += 32) {
    const size_t r = (size_t)b * T + t;
    const float lp = ztgt[r] - lse[r];
    const float w = row_weight[r];
    s = fmaf(w, lp, s);  // multiply like the reference: NaN log-probs at masked positions still poison
    wsum += w;
    nll -= lp;
  }
  s = warp_sum(s);
  wsum = warp_sum(wsum);
  nll = warp_sum(nll);
  if (lane == 0) {
    seq_logp[b] = length_normalize ? s / wsum : s;
    if (nll_sum) atomicAdd(nll_sum, nll);
  }
}

// coef[r] = grad_seq[b] * w[r] (/ len_b) * sign  — the per-row factor of dZ = coef * (onehot - softmax)
__global__ void row_coef_kernel(const float* __restrict__ grad_seq, const float* __restrict__ row_weight, int nseq,
                                int T, int length_normalize, float sign, float* __restrict__ coef) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= nseq) return;
  float wsum = 0.f;
  if (length_normalize) {
    for (int t = lane; t < T; t += 32) wsum += row_weight[(size_t)b * T + t];
    wsum = warp_sum(wsum);
  }
  const float g = grad_seq[b] * sign * (length_normalize ? 1.f / wsum : 1.f);
  for (int t = lane; t < T; t += 32) {
    const size_t r = (size_t)b * T + t;
    const float w = row_weight[r];
    coef[r] = (w == 0.f) ? 0.f : g * w;
  }
}

// DPO scalar head on n pairs (one block): loss, 5 metrics, and dloss/dpc (= -dloss/dpr = -dloss/drc = dloss/drr).
__global__ void dpo_loss_kernel(const float* __restrict__ pc, const float* __restrict__ pr,
                                const float* __restrict__ rc, const float* __restrict__ rr, int n, float beta,
                                float label_smoothing, float inv_n_global, float* __restrict__ loss,
                                float* __restrict__ metrics, float* __restrict__ dpc) {
  __shared__ float red[5][32];
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float pol = pc[i] - pr[i];
    const float ref = rc ? rc[i] - rr[i] : 0.f;
    const float x = beta * (pol - ref);
    // -logsigmoid(x) = softplus(-x), stable
    const float sp_neg = fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));  // softplus(-x)
    const float sp_pos = sp_neg + x;                                // softplus(x)
    const float sig_neg = 1.f / (1.f + expf(x));                    // sigmoid(-x)
    float l, dx;
    if (label_smoothing > 0.f) {
      const float t = 1.f - label_smoothing;
      l = t * sp_neg + (1.f - t) * sp_pos;
      dx = -(t * sig_neg - (1.f - t) * (1.f - sig_neg));
    } else {
      l = sp_neg;
      dx = -sig_neg;
    }
    dpc[i] = beta * dx * inv_n_global;
    acc[0] += l;
    acc[1] += pol - ref;
    acc[2] += (pol > ref) ? 1.f : 0.f;
    acc[3] += pc[i];
    acc[4] += pr[i];
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const float v = warp_sum(acc[k]);
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      float v = lane < nw ? red[k][lane] : 0.f;
      v = warp_sum(v);
      if (lane == 0) {
        const float m = v * inv_n_global;
        if (k == 0) *loss = m;
        metrics[k] = m;
      }
    }
  }
}

// out[i] = a[i] * s[0]   (chain rule through a scalar loss without a host round trip)
__global__ void scale_by_scalar_kernel(const float* __restrict__ a, const float* __restrict__ s, float mult, int n,
                                       float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] * s[0] * mult;
}

// NT-Xent loss from the two log-sum-exp vectors and the diagonal:
//   loss = 0.5 * ( sum_i (lse_row[i] - diag[i]) + sum_j (lse_col[j] - diag_col[j]) ) * inv_denom
// For the local (rows_a x rows_b) slice the column sum is taken over the columns this rank owns
// (col_begin .. col_begin + rows_a), whose diagonal entries are exactly diag[].
__global__ void ntxent_loss_kernel(const float* __restrict__ lse_row, const float* __restrict__ diag,
                                   const float* __restrict__ lse_col_owned, int n, float inv_denom,
                                   float* __restrict__ loss) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += (lse_row[i] - diag[i]) + (lse_col_owned[i] - diag[i]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  acc = warp_sum(acc);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    float v = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) *loss = 0.5f * v * inv_denom;
  }
}

// lse[j] = log sum_r exp(parts[r][j])   (merging per-rank column partials)
__global__ void lse_combine_kernel(const float* __restrict__ parts, int nparts, int n, float* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  float m = -INFINITY;
  for (int r = 0; r < nparts; ++r) m = fmaxf(m, parts[(size_t)r * n + j]);
  float s = 0.f;
  for (int r = 0; r < nparts; ++r) s += exp2f((parts[(size_t)r * n + j] - m) * kLog2e);
  out[j] = m + log2f(s) * kLn2;
}

// fill the statistics arrays the backward kernel wants for NT-Xent: coef = grad * mult, target = i + offset
__global__ void ntxent_coef_kernel(const float* __restrict__ grad, float mult, int n, int tgt_offset, int tgt_limit,
                                   float* __restrict__ coef, int* __restrict__ tgt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  coef[i] = grad[0] * mult;
  const int t = i + tgt_offset;
  tgt[i] = (t >= 0 && t < tgt_limit) ? t : -1;
}

// ------------------------------------------------------------------------------------------ row L2 norm
// One warp per row: y = bf16(x / max(||x||, eps)), inv_norm = 1 / max(||x||, eps).  x is fp32 or bf16.
template <typename T>
__device__ __forceinline__ float ldf(const T* p, size_t i);
template <>
__device__ __forceinline__ float ldf<float>(const float* p, size_t i) { return p[i]; }
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p, size_t i) { return __bfloat162float(p[i]); }

template <typename T>
__global__ void rownorm_fwd_kernel(const T* __restrict__ x, int rows, int dim, float eps,
                                   __nv_bfloat16* __restrict__ y, float* __restrict__ inv_norm,
                                   __nv_bfloat16* __restrict__ left3, __nv_bfloat16* __restrict__ right3,
                                   int normalize) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  float inv = 1.f;
  if (normalize) {
    float ss = 0.f;
    for (int k = lane; k < dim; k += 32) {
      const float v = ldf(x, (size_t)r * dim + k);
      ss = fmaf(v, v, ss);
    }
    ss = warp_sum(ss);
    inv = 1.f / fmaxf(sqrtf(ss), eps);
  }
  for (int k = lane; k < dim; k += 32) {
    const float v = normalize ? ldf(x, (size_t)r * dim + k) * inv : ldf(x, (size_t)r * dim + k);
    const __nv_bfloat16 hi = __float2bfloat16(v);
    if (y) y[(size_t)r * dim + k] = hi;
    if (left3) {
      // two-term bf16 split of the unit vector: <a, b> ~= a_hi.b_hi + a_lo.b_hi + a_hi.b_lo as ONE bf16 GEMM over 3*dim
      const __nv_bfloat16 lo = __float2bfloat16(v - __bfloat162float(hi));
      const size_t o = (size_t)r * 3 * dim + k;
      left3[o] = hi;
      left3[o + dim] = lo;
      left3[o + 2 * dim] = hi;
      right3[o] = hi;
      right3[o + dim] = hi;
      right3[o + 2 * dim] = lo;
    }
  }
  if (lane == 0 && inv_norm) inv_norm[r] = inv;
}

// dx = (g - xh * <xh, g>) * inv_norm with xh = x * inv_norm recomputed in fp32.  g is fp32 or bf16, rows `g_pitch`
// elements apart; with g_second >= 0 the upstream gradient is g[:, 0:dim] + g[:, g_second:g_second+dim] (the two
// column blocks a softmax-gradient GEMM over split operands [hi|hi|lo] produces).
template <typename TX, typename TG>
__global__ void rownorm_bwd_kernel(const TX* __restrict__ x, const float* __restrict__ inv_norm,
                                   const TG* __restrict__ g, int rows, int dim, int64_t g_pitch, int64_t g_second,
                                   float* __restrict__ dx) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float inv = inv_norm[r];
  const TG* gr = g + (size_t)r * g_pitch;
  auto gv = [&](int k) { return g_second >= 0 ? ldf(gr, (size_t)k) + ldf(gr, (size_t)(g_second + k)) : ldf(gr, (size_t)k); };
  float dot = 0.f;
  for (int k = lane; k < dim; k += 32) dot = fmaf(ldf(x, (size_t)r * dim + k) * inv, gv(k), dot);
  dot = warp_sum(dot);
  for (int k = lane; k < dim; k += 32) {
    const size_t i = (size_t)r * dim + k;
    dx[i] = (gv(k) - ldf(x, i) * inv * dot) * inv;
  }
}

struct SumSources {
  const float4* src[15];
  int n;
};
// A handful of CTAs has to stream hundreds of MB (the kernel runs beside a resident persistent kernel), so every
// thread keeps kSumUnroll independent 16-byte loads per source in flight.
constexpr int kSumUnroll = 8;
__global__ void __launch_bounds__(256) sum_into_kernel(float4* __restrict__ dst, const SumSources ss, size_t n4) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; i + (kSumUnroll - 1) * stride < n4; i += kSumUnroll * stride) {
    float4 a[kSumUnroll];
#pragma unroll
    for (int u = 0; u < kSumUnroll; ++u) a[u] = dst[i + u * stride];
#pragma unroll 1
    for (int s = 0; s < ss.n; ++s) {
      float4 v[kSumUnroll];
#pragma unroll
      for (int u = 0; u < kSumUnroll; ++u) v[u] = __ldcs(ss.src[s] + i + u * stride);
#pragma unroll
      for (int u = 0; u < kSumUnroll; ++u) {
        a[u].x += v[u].x;
        a[u].y += v[u].y;
        a[u].z += v[u].z;
        a[u].w += v[u].w;
      }
    }
#pragma unroll
    for (int u = 0; u < kSumUnroll; ++u) dst[i + u * stride] = a[u];
  }
  for (; i < n4; i += stride) {
    float4 a = dst[i];
    for (int s = 0; s < ss.n; ++s) {
      const float4 v = ss.src[s][i];
      a.x += v.x;
      a.y += v.y;
      a.z += v.z;
      a.w += v.w;
    }
    dst[i] = a;
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ x, size_t n, __nv_bfloat16* __restrict__ y) {
  const size_t i = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(x + i);
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(y + i) = o;
  } else {
    for (size_t k = i; k < n; ++k) y[k] = __float2bfloat16(x[k]);
  }
}

// ------------------------------------------------------------------------------ materialised logits (K6)
// One block per scored row (b, t), t < T-1: single streaming pass over V logits with a per-thread online
// (max, sum), block reduction, target gather.  Writes lse and z_tgt per row.
template <typename T>
__global__ void __launch_bounds__(256)
logits_lse_kernel(const T* __restrict__ logits, const int* __restrict__ row_label, int T_len, int vocab,
                  float* __restrict__ lse, float* __restrict__ ztgt) {
  const size_t r = blockIdx.x;
  const int t = (int)(r % T_len);
  if (t + 1 >= T_len) {
    if (threadIdx.x == 0) {
      lse[r] = 0.f;
      ztgt[r] = 0.f;
    }
    return;
  }
  const T* z = logits + r * (size_t)vocab;
  float m = -3.0e38f, s = 0.f;  // finite floor: (-inf) - (-inf) never appears
  for (int v = threadIdx.x; v < vocab; v += blockDim.x) {
    const float x = ldf(z, v) * kLog2e;
    const float mn = fmaxf(m, x);
    s = s * fast_exp2(m - mn) + fast_exp2(x - mn);
    if (x != x) s = NAN;
    m = mn;
  }
  __shared__ float sm[8], ss[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float wm = warp_max(m);
  float ws = warp_sum(s * fast_exp2(m - wm));
  if (lane == 0) {
    sm[warp] = wm;
    ss[warp] = ws;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float gm = -3.0e38f;
    for (int w = 0; w < 8; ++w) gm = fmaxf(gm, sm[w]);
    float gs = 0.f;
    for (int w = 0; w < 8; ++w) gs += ss[w] * exp2f(sm[w] - gm);
    lse[r] = (gm + log2f(gs)) * kLn2;
    const int lab = row_label[r];
    ztgt[r] = lab >= 0 ? ldf(z, lab) : 0.f;
  }
}

// dlogits[r, v] = coef[r] * ([v == label] - exp(z - lse[r])); rows with coef == 0 (masked, last position) are zeroed.
template <typename T>
__device__ __forceinline__ void stf(T* p, size_t i, float v);
template <>
__device__ __forceinline__ void stf<float>(float* p, size_t i, float v) { p[i] = v; }
template <>
__device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, size_t i, float v) { p[i] = __float2bfloat16(v); }

template <typename T>
__global__ void __launch_bounds__(256)
logits_grad_kernel(const T* __restrict__ logits, const int* __restrict__ row_label, const float* __restrict__ lse,
                   const float* __restrict__ coef, int vocab, T* __restrict__ dlogits) {
  const size_t r = blockIdx.x;
  const float c = coef[r];
  const T* z = logits + r * (size_t)vocab;
  T* dz = dlogits + r * (size_t)vocab;
  if (c == 0.f) {
    for (int v = threadIdx.x; v < vocab; v += blockDim.x) stf(dz, v, 0.f);
    return;
  }
  const float l2 = lse[r] * kLog2e;
  const int lab = row_label[r];
  for (int v = threadIdx.x; v < vocab; v += blockDim.x) {
    const float p = fast_exp2(ldf(z, v) * kLog2e - l2);
    stf(dz, v, c * ((v == lab ? 1.f : 0.f) - p));
  }
}

}  // namespace
}  // namespace pgica

// =========================================================================================== C ABI
extern "C" {

using namespace pgica;

int pgica_prep_rows(const int64_t* labels, const void* mask, int mask_kind, int64_t nseq, int64_t seqlen,
                    int64_t vocab, int32_t* row_label, float* row_weight, void* stream) {
  PGICA_REQUIRE(labels && row_label && row_weight, "prep_rows: null pointer");
  PGICA_REQUIRE(nseq > 0 && seqlen > 1 && vocab > 0, "prep_rows: need nseq > 0, seqlen > 1, vocab > 0");
  PGICA_REQUIRE(mask_kind == PGICA_MASK_NONE || mask, "prep_rows: mask pointer missing for mask_kind %d", mask_kind);
  PGICA_REQUIRE(mask_kind >= PGICA_MASK_NONE && mask_kind <= PGICA_MASK_I32, "prep_rows: unknown mask_kind %d",
                mask_kind);
  const int64_t n = nseq * seqlen;
  PGICA_REQUIRE(n < (1ll << 31), "prep_rows: too many rows");
  prep_rows_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const long long*>(labels), mask, mask_kind, (int)nseq, (int)seqlen, (int)vocab, row_label,
      row_weight);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_seq_reduce(const float* lse, const float* ztgt, const float* row_weight, int64_t nseq, int64_t seqlen,
                     int length_normalize, float* seq_logp, float* nll_sum, void* stream) {
  PGICA_REQUIRE(lse && ztgt && row_weight && seq_logp, "seq_reduce: null pointer");
  PGICA_REQUIRE(nseq > 0 && seqlen > 1, "seq_reduce: bad shape");
  if (nll_sum) PGICA_CUDA_OK(cudaMemsetAsync(nll_sum, 0, sizeof(float), (cudaStream_t)stream));
  seq_reduce_kernel<<<(unsigned)ceil_div(nseq, 4), 128, 0, (cudaStream_t)stream>>>(
      lse, ztgt, row_weight, (int)nseq, (int)seqlen, length_normalize, seq_logp, nll_sum);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_row_coef(const float* grad_seq, const float* row_weight, int64_t nseq, int64_t seqlen, int length_normalize,
                   float sign, float* coef, void* stream) {
  PGICA_REQUIRE(grad_seq && row_weight && coef, "row_coef: null pointer");
  row_coef_kernel<<<(unsigned)ceil_div(nseq, 4), 128, 0, (cudaStream_t)stream>>>(
      grad_seq, row_weight, (int)nseq, (int)seqlen, length_normalize, sign, coef);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_dpo_loss_fwd(const float* pc, const float* pr, const float* rc, const float* rr, int64_t n,
                       int64_t n_global, float beta, float label_smoothing, float* loss, float* metrics, float* dpc,
                       void* stream) {
  PGICA_REQUIRE(pc && pr && loss && metrics && dpc, "dpo_loss: null pointer");
  PGICA_REQUIRE((rc == nullptr) == (rr == nullptr), "dpo_loss: reference log-probs must come as a pair");
  PGICA_REQUIRE(n > 0 && n < (1 << 24) && n_global >= n, "dpo_loss: bad pair count");
  PGICA_REQUIRE(label_smoothing >= 0.f && label_smoothing <= 1.f, "dpo_loss: label_smoothing outside [0,1]");
  dpo_loss_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(pc, pr, rc, rr, (int)n, beta, label_smoothing,
                                                       1.f / (float)n_global, loss, metrics, dpc);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_scale_by_scalar(const float* a, const float* scalar, float mult, int64_t n, float* out, void* stream) {
  PGICA_REQUIRE(a && scalar && out && n > 0, "scale_by_scalar: bad argument");
  scale_by_scalar_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(a, scalar, mult, (int)n, out);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_ntxent_loss(const float* lse_row, const float* diag, const float* lse_col_owned, int64_t n,
                      float inv_denom, float* loss, void* stream) {
  PGICA_REQUIRE(lse_row && diag && lse_col_owned && loss && n > 0, "ntxent_loss: bad argument");
  ntxent_loss_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(lse_row, diag, lse_col_owned, (int)n, inv_denom, loss);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_lse_combine(const float* parts, int64_t nparts, int64_t n, float* out, void* stream) {
  PGICA_REQUIRE(parts && out && nparts > 0 && n > 0, "lse_combine: bad argument");
  lse_combine_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(parts, (int)nparts, (int)n, out);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_ntxent_coef(const float* grad, float mult, int64_t n, int64_t tgt_offset, int64_t tgt_limit, float* coef,
                      int32_t* tgt, void* stream) {
  PGICA_REQUIRE(grad && coef && tgt && n > 0, "ntxent_coef: bad argument");
  ntxent_coef_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(grad, mult, (int)n, (int)tgt_offset,
                                                                                  (int)tgt_limit, coef, tgt);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_rownorm_fwd(const void* x, int x_is_bf16, int64_t rows, int64_t dim, float eps, void* y_bf16,
                      float* inv_norm, void* left3_bf16, void* right3_bf16, void* stream) {
  PGICA_REQUIRE(x && y_bf16 && inv_norm && rows > 0 && dim > 0, "rownorm_fwd: bad argument");
  PGICA_REQUIRE((left3_bf16 == nullptr) == (right3_bf16 == nullptr), "rownorm_fwd: split outputs come as a pair");
  __nv_bfloat16* l3 = static_cast<__nv_bfloat16*>(left3_bf16);
  __nv_bfloat16* r3 = static_cast<__nv_bfloat16*>(right3_bf16);
  const unsigned grid = (unsigned)ceil_div(rows, 8);
  if (x_is_bf16)
    rownorm_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(x), (int)rows, (int)dim, eps, static_cast<__nv_bfloat16*>(y_bf16), inv_norm,
        l3, r3, 1);
  else
    rownorm_fwd_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(x), (int)rows, (int)dim,
                                                                      eps, static_cast<__nv_bfloat16*>(y_bf16),
                                                                      inv_norm, l3, r3, 1);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_split3_bf16(const float* x, int64_t rows, int64_t dim, void* left3_bf16, void* right3_bf16, void* stream) {
  PGICA_REQUIRE(x && left3_bf16 && right3_bf16 && rows > 0 && dim > 0, "split3: bad argument");
  rownorm_fwd_kernel<float><<<(unsigned)ceil_div(rows, 8), 256, 0, (cudaStream_t)stream>>>(
      x, (int)rows, (int)dim, 0.f, nullptr, nullptr, static_cast<__nv_bfloat16*>(left3_bf16),
      static_cast<__nv_bfloat16*>(right3_bf16), 0);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_rownorm_bwd(const void* x, int x_is_bf16, const float* inv_norm, const void* g, int g_is_bf16, int64_t rows,
                      int64_t dim, int64_t g_pitch, int64_t g_second, float* dx, void* stream) {
  PGICA_REQUIRE(x && inv_norm && g && dx && rows > 0 && dim > 0, "rownorm_bwd: bad argument");
  PGICA_REQUIRE(g_pitch >= dim && (g_second < 0 || g_second + dim <= g_pitch),
                "rownorm_bwd: gradient layout (pitch %lld, second block at %lld) does not hold %lld columns",
                (long long)g_pitch, (long long)g_second, (long long)dim);
  const unsigned grid = (unsigned)ceil_div(rows, 8);
  cudaStream_t st = (cudaStream_t)stream;
  const int r = (int)rows, d = (int)dim;
  if (x_is_bf16 && g_is_bf16)
    rownorm_bwd_kernel<<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), inv_norm,
                                             static_cast<const __nv_bfloat16*>(g), r, d, g_pitch, g_second, dx);
  else if (x_is_bf16)
    rownorm_bwd_kernel<<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), inv_norm,
                                             static_cast<const float*>(g), r, d, g_pitch, g_second, dx);
  else if (g_is_bf16)
    rownorm_bwd_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(x), inv_norm,
                                             static_cast<const __nv_bfloat16*>(g), r, d, g_pitch, g_second, dx);
  else
    rownorm_bwd_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(x), inv_norm, static_cast<const float*>(g), r, d,
                                             g_pitch, g_second, dx);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_sum_into_f32(float* dst, const void* const* srcs_host, int n_src, int64_t n, int max_ctas, void* stream) {
  PGICA_REQUIRE(dst && srcs_host && n_src >= 1 && n_src <= 15 && n > 0 && n % 4 == 0, "sum_into: bad argument");
  SumSources ss{};
  ss.n = n_src;
  for (int s = 0; s < n_src; ++s) {
    PGICA_REQUIRE(srcs_host[s] && (reinterpret_cast<uintptr_t>(srcs_host[s]) & 15u) == 0, "sum_into: source %d unaligned", s);
    ss.src[s] = static_cast<const float4*>(srcs_host[s]);
  }
  PGICA_REQUIRE((reinterpret_cast<uintptr_t>(dst) & 15u) == 0, "sum_into: destination unaligned");
  const size_t n4 = (size_t)n / 4;
  int64_t grid = ceil_div((int64_t)n4, 256);
  const int64_t cap = max_ctas > 0 ? max_ctas : device_sm_count();
  if (grid > cap) grid = cap;
  sum_into_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float4*>(dst), ss, n4);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_cast_f32_to_bf16(const float* x, int64_t n, void* y_bf16, void* stream) {
  PGICA_REQUIRE(x && y_bf16 && n > 0, "cast: bad argument");
  PGICA_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(y_bf16) & 7u) == 0,
                "cast: pointers must be 16-byte (src) / 8-byte (dst) aligned");
  cast_f32_bf16_kernel<<<(unsigned)ceil_div(ceil_div(n, 4), 256), 256, 0, (cudaStream_t)stream>>>(
      x, (size_t)n, static_cast<__nv_bfloat16*>(y_bf16));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_logits_lse(const void* logits, int logits_is_bf16, const int32_t* row_label, int64_t nseq, int64_t seqlen,
                     int64_t vocab, float* lse, float* ztgt, void* stream) {
  PGICA_REQUIRE(logits && row_label && lse && ztgt, "logits_lse: null pointer");
  PGICA_REQUIRE(nseq > 0 && seqlen > 1 && vocab > 0 && nseq * seqlen < (1ll << 31), "logits_lse: bad shape");
  const unsigned grid = (unsigned)(nseq * seqlen);
  if (logits_is_bf16)
    logits_lse_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(logits), row_label, (int)seqlen, (int)vocab, lse, ztgt);
  else
    logits_lse_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(logits), row_label,
                                                                     (int)seqlen, (int)vocab, lse, ztgt);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_logits_grad(const void* logits, int logits_is_bf16, const int32_t* row_label, const float* lse,
                      const float* coef, int64_t nseq, int64_t seqlen, int64_t vocab, void* dlogits, void* stream) {
  PGICA_REQUIRE(logits && row_label && lse && coef && dlogits, "logits_grad: null pointer");
  PGICA_REQUIRE(nseq > 0 && seqlen > 1 && vocab > 0 && nseq * seqlen < (1ll << 31), "logits_grad: bad shape");
  const unsigned grid = (unsigned)(nseq * seqlen);
  if (logits_is_bf16)
    logits_grad_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(logits), row_label, lse, coef, (int)vocab,
        static_cast<__nv_bfloat16*>(dlogits));
  else
    logits_grad_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(logits), row_label, lse,
                                                                      coef, (int)vocab, static_cast<float*>(dlogits));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

}  // extern "C"
