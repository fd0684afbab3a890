// SURVEY 8(f) row 2, last part: the AdamW step that ends every micro-step of the trainer (pkg/training/trainer.py:
// 494-520, 619-633), over ALL fp32 tensors of a parameter group in one launch, with the global-norm clip of
// pgica_grad_norm_clip (clip = 0: norm only) folded in and a non-finite norm skipping the step on the device.
//   update   one pass over p, g, m, v (fixed-size chunks, 16-byte vectors where all four pointers allow them):
//            torch/optim/adam.py::_single_tensor_adam with decoupled weight decay, element for element:
//              g' = g * clip_coef                        (one rounding, never contracted; g in memory is not written)
//              p *= 1 - lr*wd
//              m  = lerp(m, g', 1 - beta1)               (torch's lerp: m + w*(g'-m) for w < 0.5, else g' - (g'-m)*(1-w))
//              v  = beta2*v + (1 - beta2)*g'^2
//              p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps),   bc_k = 1 - beta_k^(s+1), s = the stored step
//            m and v in fp32 with fp32 scalars (double values rounded once), as torch's single-tensor step computes them.
//            The new p is formed in double from the fp32 p, m', v' and rounded once: in fp32 its update term passes
//            through about nine roundings (sqrt, two scalars, fma, quotient, step size, final fma, plus those of m'), and
//            the fp32 form leaves 4 ulps of the term magnitudes on some elements of a 16 M-element random state.  The
//            per-tensor scalars lr / bc1 and 1 / sqrt(bc2) are computed once per block from the device-resident step.
//   count    one thread per tensor: step += 1 (a second launch, so no block of the update sees a half-counted step)
// Algorithmic bytes: 28 per element (p, g, m, v read; p, m, v written).
#include <math.h>
#include <stdlib.h>

#include "common.h"

namespace pgica {
namespace {

constexpr int kChunk = 32768;  // elements per block
constexpr int kThreads = 256;

struct AdamTensor {
  float* p;
  const float* g;
  float* m;
  float* v;
  float* step;
  int64_t numel;
};

struct AdamHyper {
  double lr, beta1, beta2, eps;
  double a;    // 1 - lr*wd
  float w1;    // 1 - beta1
  float b2;    // beta2
  float omb2;  // 1 - beta2
};

struct Elem {
  float p, m, v;
};

__device__ __forceinline__ Elem adamw_elem(float p, float g, float m, float v, float coef, const AdamHyper& h,
                                           double step_size, double rsbc2) {
  const float gc = __fmul_rn(g, coef);
  m = h.w1 < 0.5f ? fmaf(h.w1, __fsub_rn(gc, m), m) : fmaf(-__fsub_rn(gc, m), __fsub_rn(1.0f, h.w1), gc);
  v = fmaf(__fmul_rn(h.omb2, gc), gc, __fmul_rn(v, h.b2));
  const double denom = fma(sqrt((double)v), rsbc2, h.eps);  // sqrt(v) / sqrt(bc2) + eps
  p = (float)fma(-step_size, (double)m / denom, (double)p * h.a);
  return {p, m, v};
}

// table: n_tensors AdamTensor entries, then n_tensors + 1 int32 chunk prefix offsets
__global__ void __launch_bounds__(kThreads) adamw_update_kernel(const AdamTensor* __restrict__ table,
                                                                const int* __restrict__ chunk_start, int n_tensors,
                                                                AdamHyper h, const float* __restrict__ grad_stats) {
  __shared__ int s_t;
  __shared__ double s_step_size, s_rsbc2;
  float coef = 1.0f;
  if (grad_stats) {
    if (!(grad_stats[2] != 0.f)) return;  // non-finite global norm: nothing is written
    coef = grad_stats[1];
  }
  const int b = blockIdx.x;
  // the tensor whose chunk range holds this block: every thread tests a few boundaries, exactly one matches
  for (int i = threadIdx.x; i < n_tensors; i += kThreads)
    if (chunk_start[i] <= b && b < chunk_start[i + 1]) s_t = i;
  __syncthreads();
  const AdamTensor t = table[s_t];
  if (threadIdx.x == 0) {
    const double s1 = (double)*t.step + 1.0;
    const double bc1 = 1.0 - pow(h.beta1, s1), bc2 = 1.0 - pow(h.beta2, s1);
    s_step_size = h.lr / bc1;
    s_rsbc2 = 1.0 / sqrt(bc2);
  }
  __syncthreads();
  const double step_size = s_step_size, rsbc2 = s_rsbc2;
  const int64_t off = (int64_t)(b - chunk_start[s_t]) * kChunk;
  const int count = (int)(t.numel - off < kChunk ? t.numel - off : kChunk);
  float* p = t.p + off;
  const float* g = t.g + off;
  float* m = t.m + off;
  float* v = t.v + off;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15u) == 0;
  const int n4 = vec ? count / 4 : 0;
  float4* p4 = reinterpret_cast<float4*>(p);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  // two 16-byte vectors of each of the four arrays in flight per thread
  int i = threadIdx.x;
  for (; i + kThreads < n4; i += 2 * kThreads) {
    float4 P[2], G[2], M[2], V[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      P[u] = p4[i + u * kThreads];
      G[u] = __ldcs(g4 + i + u * kThreads);
      M[u] = m4[i + u * kThreads];
      V[u] = v4[i + u * kThreads];
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const Elem e0 = adamw_elem(P[u].x, G[u].x, M[u].x, V[u].x, coef, h, step_size, rsbc2);
      const Elem e1 = adamw_elem(P[u].y, G[u].y, M[u].y, V[u].y, coef, h, step_size, rsbc2);
      const Elem e2 = adamw_elem(P[u].z, G[u].z, M[u].z, V[u].z, coef, h, step_size, rsbc2);
      const Elem e3 = adamw_elem(P[u].w, G[u].w, M[u].w, V[u].w, coef, h, step_size, rsbc2);
      p4[i + u * kThreads] = make_float4(e0.p, e1.p, e2.p, e3.p);
      m4[i + u * kThreads] = make_float4(e0.m, e1.m, e2.m, e3.m);
      v4[i + u * kThreads] = make_float4(e0.v, e1.v, e2.v, e3.v);
    }
  }
  for (; i < n4; i += kThreads) {
    const float4 P = p4[i], G = __ldcs(g4 + i), M = m4[i], V = v4[i];
    const Elem e0 = adamw_elem(P.x, G.x, M.x, V.x, coef, h, step_size, rsbc2);
    const Elem e1 = adamw_elem(P.y, G.y, M.y, V.y, coef, h, step_size, rsbc2);
    const Elem e2 = adamw_elem(P.z, G.z, M.z, V.z, coef, h, step_size, rsbc2);
    const Elem e3 = adamw_elem(P.w, G.w, M.w, V.w, coef, h, step_size, rsbc2);
    p4[i] = make_float4(e0.p, e1.p, e2.p, e3.p);
    m4[i] = make_float4(e0.m, e1.m, e2.m, e3.m);
    v4[i] = make_float4(e0.v, e1.v, e2.v, e3.v);
  }
  // the tail, and whole chunks whose four arrays do not share 16-byte alignment (e.g. a leaf carved from a flat
  // buffer at an odd element offset)
  for (int j = n4 * 4 + threadIdx.x; j < count; j += kThreads) {
    const Elem e = adamw_elem(p[j], g[j], m[j], v[j], coef, h, step_size, rsbc2);
    p[j] = e.p;
    m[j] = e.m;
    v[j] = e.v;
  }
}

__global__ void __launch_bounds__(kThreads) adamw_count_kernel(const AdamTensor* __restrict__ table, int n_tensors,
                                                               const float* __restrict__ grad_stats) {
  if (grad_stats && !(grad_stats[2] != 0.f)) return;
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i < n_tensors) *table[i].step += 1.0f;
}

size_t table_bytes(int n) { return align_up((size_t)n * sizeof(AdamTensor), 16) + (size_t)(n + 1) * sizeof(int); }

}  // namespace
}  // namespace pgica

extern "C" {

using namespace pgica;

int pgica_adamw_workspace_bytes(int n_tensors, size_t* bytes_host) {
  PGICA_REQUIRE(bytes_host && n_tensors >= 1, "adamw: bad argument");
  *bytes_host = align_up(table_bytes(n_tensors), 256);
  return PGICA_OK;
}

int pgica_adamw_step(void* const* params_host, const void* const* grads_host, void* const* exp_avgs_host,
                     void* const* exp_avg_sqs_host, float* const* steps_host, const int64_t* numels_host,
                     int n_tensors, double lr, double beta1, double beta2, double eps, double weight_decay,
                     const float* grad_stats, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(params_host && grads_host && exp_avgs_host && exp_avg_sqs_host && steps_host && numels_host &&
                    n_tensors >= 1 && workspace,
                "adamw: null pointer");
  PGICA_REQUIRE(isfinite(lr) && lr >= 0.0, "adamw: lr must be finite and >= 0");
  PGICA_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0, "adamw: betas must lie in [0, 1)");
  PGICA_REQUIRE(isfinite(eps) && eps >= 0.0, "adamw: eps must be finite and >= 0");
  PGICA_REQUIRE(isfinite(weight_decay) && weight_decay >= 0.0, "adamw: weight_decay must be finite and >= 0");
  const size_t need = table_bytes(n_tensors);
  if (workspace_bytes < need) {
    set_error("adamw: workspace too small");
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  int64_t chunks = 0;
  for (int i = 0; i < n_tensors; ++i) {
    PGICA_REQUIRE(numels_host[i] >= 0 && numels_host[i] < (1ll << 31), "adamw: tensor %d: numel must lie in [0, 2^31)",
                  i);
    PGICA_REQUIRE(steps_host[i] && (numels_host[i] == 0 || (params_host[i] && grads_host[i] && exp_avgs_host[i] &&
                                                             exp_avg_sqs_host[i])),
                  "adamw: tensor %d: null pointer", i);
    chunks += ceil_div(numels_host[i], kChunk);
  }
  PGICA_REQUIRE(chunks < (1ll << 31), "adamw: too many elements");
  // the tensor table, rebuilt on every call (gradients may have moved since the last one), copied ahead of the
  // launches (pageable source: staged before cudaMemcpyAsync returns)
  uint8_t* host = static_cast<uint8_t*>(malloc(need));
  PGICA_REQUIRE(host, "adamw: out of host memory");
  AdamTensor* tab = reinterpret_cast<AdamTensor*>(host);
  int* start = reinterpret_cast<int*>(host + align_up((size_t)n_tensors * sizeof(AdamTensor), 16));
  int64_t k = 0;
  for (int i = 0; i < n_tensors; ++i) {
    tab[i] = {static_cast<float*>(params_host[i]), static_cast<const float*>(grads_host[i]),
              static_cast<float*>(exp_avgs_host[i]), static_cast<float*>(exp_avg_sqs_host[i]), steps_host[i],
              numels_host[i]};
    start[i] = (int)k;
    k += ceil_div(numels_host[i], kChunk);
  }
  start[n_tensors] = (int)k;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemcpyAsync(workspace, host, need, cudaMemcpyHostToDevice, st);
  free(host);
  PGICA_CUDA_OK(e);
  const AdamTensor* d_tab = static_cast<const AdamTensor*>(workspace);
  const int* d_start = reinterpret_cast<const int*>(static_cast<const uint8_t*>(workspace) +
                                                    align_up((size_t)n_tensors * sizeof(AdamTensor), 16));
  AdamHyper h;
  h.lr = lr;
  h.beta1 = beta1;
  h.beta2 = beta2;
  h.eps = eps;
  h.a = 1.0 - lr * weight_decay;
  h.w1 = (float)(1.0 - beta1);
  h.b2 = (float)beta2;
  h.omb2 = (float)(1.0 - beta2);
  if (chunks > 0) {
    adamw_update_kernel<<<(unsigned)chunks, kThreads, 0, st>>>(d_tab, d_start, n_tensors, h, grad_stats);
    PGICA_CUDA_OK(cudaGetLastError());
    count_launches(1);
  }
  adamw_count_kernel<<<(unsigned)ceil_div(n_tensors, kThreads), kThreads, 0, st>>>(d_tab, n_tensors, grad_stats);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

}  // extern "C"
