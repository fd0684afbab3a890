// The softmax-gradient tile every backward kernel (sgg.cu, sgg_x.cu, sgg_f.cu) turns its logits into:
//
//   G(i, j) = rC[i] * (exp(s*z_ij - rL[i]) - [j == rT[i]]) + cC[j] * (exp(s*z_ij - cL[j]) - [i == cT[j]])
//
// An epilogue thread owns one row of a 128 x 128 tile, takes it out of TMEM 32 columns at a time, and writes it as bf16
// into a [128][128] tile of two 128-B-swizzled [128][64] boxes, the K-major operand layout tcgen05.mma reads.
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace pgica {

constexpr int kGTile = 128;                        // rows and columns of a G tile
constexpr uint32_t kGBoxBytes = kGTile * 64 * 2;  // 16 KB: one [128][64] bf16 box of a G tile

// Statistics of G.  A null r_lse (c_lse) drops the row (column) term, a null target pointer its one-hot.
struct SoftmaxGradStats {
  float c;  // scale * log2(e): exponentials are taken base 2
  const float *r_lse, *r_coef;
  const int* r_tgt;
  const float *c_lse, *c_coef;
  const int* c_tgt;
  // the statistics of G^T: rows and columns trade places
  SoftmaxGradStats transposed() const { return {c, c_lse, c_coef, c_tgt, r_lse, r_coef, r_tgt}; }
};

// True when 2c < 100 for c = scale * log2(e): the one-exponential form (sgg_f.cu, kShared) keeps every factor finite in
// fp32 for unit-norm rows, whose logits are bounded by the scale.  False for NaN.
inline bool bounded_logits(float c) { return 2.0f * c < 100.0f; }

// Calls f(row, col) with std::integral_constant<bool> arguments for the terms present: both, the row term or the
// column term; these are the only kernel instantiations.
template <class F>
int with_terms(bool row, bool col, F&& f) {
  if (row && col) return f(std::true_type{}, std::true_type{});
  if (row) return f(std::true_type{}, std::false_type{});
  return f(std::false_type{}, std::true_type{});
}

// One row's or one column's statistics: lse in log2 units l, coefficient cf, target tg (-1: none); zeros when the
// term is absent or the index is not `valid`.
template <bool kRow>
__device__ __forceinline__ void load_row_stat(const SoftmaxGradStats& s, int row, bool valid, float& l, float& cf,
                                              int& tg) {
  l = 0.f;
  cf = 0.f;
  tg = -1;
  if (kRow && valid) {
    l = s.r_lse[row] * kLog2e;
    cf = s.r_coef[row];
    tg = s.r_tgt ? s.r_tgt[row] : -1;
  }
}

template <bool kCol>
__device__ __forceinline__ void load_col_stat(const SoftmaxGradStats& s, int col, bool valid, float& l, float& cf,
                                              int& tg) {
  l = 0.f;
  cf = 0.f;
  tg = -1;
  if (kCol && valid) {
    l = s.c_lse[col] * kLog2e;
    cf = s.c_coef[col];
    tg = s.c_tgt ? s.c_tgt[col] : -1;
  }
}

// Column `et` of the tile's column statistics in shared memory: s_col = {lse [kGTile] | coefficient [kGTile] |
// target [kGTile]}.  kShared (one exponential for both terms, see sgg_f.cu): {raw coefficient, for the one-hot fix-up |
// the column's factor 2^(c - lse) coefficient | target}.
template <bool kShared>
__device__ __forceinline__ void stage_col_stat(float* s_col, int et, float l, float cf, int tg, float c) {
  s_col[et] = kShared ? cf : l;
  s_col[kGTile + et] = kShared ? cf * fast_exp2(c - l) : cf;
  reinterpret_cast<int*>(s_col + 2 * kGTile)[et] = tg;
}

// G for 32 columns [32 ch, 32 ch + 32) of the tile from the raw logits z of one row with statistics (rl, rc).  `row` is
// the row's global index (matched against the column targets), rrel = (row target) - (first column of the tile).
// kShared: rs = rc * 2^(c - rl), the row's factor of the shared exponential.
template <bool kRow, bool kCol, bool kShared = false>
__device__ __forceinline__ void g_chunk(const uint32_t (&z)[32], float c, float rl, float rc, float rs, int row, int rrel,
                                        const float* s_col, int ch, float (&g)[32]) {
  const float* s_cl = s_col;
  const float* s_cc = s_col + kGTile;
  const int* s_ct = reinterpret_cast<const int*>(s_col + 2 * kGTile);
#pragma unroll
  for (int jj = 0; jj < 32; ++jj) {
    if (kShared) {
      g[jj] = fast_exp2(fmaf(__uint_as_float(z[jj]), c, -c)) * (rs + s_cc[ch * 32 + jj]);
      continue;
    }
    const float t = __uint_as_float(z[jj]) * c;
    float v = 0.f;
    if (kRow) v = rc * fast_exp2(t - rl);
    if (kCol) {
      const int cj = ch * 32 + jj;
      const float ccj = s_cc[cj];
      v = fmaf(ccj, fast_exp2(t - s_cl[cj]), v);
      if (s_ct[cj] == row) v -= ccj;
    }
    g[jj] = v;
  }
  if (kRow && rrel >= 0 && (rrel >> 5) == ch) {
    const int jj0 = rrel & 31;
    const float hot = kShared ? rc + s_cl[ch * 32 + jj0] : rc;  // mirrored targets: both one-hots sit here
#pragma unroll
    for (int jj = 0; jj < 32; ++jj)
      if (jj == jj0) g[jj] -= hot;
  }
}

__device__ __forceinline__ void pack_g_chunk(const float (&g)[32], uint32_t* gp) {
#pragma unroll
  for (int i = 0; i < 16; ++i) gp[i] = pack_bf16x2(g[2 * i], g[2 * i + 1]);
}

// The 16 bf16 pairs gp of chunk ch of row `row` into the G tile at shared address `tile`.
__device__ __forceinline__ void store_g_chunk(uint32_t tile, int row, int ch, const uint32_t* gp) {
#pragma unroll
  for (int c4 = 0; c4 < 4; ++c4) {
    const uint32_t off = (uint32_t)(ch >> 1) * kGBoxBytes + sw128_offset(row, (ch & 1) * 4 + c4);
    st_smem_v4(tile + off, gp[c4 * 4 + 0], gp[c4 * 4 + 1], gp[c4 * 4 + 2], gp[c4 * 4 + 3]);
  }
}

// Columns [col, col + 32) of row `row` of Out (fp32 or bf16, ldo elements per row) from a 32-column TMEM chunk.
// kTail: element-wise stores past column k - 32 (k a multiple of 8 only); the caller has checked col < k.
template <bool kTail>
__device__ __forceinline__ void store_out_chunk(void* out, int out_bf16, int ldo, int row, int col, int k,
                                                const uint32_t (&r)[32]) {
  if (!kTail || col + 32 <= k) {
    if (out_bf16) {
      uint4* dst = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) + (size_t)row * ldo + col);
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        uint4 v;
        v.x = pack_bf16x2(__uint_as_float(r[c4 * 8 + 0]), __uint_as_float(r[c4 * 8 + 1]));
        v.y = pack_bf16x2(__uint_as_float(r[c4 * 8 + 2]), __uint_as_float(r[c4 * 8 + 3]));
        v.z = pack_bf16x2(__uint_as_float(r[c4 * 8 + 4]), __uint_as_float(r[c4 * 8 + 5]));
        v.w = pack_bf16x2(__uint_as_float(r[c4 * 8 + 6]), __uint_as_float(r[c4 * 8 + 7]));
        dst[c4] = v;
      }
    } else {
      uint4* dst = reinterpret_cast<uint4*>(static_cast<float*>(out) + (size_t)row * ldo + col);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) dst[c4] = make_uint4(r[c4 * 4], r[c4 * 4 + 1], r[c4 * 4 + 2], r[c4 * 4 + 3]);
    }
  } else {
    for (int jj = 0; jj < 32 && col + jj < k; ++jj) {
      if (out_bf16)
        static_cast<__nv_bfloat16*>(out)[(size_t)row * ldo + col + jj] = __float2bfloat16(__uint_as_float(r[jj]));
      else
        static_cast<float*>(out)[(size_t)row * ldo + col + jj] = __uint_as_float(r[jj]);
    }
  }
}

// Diagnostics build (-DPGICA_TRACE): per-role cycle accounting.  LAP(i) charges the cycles since the previous lap to
// slot i; LAP_FLUSH(buf, base, n) writes slots [0, n) to buf[block][base, base + n) of a [grid][kTraceSlots] int64 array.
constexpr int kTraceSlots = 24;
#ifdef PGICA_TRACE
__device__ __forceinline__ long long trace_clock() {
#ifdef __CUDA_ARCH__
  return clock64();
#else
  return 0;  // host pass of the template: never called
#endif
}
template <int N>
struct TraceLap {
  long long t, acc[N];
  __device__ TraceLap() : t(trace_clock()) {
    for (int i = 0; i < N; ++i) acc[i] = 0;
  }
  __device__ void operator()(int i) {
    const long long n = trace_clock();
    acc[i] += n - t;
    t = n;
  }
  __device__ void flush(long long* buf, int base, int n) {
    if (buf)
      for (int i = 0; i < n; ++i) buf[(size_t)blockIdx.x * kTraceSlots + base + i] = acc[i];
  }
};
#define LAP_DECL(N) TraceLap<N> lap
#define LAP(i) lap(i)
#define LAP_FLUSH(buf, base, n) lap.flush(buf, base, n)
#else
#define LAP_DECL(N) ((void)0)
#define LAP(i) ((void)0)
#define LAP_FLUSH(buf, base, n) ((void)0)
#endif

}  // namespace pgica
