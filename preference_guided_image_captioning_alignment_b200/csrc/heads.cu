// Head-level entry points: each composes the tensor-core kernels (gemm_lse.cu, sgg.cu) with the small
// plumbing kernels (small.cu) on the caller's stream, carving the caller's workspace.  No allocation,
// no synchronisation, no host round trip (the upstream gradient is read on the device).
#include "common.h"
#include "sgg_tile.cuh"

namespace pgica {
size_t sggx_workspace_bytes();  // sgg_x.cu
bool sggf_supported(int64_t mx, int64_t my, int64_t k);  // sgg_f.cu
bool sggf_single_chunk(int64_t mx, int64_t my, int64_t k);
size_t sggf_workspace_bytes();
int sggf_dispatch(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, const SoftmaxGradStats& stats,
                  void* out_x, int out_x_is_bf16, void* out_y, int out_y_is_bf16, void* workspace,
                  size_t workspace_bytes, cudaStream_t st, uint32_t* progress, int64_t rows_per_segment,
                  bool shared_exponential);

namespace {
// Exchange workspace of backward(): the one-product kernel's, or the dual kernel's when that takes the shape.
size_t backward_workspace_bytes(int64_t mx, int64_t my, int64_t k) {
  const size_t one = sggx_workspace_bytes();
  return sggf_supported(mx, my, k) && sggf_workspace_bytes() > one ? sggf_workspace_bytes() : one;
}

// OutX = G Y (when out_x) and OutY = G^T X (when out_y).  Both from one recomputation of the logits (sgg_f.cu) when the
// dual kernel takes the shape, the workspace holds its exchange ring and a bf16 OutY can be written in one chunk; else
// one launch per product, OutY with the statistics of G^T.  `st` carries scale * log2(e); `scale` is the same scale
// for the C entry points.  shared_exponential: one exponential per element for both terms (see sggf_kernel).
int backward(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale, const SoftmaxGradStats& st,
             void* out_x, int out_x_is_bf16, void* out_y, int out_y_is_bf16, void* ws, size_t ws_bytes, void* stream,
             bool shared_exponential) {
  if (out_x && out_y && sggf_supported(mx, my, k) && ws && ws_bytes >= sggf_workspace_bytes() &&
      (!out_y_is_bf16 || sggf_single_chunk(mx, my, k))) {
    if (shared_exponential)
      return sggf_dispatch(x, y, mx, my, k, st, out_x, out_x_is_bf16, out_y, out_y_is_bf16, ws, ws_bytes,
                           static_cast<cudaStream_t>(stream), nullptr, 0, true);
    return pgica_softmax_grad_gemm_dual(x, y, mx, my, k, scale, st.r_lse, st.r_coef, st.r_tgt, st.c_lse, st.c_coef,
                                        st.c_tgt, out_x, out_x_is_bf16, out_y, out_y_is_bf16, ws, ws_bytes, stream);
  }
  int rc;
  if (out_x) {
    rc = pgica_softmax_grad_gemm(x, y, mx, my, k, scale, st.r_lse, st.r_coef, st.r_tgt, st.c_lse, st.c_coef, st.c_tgt,
                                 out_x, out_x_is_bf16, ws, ws_bytes, stream);
    if (rc != PGICA_OK) return rc;
  }
  if (out_y) {
    const SoftmaxGradStats t = st.transposed();
    rc = pgica_softmax_grad_gemm(y, x, my, mx, k, scale, t.r_lse, t.r_coef, t.r_tgt, t.c_lse, t.c_coef, t.c_tgt, out_y,
                                 out_y_is_bf16, ws, ws_bytes, stream);
    if (rc != PGICA_OK) return rc;
  }
  return PGICA_OK;
}
}  // namespace
}  // namespace pgica

using namespace pgica;

extern "C" {

// ---- internal building blocks defined in the other translation units
// (pgica_softmax_grad_gemm and its workspace query are declared in pgica.h)

int pgica_lmhead_logprob_workspace_bytes(int64_t nseq, int64_t seqlen, int64_t d, int64_t vocab, size_t* bytes_host) {
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  size_t g = 0;
  int rc = pgica_gemm_lse_workspace_bytes(nseq * seqlen, vocab, d, &g);
  if (rc != PGICA_OK) return rc;
  // backward: one float per row for the coefficients + the G-tile exchange ring; forward: the LSE partials
  const size_t bwd =
      align_up((size_t)(nseq * seqlen) * sizeof(float), 256) + backward_workspace_bytes(nseq * seqlen, vocab, d);
  *bytes_host = g > bwd ? g : bwd;
  return PGICA_OK;
}

int pgica_lmhead_logprob_fwd(const void* hidden, const void* weight, const int64_t* labels, const void* mask,
                             int mask_kind, int64_t nseq, int64_t seqlen, int64_t d, int64_t vocab,
                             int length_normalize, float* seq_logp, float* lse, float* ztgt, int32_t* row_label,
                             float* row_weight, float* nll_sum, void* workspace, size_t workspace_bytes,
                             void* stream) {
  PGICA_REQUIRE(hidden && weight && labels && seq_logp && lse && ztgt && row_label && row_weight,
                "lmhead_logprob_fwd: null pointer");
  int rc = pgica_prep_rows(labels, mask, mask_kind, nseq, seqlen, vocab, row_label, row_weight, stream);
  if (rc != PGICA_OK) return rc;
  rc = pgica_gemm_lse(hidden, weight, nseq * seqlen, vocab, d, 1.0f, row_label, 0, lse, ztgt, workspace,
                      workspace_bytes, stream);
  if (rc != PGICA_OK) return rc;
  return pgica_seq_reduce(lse, ztgt, row_weight, nseq, seqlen, length_normalize, seq_logp, nll_sum, stream);
}

int pgica_lmhead_rows_workspace_bytes(int64_t rows, int64_t d, int64_t vocab, size_t* bytes_host) {
  return pgica_lmhead_logprob_workspace_bytes(rows, 1, d, vocab, bytes_host);
}

int pgica_lmhead_rows_bwd(const void* hidden, const void* weight, const int32_t* row_label, const float* lse,
                          const float* ncoef, int64_t rows, int64_t d, int64_t vocab, void* dhidden,
                          int dhidden_is_bf16, void* dweight, int dweight_is_bf16, void* workspace,
                          size_t workspace_bytes, void* stream) {
  PGICA_REQUIRE(hidden && weight && row_label && lse && ncoef, "lmhead_rows_bwd: null pointer");
  PGICA_REQUIRE(dhidden || dweight, "lmhead_rows_bwd: nothing to compute");
  return backward(hidden, weight, rows, vocab, d, 1.0f, {kLog2e, lse, ncoef, row_label, nullptr, nullptr, nullptr},
                  dhidden, dhidden_is_bf16, dweight, dweight_is_bf16, workspace, workspace_bytes, stream, false);
}

int pgica_lmhead_logprob_bwd(const void* hidden, const void* weight, const int32_t* row_label,
                             const float* row_weight, const float* lse, const float* grad_seq, int64_t nseq,
                             int64_t seqlen, int64_t d, int64_t vocab, int length_normalize, void* dhidden,
                             int dhidden_is_bf16, void* dweight, int dweight_is_bf16, void* workspace,
                             size_t workspace_bytes, void* stream) {
  PGICA_REQUIRE(hidden && weight && row_label && row_weight && lse && grad_seq, "lmhead_logprob_bwd: null pointer");
  PGICA_REQUIRE(dhidden || dweight, "lmhead_logprob_bwd: nothing to compute");
  const int64_t rows = nseq * seqlen;
  if (!workspace || workspace_bytes < (size_t)rows * sizeof(float)) {
    set_error("lmhead_logprob_bwd: workspace too small (%zu < %zu)", workspace_bytes, (size_t)rows * sizeof(float));
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  float* ncoef = static_cast<float*>(workspace);  // -grad_seq[b] * w (/len): multiplies (softmax - onehot)
  const size_t coef_bytes = align_up((size_t)rows * sizeof(float), 256);
  void* xws = workspace_bytes > coef_bytes ? static_cast<uint8_t*>(workspace) + coef_bytes : nullptr;
  const size_t xws_bytes = xws ? workspace_bytes - coef_bytes : 0;
  int rc = pgica_row_coef(grad_seq, row_weight, nseq, seqlen, length_normalize, -1.0f, ncoef, stream);
  if (rc != PGICA_OK) return rc;
  return pgica_lmhead_rows_bwd(hidden, weight, row_label, lse, ncoef, rows, d, vocab, dhidden, dhidden_is_bf16,
                               dweight, dweight_is_bf16, xws, xws_bytes, stream);
}

int pgica_lmhead_logprob_bwd_progress(const void* hidden, const void* weight, const int32_t* row_label,
                                      const float* row_weight, const float* lse, const float* grad_seq, int64_t nseq,
                                      int64_t seqlen, int64_t d, int64_t vocab, int length_normalize, void* dhidden,
                                      int dhidden_is_bf16, void* dweight, uint32_t* progress, int64_t rows_per_segment,
                                      int32_t* increments_per_256_rows_host, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  PGICA_REQUIRE(hidden && weight && row_label && row_weight && lse && grad_seq && dhidden && dweight && progress,
                "lmhead_logprob_bwd_progress: null pointer");
  const int64_t rows = nseq * seqlen;
  const size_t coef_bytes = align_up((size_t)rows * sizeof(float), 256);
  if (!workspace || workspace_bytes < coef_bytes + sggf_workspace_bytes()) {
    set_error("lmhead_logprob_bwd_progress: workspace too small (%zu < %zu)", workspace_bytes,
              coef_bytes + sggf_workspace_bytes());
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  PGICA_REQUIRE(sggf_supported(rows, vocab, d), "lmhead_logprob_bwd_progress: needs the dual kernel (d %% 512 == 0)");
  float* ncoef = static_cast<float*>(workspace);
  int rc = pgica_row_coef(grad_seq, row_weight, nseq, seqlen, length_normalize, -1.0f, ncoef, stream);
  if (rc != PGICA_OK) return rc;
  return pgica_softmax_grad_gemm_dual_progress(hidden, weight, rows, vocab, d, 1.0f, lse, ncoef, row_label, nullptr,
                                               nullptr, nullptr, dhidden, dhidden_is_bf16, dweight, 0, progress,
                                               rows_per_segment, increments_per_256_rows_host,
                                               static_cast<uint8_t*>(workspace) + coef_bytes,
                                               workspace_bytes - coef_bytes, stream);
}

int pgica_ntxent_workspace_bytes(int64_t rows_a, int64_t rows_b, int64_t dim, size_t* bytes_host) {
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  size_t g1 = 0, g2 = 0;
  int rc = pgica_gemm_lse_workspace_bytes(rows_a, rows_b, dim, &g1);
  if (rc != PGICA_OK) return rc;
  rc = pgica_gemm_lse_workspace_bytes(rows_b, rows_a, dim, &g2);
  if (rc != PGICA_OK) return rc;
  size_t g3 = 0;
  rc = pgica_gemm_lse_rowcol_workspace_bytes(rows_a, rows_b, dim, &g3);
  if (rc != PGICA_OK) return rc;
  size_t fwd = g1 > g2 ? g1 : g2;
  if (g3 > fwd) fwd = g3;
  const size_t bwd = 2 * align_up((size_t)rows_a * 4, 256) + 2 * align_up((size_t)rows_b * 4, 256) +
                     backward_workspace_bytes(rows_a, rows_b, dim);
  *bytes_host = fwd > bwd ? fwd : bwd;
  return PGICA_OK;
}

int pgica_ntxent_fwd(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                     int64_t diag_offset, float* lse_row, float* diag, float* lse_col_part, void* workspace,
                     size_t workspace_bytes, void* stream) {
  PGICA_REQUIRE(a && b && lse_row && diag && lse_col_part, "ntxent_fwd: null pointer");
  PGICA_REQUIRE(diag_offset >= 0 && diag_offset + rows_a <= rows_b,
                "ntxent_fwd: positives (i, i + %lld) fall outside the %lld columns", (long long)diag_offset,
                (long long)rows_b);
  int rc = pgica_gemm_lse(a, b, rows_a, rows_b, dim, inv_tau, nullptr, diag_offset, lse_row, diag, workspace,
                          workspace_bytes, stream);
  if (rc != PGICA_OK) return rc;
  return pgica_gemm_lse(b, a, rows_b, rows_a, dim, inv_tau, nullptr, -diag_offset, lse_col_part, nullptr, workspace,
                        workspace_bytes, stream);
}

int pgica_ntxent_fwd_bounded(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                             int64_t diag_offset, float* lse_row, float* diag, float* lse_col_part, void* workspace,
                             size_t workspace_bytes, void* stream) {
  // bounded scheme: |t| <= inv_tau * log2(e) for unit-norm rows; keep 2 * that well inside the fp32 exponent range
  if (!bounded_logits(inv_tau * kLog2e))
    return pgica_ntxent_fwd(a, b, rows_a, rows_b, dim, inv_tau, diag_offset, lse_row, diag, lse_col_part, workspace,
                            workspace_bytes, stream);
  PGICA_REQUIRE(a && b && lse_row && diag && lse_col_part, "ntxent_fwd_bounded: null pointer");
  PGICA_REQUIRE(diag_offset >= 0 && diag_offset + rows_a <= rows_b,
                "ntxent_fwd_bounded: positives (i, i + %lld) fall outside the %lld columns", (long long)diag_offset,
                (long long)rows_b);
  return pgica_gemm_lse_rowcol(a, b, rows_a, rows_b, dim, inv_tau, nullptr, diag_offset, lse_row, diag, lse_col_part,
                               workspace, workspace_bytes, stream);
}

static int ntxent_bwd_impl(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                           int64_t diag_offset, const float* lse_row, const float* lse_col, const float* grad_loss,
                           float grad_mult, void* da, int da_is_bf16, void* db, int db_is_bf16, void* workspace,
                           size_t workspace_bytes, void* stream, bool bounded) {
  PGICA_REQUIRE(a && b && lse_row && lse_col && grad_loss, "ntxent_bwd: null pointer");
  PGICA_REQUIRE(da || db, "ntxent_bwd: nothing to compute");
  const size_t sa = align_up((size_t)rows_a * 4, 256), sb = align_up((size_t)rows_b * 4, 256);
  if (!workspace || workspace_bytes < 2 * sa + 2 * sb) {
    set_error("ntxent_bwd: workspace too small (%zu < %zu)", workspace_bytes, 2 * sa + 2 * sb);
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  uint8_t* w = static_cast<uint8_t*>(workspace);
  float* rcoef = reinterpret_cast<float*>(w);
  int32_t* rtgt = reinterpret_cast<int32_t*>(w + sa);
  float* ccoef = reinterpret_cast<float*>(w + 2 * sa);
  int32_t* ctgt = reinterpret_cast<int32_t*>(w + 2 * sa + sb);
  const size_t stat_bytes = 2 * sa + 2 * sb;
  void* xws = workspace_bytes > stat_bytes ? w + stat_bytes : nullptr;
  const size_t xws_bytes = xws ? workspace_bytes - stat_bytes : 0;
  // dS = grad * mult * (P_row + P_col - 2 I);  dA = dS B / tau;  dB = dS^T A / tau
  int rc = pgica_ntxent_coef(grad_loss, grad_mult * inv_tau, rows_a, diag_offset, rows_b, rcoef, rtgt, stream);
  if (rc != PGICA_OK) return rc;
  rc = pgica_ntxent_coef(grad_loss, grad_mult * inv_tau, rows_b, -diag_offset, rows_a, ccoef, ctgt, stream);
  if (rc != PGICA_OK) return rc;
  // bounded: unit-norm rows, so |logit| <= inv_tau, and the column targets built above mirror the row targets: ONE
  // exponential per element serves both softmax terms in the dual kernel
  return backward(a, b, rows_a, rows_b, dim, inv_tau, {inv_tau * kLog2e, lse_row, rcoef, rtgt, lse_col, ccoef, ctgt}, da,
                  da_is_bf16, db, db_is_bf16, xws, xws_bytes, stream, bounded);
}

int pgica_ntxent_bwd(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                     int64_t diag_offset, const float* lse_row, const float* lse_col, const float* grad_loss,
                     float grad_mult, void* da, int da_is_bf16, void* db, int db_is_bf16, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return ntxent_bwd_impl(a, b, rows_a, rows_b, dim, inv_tau, diag_offset, lse_row, lse_col, grad_loss, grad_mult, da,
                         da_is_bf16, db, db_is_bf16, workspace, workspace_bytes, stream, false);
}

int pgica_ntxent_bwd_bounded(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                             int64_t diag_offset, const float* lse_row, const float* lse_col, const float* grad_loss,
                             float grad_mult, void* da, int da_is_bf16, void* db, int db_is_bf16, void* workspace,
                             size_t workspace_bytes, void* stream) {
  // same bound as pgica_ntxent_fwd_bounded; a temperature too small for it takes the two-exponential form
  const bool ok = inv_tau > 0.f && bounded_logits(inv_tau * kLog2e);
  return ntxent_bwd_impl(a, b, rows_a, rows_b, dim, inv_tau, diag_offset, lse_row, lse_col, grad_loss, grad_mult, da,
                         da_is_bf16, db, db_is_bf16, workspace, workspace_bytes, stream, ok);
}

}  // extern "C"
