/*
 * pgica.h — C ABI of the B200 (sm_100a) alignment-loss-head library.
 *
 * The reference (A-SHOJAEI/preference-guided-image-captioning-alignment) is pure Python/PyTorch and
 * has no FFI of its own; each entry point below therefore cites the reference *Python* function whose
 * arithmetic it replaces (paths relative to the reference repository root, "pkg/" =
 * src/preference_guided_image_captioning_alignment/).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions (all entry points):
 *   - return 0 on success, a negative PGICA_ERR_* code otherwise; the message for the calling thread is
 *     available from pgica_last_error().  Nothing throws or exits across this boundary.
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`; the caller owns every buffer,
 *     including `workspace`; the library allocates nothing that outlives a call.
 *   - `stream` is a cudaStream_t (0 = legacy default stream); kernels are enqueued on it, the call does
 *     not synchronise.
 *   - matrices are row-major, contiguous, base pointers 16-byte aligned; bf16 = __nv_bfloat16.
 *   - there is no CPU fallback: on a device that is not sm_100 every compute entry point fails with
 *     PGICA_ERR_UNSUPPORTED_DEVICE.
 */
#ifndef PGICA_H_
#define PGICA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGICA_ABI_VERSION 1

#define PGICA_OK 0
#define PGICA_ERR_INVALID_ARGUMENT (-1)
#define PGICA_ERR_CUDA (-2)
#define PGICA_ERR_UNSUPPORTED_DEVICE (-3)
#define PGICA_ERR_WORKSPACE_TOO_SMALL (-4)

/* dtype tags for mask / float inputs */
#define PGICA_MASK_NONE 0 /* no mask: every position valid (components.py:341-344)  */
#define PGICA_MASK_I64 1  /* int64 {0,1}          (tokenizer attention_mask)        */
#define PGICA_MASK_F32 2  /* float32, MULTIPLIED into the log-prob like the reference */
#define PGICA_MASK_U8 3   /* bool / uint8                                            */
#define PGICA_MASK_I32 4

int pgica_abi_version(void);
const char* pgica_last_error(void);
/* 0 when the current CUDA device is sm_100 (B200); PGICA_ERR_UNSUPPORTED_DEVICE otherwise. */
int pgica_device_check(void);
int pgica_sm_count(void);
/* number of CUDA kernels this library has launched in this process so far */
int64_t pgica_kernel_launches(void);
/* Process-wide tuning options (kernel selection / role split).  Defaults are seeded once, at load time, from the
 * environment variables PGICA_<NAME>; the call path never reads the environment.  Names: "sgg_fused" (1: dual backward
 * kernel when both gradients are wanted; 0: one launch per product), "sggf_plan_r2" / "sggf_plan_c2" (pin the dual
 * kernel's role split; 0 = planner), "sggf_coop" (1: cooperative launch, a refused launch is an error; 0: plain
 * launch), "sggf_single_chunk" (1: keep all of x in one chunk whenever it fits — y streamed once, out_y written once),
 * "sggf_col_groups" (1: the planner may use column groups, 0: never, n > 1: exactly n),
 * "sggf_spread", "sggf_slots", "sggf_producers_only" (tuning / diagnostics), "sgg_cluster"
 * (cluster size of the one-product kernel).  set: 0 or PGICA_ERR_INVALID_ARGUMENT; get: INT64_MIN for an unknown name. */
int pgica_set_option(const char* name, int64_t value);
int64_t pgica_get_option(const char* name);

/* ------------------------------------------------------------------------------------------------
 * K1/K3 core — tensor-core GEMM with a fused online log-sum-exp + target-gather epilogue.
 *
 *   z[i][j] = scale * <a[i,:], b[j,:]>          (never written to memory)
 *   lse[i]  = log sum_j exp(z[i][j])            tgt[i] = z[i][label(i)]
 *
 * label(i) = labels[i] when `labels` != NULL (a negative or >= cols entry yields tgt[i] = 0), else
 * label(i) = i + diag_offset (NT-Xent positives on the diagonal).
 *
 * Replaces, for the LM head: transformers GPT2LMHeadModel.lm_head (modeling_gpt2.py:706, called from
 * pkg/models/model.py:604-610) + F.log_softmax + gather of pkg/models/components.py:346-352 and
 * pkg/models/model.py:1074-1079; for NT-Xent: torch.matmul(...)/temperature + the logsumexp inside
 * F.cross_entropy of pkg/models/model.py:988-995 and pkg/models/components.py:78-81,135-136.
 *
 * a: bf16 [rows][k], b: bf16 [cols][k], k % 8 == 0, scale > 0.  lse, tgt: fp32 [rows].
 * ---------------------------------------------------------------------------------------------- */
int pgica_gemm_lse_workspace_bytes(int64_t rows, int64_t cols, int64_t k, size_t* bytes_host);
int pgica_gemm_lse(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale,
                   const int32_t* labels, int64_t diag_offset, float* lse, float* tgt, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Row AND column log-sum-exp from ONE pass over the tiles (the symmetric cross-entropy of NT-Xent needs both:
 * pkg/models/model.py:994-995, pkg/models/components.py:135-136): lse_col[j] = log sum_i exp(scale*<a_i, b_j>) next to
 * lse_row / tgt as in pgica_gemm_lse.  Every 32-row group of the epilogue publishes, per 32-column chunk, the column
 * sums of exp2(t - shift) with shift = the largest running row maximum in the group; a merge kernel folds the groups.
 * PRECONDITION: bounded logits — 2 * scale * log2(e) * max|<a_i, b_j>| < 100 (unit-norm embeddings with
 * temperature >= 0.03), so that no term can underflow against its group's shift; callers that cannot promise that use
 * two pgica_gemm_lse launches (exact for any input).  Workspace: pgica_gemm_lse_rowcol_workspace_bytes(). */
int pgica_gemm_lse_rowcol_workspace_bytes(int64_t rows, int64_t cols, int64_t k, size_t* bytes_host);
int pgica_gemm_lse_rowcol(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale,
                          const int32_t* labels, int64_t diag_offset, float* lse_row, float* tgt, float* lse_col,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Dense scaled similarity sim[i][j] = scale*<a_i, b_j> (fp32 [rows][cols]) for retrieval-style scoring —
 * TemperatureScaledSimilarity.forward, pkg/models/components.py:61-83 after normalisation — plus the row
 * log-sum-exp.  Same kernel as pgica_gemm_lse with the store epilogue enabled; workspace as for gemm_lse. */
int pgica_similarity(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale, float* sim,
                     float* lse, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2/K4 core — "softmax-gradient GEMM": the backward of both heads, logits recomputed tile-wise.
 *
 *   out[i,:] = sum_j G(i,j) * y[j,:],   z_ij = <x[i,:], y[j,:]>
 *   G(i,j)   = r_coef[i] * (exp(scale*z_ij - r_lse[i]) - [j == r_tgt[i]])      (row term, if r_lse != NULL)
 *            + c_coef[j] * (exp(scale*z_ij - c_lse[j]) - [i == c_tgt[j]])      (column term, if c_lse != NULL)
 *
 * x: bf16 [mx][k], y: bf16 [my][k], out: [mx][k] fp32 or bf16.  Replaces what autograd derives from
 * pkg/models/components.py:346-358 / pkg/models/model.py:1074-1083 (log_softmax, gather, mask, sum) chained
 * into the lm_head matmul, and from F.cross_entropy x2 + matmul in pkg/models/model.py:988-998 /
 * pkg/models/components.py:131-141 (closed forms: SURVEY.md Appendix A).
 * workspace (pgica_softmax_grad_gemm_workspace_bytes, 128-byte aligned): the exchange ring through which the CTAs of
 * a cluster hand each other 128 x 128 bf16 tiles of G (8 tiles per resident cluster, L2-resident, overwritten every
 * 8 tiles).  With workspace == NULL (or k not a multiple of 512) the single-CTA kernel runs, one CTA per
 * (row block, 256-column slice), each recomputing its own tiles.
 * ---------------------------------------------------------------------------------------------- */
int pgica_softmax_grad_gemm_workspace_bytes(int64_t mx, int64_t my, int64_t k, size_t* bytes_host);
int pgica_softmax_grad_gemm(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale,
                            const float* r_lse, const float* r_coef, const int32_t* r_tgt, const float* c_lse,
                            const float* c_coef, const int32_t* c_tgt, void* out, int out_is_bf16, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2+K4 in one launch — "dual softmax-gradient GEMM": both products of a backward pass from ONE tile-wise
 * recomputation of the logits (3 GEMM-units of tensor work instead of the 4 that two pgica_softmax_grad_gemm
 * calls execute):
 *
 *   out_x[i,:] = sum_j G(i,j) * y[j,:]      out_y[j,:] = sum_i G(i,j) * x[i,:]      (G as above)
 *
 * DPO head: x = hidden, y = LM-head weight, row term  =>  out_x = dhidden, out_y = dweight.
 * NT-Xent:  x = a, y = b, both terms                  =>  out_x = da,      out_y = db.
 * k must be a multiple of 512 (<= 2048).  One persistent cooperative grid over all SMs (sgg_f.cu): CTAs either
 * recompute G tiles or keep a 128 x 512 slice of out_x / out_y resident in TMEM; tiles travel through an
 * L2-resident exchange ring inside `workspace` (pgica_softmax_grad_gemm_dual_workspace_bytes, 256-byte aligned).
 * out_y must be fp32 when x has more row blocks than fit one chunk (it is then accumulated in place).
 * When x has FEW row blocks (the compacted Stage-2 batches: 2-4) and out_x is fp32, several X-holder pairs share the
 * sweep over y ("column groups"; out_x is zeroed and the partial sums add-reduced), so the launch scales with the
 * rows of x instead of costing a fixed ~0.5 ms for the GPT-2 vocabulary.
 * ---------------------------------------------------------------------------------------------- */
int pgica_softmax_grad_gemm_dual_workspace_bytes(int64_t mx, int64_t my, int64_t k, size_t* bytes_host);
/* The role split the kernel's planner picks when `npairs` CTA pairs are resident (74 on a B200): plan_host[0..5] =
 * row pairs per chunk, column pairs per pass, X-holder pairs, Y-holder pairs, producer pairs, column groups of the
 * X-holders.  flags bit 0: x must stay in one chunk; bit 1: column groups allowed (fp32 out_x).  Host arithmetic only. */
int pgica_softmax_grad_gemm_dual_plan(int64_t mx, int64_t my, int64_t k, int npairs, int flags, int32_t* plan_host);
int pgica_softmax_grad_gemm_dual(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale,
                                 const float* r_lse, const float* r_coef, const int32_t* r_tgt, const float* c_lse,
                                 const float* c_coef, const int32_t* c_tgt, void* out_x, int out_x_is_bf16,
                                 void* out_y, int out_y_is_bf16, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dual softmax-gradient GEMM that PUBLISHES ITS PROGRESS on out_y, so that the data-parallel all-reduce of the LM-head
 * weight gradient (SURVEY 8(e); what DDP's bucket reducer does for the reference, pkg/training/trainer.py:201,492,616)
 * can run over NVLink while the tensor cores are still computing the rest of the vocabulary.  out_y rows are cut into
 * segments of rows_per_segment (a multiple of 256); whenever a drain warp has seen the TMA stores of a final out_y tile
 * complete it adds 1 to progress[segment] with release semantics at GPU scope (the consumer runs on this GPU and
 * relays to its peers).  A full segment has received
 * (*increments_per_256_rows_host) * rows_per_segment / 256 increments (fewer for the ragged last one: count whole
 * 256-row pairs of ceil(my / 256)); the counters only ever grow — the caller compares against a per-launch target.
 * pgica_peer_allreduce_progress below is the consumer.  out_y is fp32 and x must fit one chunk of the kernel.
 * ---------------------------------------------------------------------------------------------- */
int pgica_softmax_grad_gemm_dual_progress(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale,
                                          const float* r_lse, const float* r_coef, const int32_t* r_tgt,
                                          const float* c_lse, const float* c_coef, const int32_t* c_tgt, void* out_x,
                                          int out_x_is_bf16, void* out_y, int out_y_is_bf16, uint32_t* progress,
                                          int64_t rows_per_segment, int32_t* increments_per_256_rows_host,
                                          void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sum-all-reduce of ONE fp32 buffer that lives at the same offset in the (peer-mapped, e.g. torch symmetric) memory of
 * every GPU of an NVLink node, segment by segment, each segment as soon as every rank's producer kernel has finished
 * it — a small kernel that runs BESIDE the producer (256 threads and a few dozen registers per CTA, no shared
 * memory: it fits on the SMs the persistent dual kernel occupies):
 *
 *   for each segment s:  wait until progress[s] >= progress_target_host[s]          (local producer done; NULL: skip)
 *                        flag barrier with the other ranks over peer memory            (every rank's segment s is final)
 *                        owner rank r sums ITS 1/world slice of the segment from all `world` buffers (16-byte loads
 *                        over NVLink, fixed rank order: deterministic, identical on every rank) and stores the result
 *                        into all `world` buffers
 *   final flag barrier (every owner's stores have landed everywhere)
 *
 * bufs_host[r] / flags_host[r]: rank r's buffer / flag area as mapped into THIS process (HOST arrays of `world`
 * device pointers; world <= 16).  flags: >= 4 * world * (nseg + 1) bytes per rank, zeroed once before first use.
 * seg_begin_host[0..nseg]: segment boundaries in ELEMENTS, multiples of 4 * world.  epoch: 1, 2, 3, ... for successive
 * calls on the same flags.  local_sync: 8 bytes of device scratch of this rank, zeroed once.  max_ctas: grid size
 * (0 = one CTA per SM; the same value for every call on one local_sync).  With progress != NULL the launch is preceded,
 * on `stream`, by a cuStreamWaitValue32 on progress[0]: the kernel only becomes resident once the producer's grid is
 * (its CTAs spin, and must not take SM resources a cooperative producer still needs to become resident).  `stream` must
 * therefore not be the stream the producer was launched on.  Replaces the NCCL all-reduce after the backward
 * (distributed.allreduce_dweight).
 * multicast_buf: the same buffer through an NVSwitch multicast mapping of all `world` GPUs (NVLS; e.g. torch symmetric
 * memory's multicast_ptr plus the buffer's offset), or NULL.  When given, the owner's sum is one multimem.ld_reduce
 * (added inside the switch; the order of the fp32 additions is the switch's) and its result one multimem.st to every
 * rank — a world-th of the SM work, which matters because the SMs are shared with the producer.
 * ---------------------------------------------------------------------------------------------- */
int pgica_peer_allreduce_progress(const void* const* bufs_host, const void* const* flags_host, void* multicast_buf,
                                  int world, int rank, const uint32_t* progress, const uint32_t* progress_target_host,
                                  const int64_t* seg_begin_host, int nseg, uint32_t epoch, uint32_t* local_sync,
                                  int max_ctas, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stage-2 head, hidden-state level (logits never materialised).
 *
 * pgica_lmhead_logprob_fwd: for nseq sequences of seqlen positions, hidden bf16 [nseq*seqlen][d], weight bf16
 *   [vocab][d] (tied wte / lm_head), labels int64 [nseq][seqlen], mask [nseq][seqlen] of kind `mask_kind`:
 *     seq_logp[b] = sum_{t<seqlen-1} mask[b][t+1] * log softmax(W h[b][t])[labels[b][t+1]]
 *   divided by sum_t mask[b][t+1] when length_normalize != 0.
 *   length_normalize = 0 is compute_sequence_logprobs (pkg/models/components.py:321-362) on
 *   lm_head(hidden) (modeling_gpt2.py:706); = 1 is PreferenceLoss._compute_log_probs
 *   (pkg/models/model.py:1052-1085).  Also returns, per row r = b*seqlen + t: lse[r], ztgt[r] (target logit),
 *   row_label[r] (int32, -1 where nothing is scored) and row_weight[r] — the plumbing the backward reuses —
 *   and, if nll_sum != NULL, sum over all scored positions of -log p (numerator of the HF causal-LM loss,
 *   transformers loss_utils.py:45-67 as reached from pkg/models/model.py:604-610).
 * pgica_lmhead_logprob_bwd: given grad_seq[b] = dLoss/dseq_logp[b], writes dhidden [nseq*seqlen][d] and/or
 *   dweight [vocab][d] (each may be NULL).
 * workspace: pgica_lmhead_logprob_workspace_bytes() bytes, scratch only.
 * ---------------------------------------------------------------------------------------------- */
int pgica_lmhead_logprob_workspace_bytes(int64_t nseq, int64_t seqlen, int64_t d, int64_t vocab, size_t* bytes_host);
int pgica_lmhead_logprob_fwd(const void* hidden, const void* weight, const int64_t* labels, const void* mask,
                             int mask_kind, int64_t nseq, int64_t seqlen, int64_t d, int64_t vocab,
                             int length_normalize, float* seq_logp, float* lse, float* ztgt, int32_t* row_label,
                             float* row_weight, float* nll_sum, void* workspace, size_t workspace_bytes,
                             void* stream);
int pgica_lmhead_logprob_bwd(const void* hidden, const void* weight, const int32_t* row_label,
                             const float* row_weight, const float* lse, const float* grad_seq, int64_t nseq,
                             int64_t seqlen, int64_t d, int64_t vocab, int length_normalize, void* dhidden,
                             int dhidden_is_bf16, void* dweight, int dweight_is_bf16, void* workspace,
                             size_t workspace_bytes, void* stream);
/* pgica_lmhead_logprob_bwd through pgica_softmax_grad_gemm_dual_progress: dweight (fp32, typically inside a symmetric
 * buffer) is written locally and its progress published for pgica_peer_allreduce_progress. */
int pgica_lmhead_logprob_bwd_progress(const void* hidden, const void* weight, const int32_t* row_label,
                                      const float* row_weight, const float* lse, const float* grad_seq, int64_t nseq,
                                      int64_t seqlen, int64_t d, int64_t vocab, int length_normalize, void* dhidden,
                                      int dhidden_is_bf16, void* dweight, uint32_t* progress, int64_t rows_per_segment,
                                      int32_t* increments_per_256_rows_host, void* workspace, size_t workspace_bytes,
                                      void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stage-2 head on COMPACTED rows.  Rows whose mask weight is zero, and the never-scored last position of every
 * sequence, add nothing to the loss or to any gradient (log_probs * mask, pkg/models/model.py:1081-1083,
 * pkg/models/components.py:355-358; closed form SURVEY.md Appendix A), and with the reference's tokenisation
 * (padding="max_length", 128 positions, 10-20 real tokens, pkg/data/preprocessing.py:223-231) they are > 80 % of a real
 * batch.  The caller builds the list of scored rows, gathers them into a dense bf16 [n][d] matrix (one or more
 * sequence sets, e.g. preferred ++ rejected, may share the matrix), runs pgica_gemm_lse on it for the forward and
 * pgica_lmhead_rows_bwd for both gradients, and scatters the per-row results back:
 *
 *   pgica_compact_rows      index[0..count) = ascending rows r with row_weight[r] != 0 (NaN counts as scored, so an
 *                           unmasked out-of-vocabulary label still poisons its sequence); count is a DEVICE int32 —
 *                           the one value the host has to read to size the launches that follow.
 *   pgica_gather_rows_bf16  dst[i][:] = bf16(src[index[i]][:]) (src fp32 or bf16; d % 8 == 0), and, when label_in !=
 *                           NULL, label_out[i] = label_in[index[i]].
 *   pgica_gather_u32        dst[i] = src[index[i]] for 4-byte elements (the per-row backward coefficients).
 *   pgica_scatter_u32       dst[0..dst_n) = 0, then dst[index[i]] = src[i] (lse / target logit back to [nseq*seqlen]).
 *   pgica_scatter_rows      dst[0..dst_rows)[:] = 0, then dst[index[i]][:] = src[i][:] (dhidden back in place, in the
 *                           caller's dtype): masked rows get the exact zero gradient the reference gives them.
 *   pgica_lmhead_rows_bwd   dhidden[n][d] and/or dweight[vocab][d] from prepared per-row statistics: lse[i],
 *                           ncoef[i] = -dLoss/dlogp_i, row_label[i]; dZ = ncoef * (softmax - onehot).  The dual
 *                           kernel when both are wanted and d % 512 == 0, else one launch per product.  Workspace:
 *                           pgica_lmhead_rows_workspace_bytes().
 * ---------------------------------------------------------------------------------------------- */
int pgica_compact_rows(const float* row_weight, int64_t rows, int32_t* index, int32_t* count, void* stream);
int pgica_gather_rows_bf16(const void* src, int src_is_bf16, const int32_t* index, int64_t n, int64_t d,
                           void* dst_bf16, const int32_t* label_in, int32_t* label_out, void* stream);
int pgica_gather_u32(const void* src, const int32_t* index, int64_t n, void* dst, void* stream);
int pgica_scatter_u32(const void* src, const int32_t* index, int64_t n, void* dst, int64_t dst_n, void* stream);
int pgica_scatter_rows(const void* src, int src_is_bf16, const int32_t* index, int64_t n, int64_t d, void* dst,
                       int dst_is_bf16, int64_t dst_rows, void* stream);
int pgica_lmhead_rows_workspace_bytes(int64_t rows, int64_t d, int64_t vocab, size_t* bytes_host);
int pgica_lmhead_rows_bwd(const void* hidden, const void* weight, const int32_t* row_label, const float* lse,
                          const float* ncoef, int64_t rows, int64_t d, int64_t vocab, void* dhidden,
                          int dhidden_is_bf16, void* dweight, int dweight_is_bf16, void* workspace,
                          size_t workspace_bytes, void* stream);

/* DPOPreferenceLoss.forward (pkg/models/components.py:192-249) and the tail of PreferenceLoss.forward
 * (pkg/models/model.py:1046-1048) on n local pairs of an n_global-pair batch (n_global = n on one GPU):
 *   x = beta*((pc-pr) - (rc-rr)),  loss = sum(-logsigmoid(x))/n_global  (label smoothing: cDPO form)
 *   metrics[5] = {dpo_loss, reward_margin, reward_accuracy, policy_chosen_logprob, policy_rejected_logprob}
 *   (local sums / n_global), dpc[i] = dloss/dpc[i]  (= -dloss/dpr = -dloss/drc = dloss/drr).
 * rc = rr = NULL means reference-free.  All buffers fp32 on the device. */
int pgica_dpo_loss_fwd(const float* pc, const float* pr, const float* rc, const float* rr, int64_t n,
                       int64_t n_global, float beta, float label_smoothing, float* loss, float* metrics, float* dpc,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stage-1 head: symmetric NT-Xent on a (rows_a x rows_b) slice of the similarity matrix; positives are
 * (i, i + diag_offset).  a: bf16 [rows_a][dim], b: bf16 [rows_b][dim], inv_tau = 1/temperature.
 *   fwd: lse_row[i] = logsumexp_j S[i][j], diag[i] = S[i][i+diag_offset], lse_col_part[j] = logsumexp_i S[i][j]
 *        (complete when rows_a == rows_b; one rank's partial otherwise — merge with pgica_lse_combine).
 *   bwd: da = dS b / tau, db = dS^T a / tau with dS = grad_loss[0]*grad_mult*(P_row + P_col - 2 I)
 *        (grad_mult = 1/(2 B_global) for reduction "mean", 1/2 for "sum").
 * Replaces pkg/models/model.py:970-1000 and pkg/models/components.py:117-145 (and their autograd).
 * ---------------------------------------------------------------------------------------------- */
int pgica_ntxent_workspace_bytes(int64_t rows_a, int64_t rows_b, int64_t dim, size_t* bytes_host);
int pgica_ntxent_fwd(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                     int64_t diag_offset, float* lse_row, float* diag, float* lse_col_part, void* workspace,
                     size_t workspace_bytes, void* stream);
/* The same from ONE pass over the similarity tiles (pgica_gemm_lse_rowcol) for callers that guarantee unit-norm rows
 * (|<a_i, b_j>| <= 1); falls back to the two-pass form by itself when inv_tau is too large for the bounded scheme. */
int pgica_ntxent_fwd_bounded(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                             int64_t diag_offset, float* lse_row, float* diag, float* lse_col_part, void* workspace,
                             size_t workspace_bytes, void* stream);
int pgica_ntxent_bwd(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                     int64_t diag_offset, const float* lse_row, const float* lse_col, const float* grad_loss,
                     float grad_mult, void* da, int da_is_bf16, void* db, int db_is_bf16, void* workspace,
                     size_t workspace_bytes, void* stream);
/* The same for unit-norm rows: the dual backward kernel then takes ONE exponential per element for both softmax terms
 * (2^(z c - c) times a per-row and a per-column factor); falls back like pgica_ntxent_fwd_bounded. */
int pgica_ntxent_bwd_bounded(const void* a, const void* b, int64_t rows_a, int64_t rows_b, int64_t dim, float inv_tau,
                             int64_t diag_offset, const float* lse_row, const float* lse_col, const float* grad_loss,
                             float grad_mult, void* da, int da_is_bf16, void* db, int db_is_bf16, void* workspace,
                             size_t workspace_bytes, void* stream);
/* loss = 0.5 * inv_denom * sum_i [(lse_row[i]-diag[i]) + (lse_col_owned[i]-diag[i])]   (model.py:994-998) */
int pgica_ntxent_loss(const float* lse_row, const float* diag, const float* lse_col_owned, int64_t n,
                      float inv_denom, float* loss, void* stream);
/* out[j] = log sum_r exp(parts[r][j]), parts fp32 [nparts][n] (column statistics gathered from all ranks) */
int pgica_lse_combine(const float* parts, int64_t nparts, int64_t n, float* out, void* stream);
int pgica_ntxent_coef(const float* grad, float mult, int64_t n, int64_t tgt_offset, int64_t tgt_limit, float* coef,
                      int32_t* tgt, void* stream);

/* F.normalize(x, p=2, dim=-1) (pkg/models/components.py:74-75, pkg/models/model.py:828-829) and its backward
 * dx = (g - xh <xh, g>) / max(||x||, eps).  y is bf16 (the tensor-core operand); x fp32 or bf16; dx fp32.
 * left3 / right3 (optional, both or neither; bf16 [rows][3*dim]) receive the two-term split of the unit rows,
 * [hi|lo|hi] and [hi|hi|lo], so that <left3_i, right3_j> = a_hi.b_hi + a_lo.b_hi + a_hi.b_lo: the forward
 * similarity at ~fp32 accuracy from a single bf16 tensor-core GEMM of depth 3*dim. */
int pgica_rownorm_fwd(const void* x, int x_is_bf16, int64_t rows, int64_t dim, float eps, void* y_bf16,
                      float* inv_norm, void* left3_bf16, void* right3_bf16, void* stream);
/* g: [rows][g_pitch]; the upstream gradient is g[:, 0:dim], plus g[:, g_second:g_second+dim] when g_second >= 0
 * (the two column blocks that a softmax-gradient GEMM over the split operand [hi|hi|lo] yields for hi and lo). */
int pgica_rownorm_bwd(const void* x, int x_is_bf16, const float* inv_norm, const void* g, int g_is_bf16, int64_t rows,
                      int64_t dim, int64_t g_pitch, int64_t g_second, float* dx, void* stream);
int pgica_cast_f32_to_bf16(const float* x, int64_t n, void* y_bf16, void* stream);
/* The same two-term split WITHOUT normalising (inputs used as given, pkg/models/model.py:988): fp32 embeddings that
 * are not bf16-representable keep ~fp32 accuracy in the similarity.  left3 / right3: bf16 [rows][3*dim]. */
int pgica_split3_bf16(const float* x, int64_t rows, int64_t dim, void* left3_bf16, void* right3_bf16, void* stream);

/* dst[i] += sum_s srcs[s][i], fp32, n elements (n % 4 == 0, 16-byte aligned pointers), n_src <= 15 sources given as a
 * HOST array of device pointers.  The reduction step of the copy-engine all-reduce of the LM-head weight gradient
 * (distributed.PeerAllReduce: chunks pulled from the peers over NVLink, summed here, pushed back); what DDP's
 * bucket all-reduce does for the reference (pkg/training/trainer.py:201,492,616).  max_ctas bounds the grid so the
 * kernel fits beside a resident persistent kernel (0 = one CTA per SM).  HBM-bound: (n_src + 2) * 4 bytes / element. */
int pgica_sum_into_f32(float* dst, const void* const* srcs_host, int n_src, int64_t n, int max_ctas, void* stream);

/* Plumbing pieces of the Stage-2 head, exported so the parity tests can pin them bit-exactly:
 * shift / label / mask layout (components.py:339-344), per-sequence masked sum (components.py:355-360,
 * model.py:1082-1083), per-row backward coefficients. */
int pgica_prep_rows(const int64_t* labels, const void* mask, int mask_kind, int64_t nseq, int64_t seqlen,
                    int64_t vocab, int32_t* row_label, float* row_weight, void* stream);
int pgica_seq_reduce(const float* lse, const float* ztgt, const float* row_weight, int64_t nseq, int64_t seqlen,
                     int length_normalize, float* seq_logp, float* nll_sum, void* stream);
int pgica_row_coef(const float* grad_seq, const float* row_weight, int64_t nseq, int64_t seqlen, int length_normalize,
                   float sign, float* coef, void* stream);
int pgica_scale_by_scalar(const float* a, const float* scalar, float mult, int64_t n, float* out, void* stream);

/* Materialised-logits path (strict signature compatibility with PreferenceLoss.forward /
 * compute_sequence_logprobs, which receive (nseq, seqlen, vocab) logits): streaming log-sum-exp + gather, and
 * dlogits = coef * (onehot - softmax).  HBM-bound; logits fp32 or bf16. */
int pgica_logits_lse(const void* logits, int logits_is_bf16, const int32_t* row_label, int64_t nseq, int64_t seqlen,
                     int64_t vocab, float* lse, float* ztgt, void* stream);
int pgica_logits_grad(const void* logits, int logits_is_bf16, const int32_t* row_label, const float* lse,
                      const float* coef, int64_t nseq, int64_t seqlen, int64_t vocab, void* dlogits, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stage-1 head at small batch (B <= 128, D in {128, 256, 384, 512}): the whole symmetric NT-Xent of
 * pkg/models/model.py:970-1000 — similarity, both log-sum-exps, loss (mean when reduce_mean != 0, else sum; both
 * halved) AND the gradients of that loss w.r.t. a and b — in ONE launch of one CTA (ntxent_small.cu).  The trainer's
 * default batch is 8 (configs/default.yaml:35), BASELINE config 1 is 64: at these sizes the head is launch latency.
 * a, b: bf16 [rows][dim], used as given.  da, db: fp32 [rows][dim], 16-byte aligned, gradients for upstream gradient 1.
 * ---------------------------------------------------------------------------------------------- */
int pgica_ntxent_small_supported(int64_t rows, int64_t dim);
int pgica_ntxent_small(const void* a, const void* b, int64_t rows, int64_t dim, float inv_tau, int reduce_mean,
                       float* loss, float* lse_row, float* lse_col, float* da, float* db, void* stream);
/* Same launch for fp32 embeddings given as their bf16 splits (pgica_split3_bf16 / pgica_rownorm_fwd): a_left3 =
 * [hi|lo|hi], b_right3 = [hi|hi|lo], bf16 [rows][3*dim].  The similarity runs over depth 3*dim (fp32-level accuracy in
 * the loss, pkg/models/model.py:988 computes it in fp32); the gradient products use the hi parts.  da, db: [rows][dim]. */
int pgica_ntxent_small_split(const void* a_left3, const void* b_right3, int64_t rows, int64_t dim, float inv_tau,
                             int reduce_mean, float* loss, float* lse_row, float* lse_col, float* da, float* db,
                             void* stream);

/* ------------------------------------------------------------------------------------------------
 * SURVEY 8(f) row 2 — finite-check + global L2 gradient norm + clip over ALL gradient tensors at once:
 * NaNSafeGradientNorm.forward (pkg/models/components.py:283-318) and the per-parameter isfinite() scan +
 * clip_grad_norm_ of the trainer (pkg/training/trainer.py:494-515, 619-628).
 *   grads_host[i]: device pointer of gradient i (fp32, or bf16 when is_bf16_host[i] != 0), numels_host[i] elements;
 *   stats (device, 3 floats): total_norm, clip_coef = min(1, max_norm / (total_norm + 1e-6)), is_finite (1 / 0).
 *   clip bit 0: gradients are multiplied by clip_coef in place when the norm is finite and clip_coef < 1 (a non-finite
 *   norm leaves them untouched, like the reference).  clip bit 1: the chunk table the previous call uploaded into
 *   this very workspace for these very tensors is still there (skips a host->device copy per step).
 *   Three launches, no host synchronisation; deterministic.
 * workspace: pgica_grad_norm_clip_workspace_bytes() bytes (chunk table + per-chunk partial sums).
 * ---------------------------------------------------------------------------------------------- */
int pgica_grad_norm_clip_workspace_bytes(const int64_t* numels_host, int n_tensors, size_t* bytes_host);
int pgica_grad_norm_clip(const void* const* grads_host, const int64_t* numels_host, const int32_t* is_bf16_host,
                         int n_tensors, float max_norm, int clip, float* stats, void* workspace,
                         size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SURVEY 8(f) row 2, the optimizer step that follows the clip (pkg/training/trainer.py:494-520, 619-633:
 * torch.optim.AdamW after clip_grad_norm_) — AdamW over ALL tensors of a parameter group in one launch, element for
 * element torch/optim/adam.py::_single_tensor_adam with decoupled weight decay (s = the stored step):
 *   p *= 1 - lr*wd;  m = lerp(m, g, 1 - beta1);  v = beta2*v + (1 - beta2)*g^2;
 *   p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps),  bc1 = 1 - beta1^(s+1),  bc2 = 1 - beta2^(s+1)
 * The per-tensor scalars are computed in double and rounded once to fp32; the arithmetic is fp32.
 *   params_host[i], grads_host[i], exp_avgs_host[i], exp_avg_sqs_host[i]: device pointers of contiguous fp32 tensors of
 *   numels_host[i] < 2^31 elements (any 4-byte alignment); steps_host[i]: device pointer of tensor i's fp32 step
 *   counter, read by the update and incremented by a second launch after it.
 *   grad_stats: NULL, or the 3 floats pgica_grad_norm_clip writes (clip = 0 computes them without touching the
 *   gradients).  With grad_stats, a non-finite norm (grad_stats[2] == 0) writes nothing — no p, m, v or step — and a
 *   finite one runs the update on g * grad_stats[1] (one fp32 multiply: bit for bit what clipping the gradients in
 *   place first gives).  The gradients in memory are never written.
 *   Two launches, no host synchronisation; the tensor table (one entry per tensor) is uploaded on every call.
 * workspace: pgica_adamw_workspace_bytes() bytes.
 * ---------------------------------------------------------------------------------------------- */
int pgica_adamw_workspace_bytes(int n_tensors, size_t* bytes_host);
int pgica_adamw_step(void* const* params_host, const void* const* grads_host, void* const* exp_avgs_host,
                     void* const* exp_avg_sqs_host, float* const* steps_host, const int64_t* numels_host,
                     int n_tensors, double lr, double beta1, double beta2, double eps, double weight_decay,
                     const float* grad_stats, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SURVEY 8(f) row 4 — the caption decoder's cross-attention over ONE key/value token (pkg/models/model.py:528-535,
 * 594-601: nn.MultiheadAttention(query = token embeddings, key = value = the projected image) followed by
 * attention_norm(text + attended)).  With a single key the softmax is identically 1, so
 *     y[b,t,:] = LayerNorm(x[b,t,:] + out_bias + sum_h w[b,t,h] * u[b,h,:]),   u[b,h,:] = W_o[:, head h] v_h[b]
 * where w is NULL (all ones: evaluation; pass heads = 1 and the head-summed u) or the attention-dropout weights
 * keep[b,t,h] / (1 - p) in training.  x, y, dx: fp32 [batch][seqlen][dim]; u, du: [batch][heads][dim]; w:
 * [batch][seqlen][heads]; mean, rstd: [batch*seqlen].  The backward owns one sequence per block (deterministic) and
 * returns per-sequence partials [batch][dim] of dgamma, dbeta and sum_t dpre (= d out_bias) for the caller to add up.
 * HBM-bound: x read and y written once forward; dy, x read and dx written once backward.
 * ---------------------------------------------------------------------------------------------- */
int pgica_xattn_ln_fwd(const float* x, const float* u, const float* w, const float* out_bias, const float* gamma,
                       const float* beta, int64_t batch, int64_t seqlen, int64_t dim, int64_t heads, float eps, float* y,
                       float* mean, float* rstd, void* stream);
int pgica_xattn_ln_bwd(const float* dy, const float* x, const float* u, const float* w, const float* out_bias,
                       const float* gamma, const float* mean, const float* rstd, int64_t batch, int64_t seqlen,
                       int64_t dim, int64_t heads, float* dx, float* du, float* dgamma_part, float* dbeta_part,
                       float* dpre_sum_part, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SURVEY 8(f) row 3 — tail of the projection heads that feed the contrastive head (pkg/models/model.py:136-142,
 * 338-344: ... Linear -> LayerNorm; :826-829: F.normalize): e = LayerNorm(z) (the model also hands it to the decoder),
 * n = e / max(||e||, eps_norm) (the NT-Xent operand), one launch; the backward takes the gradients of both outputs
 * (either may be NULL).  stats: [rows][3] = mean, rstd, 1/max(||e||, eps).  dgamma_part / dbeta_part: one row of
 * `dim` floats per block of 8 input rows (ceil(rows / 8) rows), summed by the caller.
 * ---------------------------------------------------------------------------------------------- */
int pgica_ln_l2norm_fwd(const float* z, const float* gamma, const float* beta, int64_t rows, int64_t dim, float eps_ln,
                        float eps_norm, float* e, float* n, float* stats, void* stream);
int pgica_ln_l2norm_bwd(const float* z, const float* gamma, const float* beta, const float* stats, const float* de,
                        const float* dn, int64_t rows, int64_t dim, float* dz, float* dgamma_part, float* dbeta_part,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PGICA_H_ */
