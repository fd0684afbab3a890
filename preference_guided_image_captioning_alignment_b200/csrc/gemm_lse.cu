// K1/K3: z = scale * A B^T on tcgen05 tensor cores with the softmax statistics taken straight out of
// TMEM — running max / sum-of-exp per row and the target logit — so the (rows x cols) logit matrix is
// never written anywhere.  Persistent CTA PAIRS (2-CTA clusters, tcgen05 cta_group::2): a pair owns a 256-row x
// 256-column tile, CTA rho holds the accumulator of row block 2mp + rho and loads only ITS half of the B tile —
// 32 KB per k-step and SM instead of 48 KB, which is what the tensor pipe was waiting for in the single-CTA form
// (shared-memory fill + operand reads exceeded the SM's shared-memory bandwidth).  Warp-specialised:
//   warp 0      TMA producer (A tile 128x64, B half tile 128x64 per k-step, SWIZZLE_128B, 6-stage ring; completion
//               bytes of both CTAs are credited to the leader's barrier)
//   warp 1      tcgen05.mma issuer (one elected thread of the LEADER CTA), M = 256, N = 256; accumulators 128x256 fp32
//               per CTA, double-buffered in TMEM; commits multicast to both CTAs' barriers
//   warp 2      TMEM allocator
//   warps 4..7  epilogue (each CTA its own 128 rows): tcgen05.ld 32 columns at a time, online log-sum-exp in the
//               log2 domain
// Tiles are linearised column-tile-major (all row-block pairs of column tile 0, then of column tile 1, ...) and dealt
// round-robin to the persistent pairs, so at any moment the whole grid works on the same four or five B tiles:
// B (the 103 MB LM-head weight) is then read from HBM once instead of once per row block.  Every tile writes its
// rows' (max, sum, target) as a partial; lse_merge_kernel folds the column tiles of a row (deterministic, no atomics).
#include <algorithm>

#include "common.h"
#include "ptx.cuh"

namespace pgica {

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockN = 256;
constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
constexpr int kStages = 7;
constexpr int kAccStages = 2;
constexpr uint32_t kABytes = kBlockM * kBlockK * 2;
constexpr uint32_t kBBytes = (kBlockN / 2) * kBlockK * 2;  // this CTA's half of the B tile
// Epilogue: 8 warps = 2 per scheduler (a lone warp leaves its scheduler idle on every dependent FFMA / MUFU / shuffle; the
// dual backward kernel's ncu stall samples showed 0.31 instructions per cycle with one).  Warp w reads TMEM lane quarter
// w & 3 and column group (w - 4) >> 2 of the tile: each group publishes its own (max, sum, target) partial.
// The one-pass NT-Xent forward (kCols: two exponentials per element and a butterfly sum) is epilogue-bound and takes two
// groups; the plain forward (the LM head at k = 1024: tensor-bound, 0.94 of peak) keeps one — a second group doubles the
// partials lse_merge_kernel has to fold, +1 % on that launch.
constexpr int kMaxEpiGroups = 2;
constexpr int epi_groups(bool cols) { return cols ? 2 : 1; }
constexpr int block_threads(bool cols) { return 128 + 128 * epi_groups(cols); }
constexpr int kEpilogueWarp0 = 4;
constexpr float kLn2 = 0.6931471805599453f;

struct GemmLseParams {
  int rows, cols, k;
  int num_m_blocks, num_m_pairs, num_n_tiles, rows_pad;
  int num_parts;    // num_n_tiles * column groups of the launched kernel
  float scale;
  const int* labels;
  int diag_offset;
  float* part_max;  // [num_parts][rows_pad]  max of scale*log2e*z over the columns of a tile's group
  float* part_sum;  // [..][rows_pad]  sum of exp2(. - max);  max = -inf, sum = 0 when the group lies past the last column
  float* part_tgt;  // [..][rows_pad]  scale*z at the label column, -inf if it is not among these columns
  float* z_out;     // optional dense [rows][cols] copy of scale*z (similarity-matrix API only)
  // optional COLUMN statistics from the same tiles (NT-Xent with bounded logits: S is computed once instead of twice).
  // Every warp of the epilogue owns 32 rows; per 32-column chunk it publishes the column sums of exp2(t - shift) over
  // its rows (col_sum[group][column]) and the shift it used (col_shift[group][tile * 8 + chunk] = the largest running
  // row maximum among its rows).  col_merge_kernel folds the groups of a column.
  float* col_sum;   // [rows_pad / 32][cols_pad]
  float* col_shift; // [rows_pad / 32][num_n_tiles * 8]
  int cols_pad;
};

// What the epilogue warps do with a tile.  The two retrieval-rank passes run the same tiles in the same k-order as each
// other, so a positive's score found in the first pass is bit-identical to the value the second pass compares with.
enum TileEpilogue : int {
  kEpiLse = 0,        // online log-sum-exp + target gather (pgica_gemm_lse, pgica_similarity)
  kEpiLseCols = 1,    // the same plus the column statistics (pgica_gemm_lse_rowcol)
  kEpiPositives = 2,  // retrieval pass 1: only tiles holding a (owner[j], j) pair; publishes p (rows) and q (columns)
  kEpiRanks = 3,      // retrieval pass 2: every tile; counts scores above p along rows and above q along columns
};

// Retrieval ranks (pgica_retrieval_ranks).  Rows are images, columns captions; caption j belongs to row owner(j).
struct RankParams {
  const int32_t* col_owner;  // [cols] owner of each column; NULL = column j belongs to row j (j < rows).  Entries outside
                             // [0, rows) own nothing.
  uint8_t* tile_mask;        // [num_n_tiles * num_m_pairs], indexed like the tile walk: 1 = the tile holds a positive
  uint32_t* pos_key;         // [rows] p of the row as an order-preserving key (pos_key_of); 0 = the row owns no column
  float* pos_col;            // [cols] q of the column; NaN when it has no owner (a NaN threshold counts nothing)
  int32_t* row_rank;         // [rows] outputs
  int32_t* col_rank;         // [cols]
};

// Order-preserving uint32 key of an fp32 score for atomicMax: -inf < ... < -0 < +0 < ... < +inf < NaN, and 0 below all
// of them, so a row's maximum over several tiles (and pair CTAs) is one integer max that propagates NaN.
__device__ __forceinline__ uint32_t pos_key_of(float v) {
  const uint32_t u = __float_as_uint(v);
  return v != v ? 0xFFFFFFFFu : ((u & 0x80000000u) ? ~u : (u | 0x80000000u));
}
__device__ __forceinline__ float pos_value(uint32_t key) {  // key 0 (no positive) decodes to NaN: nothing counts
  return key == 0xFFFFFFFFu ? NAN : __uint_as_float((key & 0x80000000u) ? (key & 0x7FFFFFFFu) : ~key);
}
__device__ __forceinline__ int col_owner_of(const RankParams& r, int rows, int col) {
  const int o = r.col_owner ? r.col_owner[col] : (col < rows ? col : -1);
  return (o >= 0 && o < rows) ? o : -1;
}

__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

constexpr size_t kSmemBytes = 1024 /*align slack*/ + kStages * (kABytes + kBBytes) + 256 /*barriers*/;

template <bool kPositives>
__device__ __forceinline__ void rank_epilogue(const GemmLseParams& p, const RankParams& r, int warp, int lane, uint32_t rho,
                                              uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar, int t_begin,
                                              int t_step, int t_end);

// The tile pipeline of every kernel in this file: barrier and TMEM set-up, the TMA producers, the MMA issuer, the
// epilogue selected by kMode, teardown.  In kEpiPositives every role skips the tiles tile_mask leaves out before any TMA
// or MMA, so their ring and accumulator phases stay in step.
template <int kMode>
__device__ __forceinline__ void gemm_tiles(const CUtensorMap& tm_a, const CUtensorMap& tm_b, const GemmLseParams p,
                                           const RankParams r) {
  constexpr bool kCols = kMode == kEpiLseCols;
  constexpr int kEpiGroups = epi_groups(kMode != kEpiLse);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * kABytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * (kABytes + kBBytes));
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + kAccStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rho = cluster_ctarank();  // 0 = leader of the pair
  const int total_tiles = p.num_m_pairs * p.num_n_tiles;
  const int t_begin = (int)blockIdx.x >> 1, t_step = (int)gridDim.x >> 1, t_end = total_tiles;
  const int num_kb = (p.k + kBlockK - 1) / kBlockK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < kAccStages; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 2 * 128 * kEpiGroups);  // leader's: the epilogue threads of both CTAs
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kAccStages * kBlockN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 || warp == 2) {
    // TMA producers: two warps, one per stage parity (a single warp's wait + expect_tx + two TMA issues per stage take
    // most of the time the tensor pipe needs to consume a stage); each whole warp walks the tile schedule, one
    // elected lane issues the copies
    const int par = warp >> 1;
    int stage = 0;
    uint32_t phase = 0, stage_no = 0;
    const uint32_t lbar0 = mapa_u32(smem_u32(&full_bar[0]), 0);  // the leader's full barriers (shared::cluster)
    for (int t = t_begin; t < t_end; t += t_step) {
      if constexpr (kMode == kEpiPositives) {
        if (!r.tile_mask[t]) continue;
      }
      const int n_tile = t / p.num_m_pairs;
      const int m_blk = 2 * (t - n_tile * p.num_m_pairs) + (int)rho;
      for (int kb = 0; kb < num_kb; ++kb, ++stage_no) {
        if ((int)(stage_no & 1u) == par) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            if (rho == 0) mbar_expect_tx(&full_bar[stage], 2 * (kABytes + kBBytes));  // both CTAs' bytes
            const uint32_t lbar = lbar0 + stage * 8;
            tma_load_2d_pair(smem_a + stage * kABytes, &tm_a, lbar, kb * kBlockK, m_blk * kBlockM);
            tma_load_2d_pair(smem_b + stage * kBBytes, &tm_b, lbar, kb * kBlockK, n_tile * kBlockN + (int)rho * (kBlockN / 2));
          }
          __syncwarp();
        }
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && rho == 0) {
    // Whole warp walks the pipeline (warp-uniform control flow keeps descriptors in uniform registers); one elected
    // lane of the leader CTA issues the tcgen05 instructions for the pair.
    constexpr uint32_t idesc = make_idesc_bf16(2 * kBlockM, kBlockN, 0, 0);
    const uint64_t desc_hi = make_smem_desc(0, 16, 1024);  // everything but the start address
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    for (int t = t_begin; t < t_end; t += t_step) {
      if constexpr (kMode == kEpiPositives) {
        if (!r.tile_mask[t]) continue;
      }
      mbar_wait_cluster(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + acc * kBlockN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait_cluster(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint64_t da = desc_hi | ((smem_u32(smem_a + stage * kABytes) >> 4) & 0x3FFF);
          const uint64_t db = desc_hi | ((smem_u32(smem_b + stage * kBBytes) >> 4) & 0x3FFF);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k)
            umma2_bf16_ss(d_tmem, da + k * (kUmmaK * 2 / 16), db + k * (kUmmaK * 2 / 16), idesc, (kb | k) != 0 ? 1u : 0u);
          umma2_commit_both(&empty_bar[stage]);
          if (kb == num_kb - 1) umma2_commit_both(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (++acc == kAccStages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp < kEpilogueWarp0) {
    // warp 1 of the second CTA, warp 3: idle
  } else if constexpr (kMode >= kEpiPositives) {
    rank_epilogue<kMode == kEpiPositives>(p, r, warp, lane, rho, tmem_base, tfull_bar, tempty_bar, t_begin, t_step, t_end);
  } else {
    const int quarter = warp & 3;  // TMEM lane quarter this warp may read
    const int wg = (warp - kEpilogueWarp0) >> 2;  // column group of the tile
    constexpr int kChunks = kBlockN / 32 / kEpiGroups;
    const int row_in_blk = quarter * 32 + lane;
    const float c = p.scale * kLog2e;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = t_begin; t < t_end; t += t_step) {
      const int n_tile = t / p.num_m_pairs;
      const int m_blk = 2 * (t - n_tile * p.num_m_pairs) + (int)rho;  // may be one past the end (odd block count)
      const int row = m_blk * kBlockM + row_in_blk;
      float run_m = -INFINITY, run_s = 0.f, run_t = -INFINITY;
      int label = -1;
      if (row < p.rows) label = p.labels ? p.labels[row] : row + p.diag_offset;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after_sync();

      const int n0 = n_tile * kBlockN;
      const bool tail = n0 + kBlockN > p.cols;
      const int rel = label - n0;  // label column relative to this tile
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * kBlockN;
#pragma unroll 1
      for (int cl = 0; cl < kChunks; ++cl) {
        const int ch = wg * kChunks + cl;
        if (tail && n0 + ch * 32 >= p.cols) break;  // warp-uniform: nothing valid from here on
        uint32_t r[32];
        tmem_ld_32x32(taddr + ch * 32, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (tail) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (n0 + ch * 32 + j >= p.cols) v[j] = -INFINITY;
        }
        if (p.z_out != nullptr) {
          if (row < p.rows) {
            float* dst = p.z_out + static_cast<size_t>(row) * p.cols + n0 + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + ch * 32 + j < p.cols) dst[j] = v[j] * p.scale;
          }
        }
        float cm = v[0];
#pragma unroll
        for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
        const float m_new = fmaxf(run_m, cm * c);
        const float corr = fast_exp2(run_m - m_new);
        float s0 = 0.f, s1 = 0.f;
        if (!kCols) {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            s0 += fast_exp2(fmaf(v[j], c, -m_new));
            s1 += fast_exp2(fmaf(v[j + 1], c, -m_new));
          }
        } else {
          // the same exponentials, kept: rescaled to the warp's common shift and summed DOWN the 32 rows of the warp
          // (butterfly: 31 shuffles, lane l ends up with the sum of column l of the chunk)
          float e[32];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            e[j] = fast_exp2(fmaf(v[j], c, -m_new));
            e[j + 1] = fast_exp2(fmaf(v[j + 1], c, -m_new));
            s0 += e[j];
            s1 += e[j + 1];
          }
          const bool rvalid = row < p.rows;
          float sh = rvalid ? m_new : -INFINITY;
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) sh = fmaxf(sh, __shfl_xor_sync(0xffffffffu, sh, o));
          const float f = rvalid ? fast_exp2(m_new - sh) : 0.f;  // <= 1; rows past the end contribute nothing
#pragma unroll
          for (int j = 0; j < 32; ++j) e[j] *= f;
#pragma unroll
          for (int o = 16; o >= 1; o >>= 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int kk = 0; kk < o; ++kk) {
              const float send = upper ? e[kk] : e[kk + o];
              const float keep = upper ? e[kk + o] : e[kk];
              e[kk] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
          }
          if (m_blk < p.num_m_blocks) {
            const size_t g = static_cast<size_t>(m_blk) * 4 + quarter;
            const int col = n0 + ch * 32 + lane;
            if (col < p.cols) p.col_sum[g * p.cols_pad + col] = e[0];
            if (lane == 0) p.col_shift[g * (static_cast<size_t>(p.num_n_tiles) * 8) + n_tile * 8 + ch] = sh;
          }
        }
        run_s = fmaf(run_s, corr, s0 + s1);
        run_m = m_new;
        if ((rel >> 5) == ch && rel >= 0) {
          const int jj = rel & 31;
          float z = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j == jj) z = v[j];
          run_t = z * p.scale;
        }
      }
      tc_fence_before_sync();
      mbar_arrive_cluster(&tempty_bar[acc], 0);  // tell the leader: this CTA has read the accumulator
      if (++acc == kAccStages) {
        acc = 0;
        acc_phase ^= 1;
      }
      if (m_blk < p.num_m_blocks) {
        const size_t o = (static_cast<size_t>(n_tile) * kEpiGroups + wg) * p.rows_pad + m_blk * kBlockM + row_in_blk;
        p.part_max[o] = run_m;
        p.part_sum[o] = run_s;
        p.part_tgt[o] = run_t;
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // the pair shares barriers and TMEM commits: nobody leaves early
  if (warp == 2)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kAccStages * kBlockN)
                 : "memory");
}

template <bool kCols>  // kCols: also publish the column statistics (a separate instantiation: the plain forward keeps its code)
__global__ void __launch_bounds__(block_threads(kCols), 1)
gemm_lse_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                const GemmLseParams p) {
  gemm_tiles<kCols ? kEpiLseCols : kEpiLse>(tm_a, tm_b, p, RankParams{});
}

// Retrieval ranks, pass 1 (kPositives) and pass 2: the same tile pipeline with the rank-counting epilogue.
template <bool kPositives>
__global__ void __launch_bounds__(block_threads(true), 1)
gemm_rank_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const GemmLseParams p, const RankParams r) {
  gemm_tiles<kPositives ? kEpiPositives : kEpiRanks>(tm_a, tm_b, p, r);
}

// Epilogue of the rank passes: 8 warps, warp w reads TMEM lane quarter w & 3 (32 rows) and column half (w - 4) >> 2.
//   pass 1: per 32-column chunk every lane holds the owner of its column; the row that owns column j keeps the running
//           max of its positives (one atomicMax of the key per tile) and stores q[j] (exactly one writer per column).
//   pass 2: rows count their scores above p in a per-thread counter over the tile's chunks; columns are counted per
//           chunk with one ballot per column (the warp's 32 rows against lane j's q) and one popc.  Both are added to the
//           int32 outputs with red.global.add: exact and order-independent.
template <bool kPositives>
__device__ __forceinline__ void rank_epilogue(const GemmLseParams& p, const RankParams& r, int warp, int lane, uint32_t rho,
                                              uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar, int t_begin,
                                              int t_step, int t_end) {
  constexpr int kChunks = kBlockN / 32 / 2;
  const int quarter = warp & 3;
  const int wg = (warp - kEpilogueWarp0) >> 2;
  const int row_in_blk = quarter * 32 + lane;
  int acc = 0;
  uint32_t acc_phase = 0;
  for (int t = t_begin; t < t_end; t += t_step) {
    if (kPositives && !r.tile_mask[t]) continue;
    const int n_tile = t / p.num_m_pairs;
    const int m_blk = 2 * (t - n_tile * p.num_m_pairs) + (int)rho;  // may be one past the end (odd block count)
    const int row = m_blk * kBlockM + row_in_blk;
    const bool rvalid = row < p.rows;
    const int n0 = n_tile * kBlockN;
    uint32_t key = 0;
    if (!kPositives && rvalid) key = r.pos_key[row];
    const float thr = pos_value(key);
    int row_count = 0;
    mbar_wait(&tfull_bar[acc], acc_phase);
    tc_fence_after_sync();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * kBlockN;
#pragma unroll 1
    for (int cl = 0; cl < kChunks; ++cl) {
      const int c0 = n0 + (wg * kChunks + cl) * 32;
      if (c0 >= p.cols) break;  // warp-uniform: nothing valid from here on
      const int col = c0 + lane;
      int own = -1;
      float q = NAN;
      if (col < p.cols) {
        if (kPositives)
          own = col_owner_of(r, p.rows, col);
        else
          q = r.pos_col[col];
      }
      uint32_t u[32];
      tmem_ld_32x32(taddr + (c0 - n0), u);
      tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(u[j]);
      if (c0 + 32 > p.cols) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (c0 + j >= p.cols) v[j] = -INFINITY;  // above no threshold
      }
      if (kPositives) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (__shfl_sync(0xffffffffu, own, j) == row) {  // own is -1 or < rows: rows past the end never match
            key = max(key, pos_key_of(v[j]));
            r.pos_col[c0 + j] = v[j];
          }
        }
      } else {
        uint32_t mine = 0;  // ballot over the warp's rows for this lane's column
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          row_count += v[j] > thr ? 1 : 0;
          const float qj = __shfl_sync(0xffffffffu, q, j);  // every lane, rows past the end included
          const uint32_t b = __ballot_sync(0xffffffffu, rvalid && v[j] > qj);
          if (lane == j) mine = b;
        }
        const int cc = __popc(mine);
        if (cc != 0) atomicAdd(&r.col_rank[col], cc);  // q is NaN past the last column: cc == 0 there
      }
    }
    tc_fence_before_sync();
    mbar_arrive_cluster(&tempty_bar[acc], 0);  // tell the leader: this CTA has read the accumulator
    if (++acc == kAccStages) {
      acc = 0;
      acc_phase ^= 1;
    }
    if (kPositives) {
      if (key != 0) atomicMax(&r.pos_key[row], key);
    } else if (rvalid) {
      if (key == 0) {
        if (n_tile == 0 && wg == 0) r.row_rank[row] = -1;  // owns no column: no tile adds to it
      } else if (row_count != 0) {
        atomicAdd(&r.row_rank[row], row_count);
      }
    }
  }
}

// Retrieval set-up, launch 1 of 2: clear the tile mask, the row keys and the row counts.
__global__ void rank_init_kernel(const GemmLseParams p, const RankParams r, int mask_bytes) {
  const int n = mask_bytes > p.rows ? mask_bytes : p.rows;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (i < mask_bytes) r.tile_mask[i] = 0;
    if (i < p.rows) {
      r.pos_key[i] = 0;
      r.row_rank[i] = 0;
    }
  }
}

// Launch 2 of 2, one thread per column: range-check the owner, mark the tile that holds (owner[j], j), clear q[j] and the
// column count (-1 for a column without an owner, which no pass touches again).
__global__ void rank_mark_kernel(const GemmLseParams p, const RankParams r) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.cols) return;
  const int o = col_owner_of(r, p.rows, j);
  r.pos_col[j] = NAN;
  r.col_rank[j] = o >= 0 ? 0 : -1;
  if (o >= 0) r.tile_mask[(j / kBlockN) * p.num_m_pairs + o / (2 * kBlockM)] = 1;
}

// Fold the column-tile partials of every row into lse (natural log) and the target logit.  A block handles 32 rows
// with 8 threads per row: thread (r, g) walks tiles g, g+8, ... (loads coalesced across r), then the 8 running
// (max, sum, target) triples of a row are combined in a fixed order through shared memory.
constexpr int kMergeRows = 32, kMergeGroups = 8;
__global__ void __launch_bounds__(kMergeRows* kMergeGroups)
lse_merge_kernel(const GemmLseParams p, float* __restrict__ lse, float* __restrict__ tgt) {
  __shared__ float s_m[kMergeGroups][kMergeRows], s_s[kMergeGroups][kMergeRows], s_t[kMergeGroups][kMergeRows];
  const int r = threadIdx.x % kMergeRows, g = threadIdx.x / kMergeRows;
  const int row = blockIdx.x * kMergeRows + r;
  float m = -INFINITY, sum = 0.f, t = -INFINITY;
  if (row < p.rows) {
    for (int s = g; s < p.num_parts; s += kMergeGroups) {
      const size_t o = static_cast<size_t>(s) * p.rows_pad + row;
      const float pm = p.part_max[o], ps = p.part_sum[o];
      if (pm == -INFINITY && ps == 0.f) continue;  // a column group past the last column; (-inf, NaN) — a NaN row, whose
                                                   // maximum fmaxf leaves at -inf — falls through and poisons the sum
      const float mn = fmaxf(m, pm);
      sum = sum * exp2f(m - mn) + ps * exp2f(pm - mn);
      m = mn;
      t = fmaxf(t, p.part_tgt[o]);
    }
  }
  s_m[g][r] = m;
  s_s[g][r] = sum;
  s_t[g][r] = t;
  __syncthreads();
  if (g == 0 && row < p.rows) {
    float M = -INFINITY;
#pragma unroll
    for (int i = 0; i < kMergeGroups; ++i) M = fmaxf(M, s_m[i][r]);
    float S = 0.f, T = -INFINITY;
    bool bad = false;
#pragma unroll
    for (int i = 0; i < kMergeGroups; ++i) {
      const float mi = s_m[i][r], si = s_s[i][r];
      bad |= (si != si) || (mi != mi);
      if (mi > -INFINITY) S += si * exp2f(mi - M);
      T = fmaxf(T, s_t[i][r]);
    }
    float out = (M + log2f(S)) * kLn2;
    if (bad) out = NAN;
    lse[row] = out;
    if (tgt) tgt[row] = (T == -INFINITY) ? 0.f : T;
  }
}

// Fold the row groups of every column: lse_col[j] = ln sum_g col_sum[g][j] * exp2(shift[g][chunk(j)])  (log2 domain in).
// One thread per column (loads coalesced across columns); groups that hold no valid row carry shift = -inf, sum = 0.
__global__ void __launch_bounds__(512) col_merge_kernel(const GemmLseParams p, int groups, float* __restrict__ lse_col) {
  // block = 32 columns x 16 group lanes: coalesced 128-byte reads of col_sum, the groups of a column folded by 16 threads
  __shared__ float sm_m[16][33], sm_s[16][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  const size_t shift_pitch = static_cast<size_t>(p.num_n_tiles) * 8;
  const int slot = blockIdx.x;  // 32 columns share a shift; kBlockN is a multiple of 32, so slot == j / 32 for every tile
  float M = -INFINITY, S = 0.f;
  if (j < p.cols) {
#pragma unroll 4
    for (int g = ty; g < groups; g += 16) {
      const float sh = p.col_shift[g * shift_pitch + slot];
      const float v = p.col_sum[static_cast<size_t>(g) * p.cols_pad + j];
      if (sh > -INFINITY) {
        if (sh > M) {
          S = S * exp2f(M - sh) + v;
          M = sh;
        } else {
          S += v * exp2f(sh - M);
        }
      }
    }
  }
  sm_m[ty][tx] = M;
  sm_s[ty][tx] = S;
  __syncthreads();
  if (ty == 0 && j < p.cols) {
    float Mx = -INFINITY;
#pragma unroll
    for (int t = 0; t < 16; ++t) Mx = fmaxf(Mx, sm_m[t][tx]);
    float Sx = 0.f;
#pragma unroll
    for (int t = 0; t < 16; ++t)
      if (sm_m[t][tx] > -INFINITY) Sx += sm_s[t][tx] * exp2f(sm_m[t][tx] - Mx);
    lse_col[j] = (Mx + log2f(Sx)) * kLn2;
  }
}

int plan(int64_t rows, int64_t cols, int64_t k, GemmLseParams* p, int* grid, size_t* ws_bytes) {
  PGICA_REQUIRE(rows > 0 && cols > 0 && k > 0, "gemm_lse: empty problem (rows %lld cols %lld k %lld)", (long long)rows,
                (long long)cols, (long long)k);
  PGICA_REQUIRE(k % 8 == 0, "gemm_lse: k (%lld) must be a multiple of 8 (16-byte row pitch for TMA)", (long long)k);
  PGICA_REQUIRE(rows < (1ll << 30) && cols < (1ll << 30), "gemm_lse: dimension too large");
  p->rows = (int)rows;
  p->cols = (int)cols;
  p->k = (int)k;
  p->num_m_blocks = (int)ceil_div(rows, kBlockM);
  p->num_m_pairs = (p->num_m_blocks + 1) / 2;
  p->num_n_tiles = (int)ceil_div(cols, kBlockN);
  p->rows_pad = p->num_m_blocks * kBlockM;
  const int64_t total = (int64_t)p->num_m_pairs * p->num_n_tiles;  // 256 x 256 tiles, one CTA pair each
  PGICA_REQUIRE(total < (1ll << 30), "gemm_lse: too many tiles");
  const int pairs = device_sm_count() / 2;
  *grid = 2 * (int)(total < pairs ? total : pairs);
  *ws_bytes = 3 * align_up((size_t)p->num_n_tiles * kMaxEpiGroups * p->rows_pad * sizeof(float), 256);
  return PGICA_OK;
}

size_t col_stats_bytes(const GemmLseParams& p, size_t* sum_bytes) {
  const size_t groups = static_cast<size_t>(p.rows_pad) / 32;
  const size_t cols_pad = align_up((size_t)p.cols, 32);
  *sum_bytes = align_up(groups * cols_pad * sizeof(float), 256);
  return *sum_bytes + align_up(groups * (size_t)p.num_n_tiles * 8 * sizeof(float), 256);
}

// Launch one of the tile kernels on CTA pairs (2-CTA clusters) with the full shared-memory ring.
template <class Kernel, class... Args>
int launch_pairs(Kernel kern, int grid, int threads, cudaStream_t st, const Args&... args) {
  PGICA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PGICA_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, args...));
  count_launches(1);
  return PGICA_OK;
}

// Workspace of the retrieval ranks: tile mask, row keys, column positives.  Nothing grows with rows * cols but the mask.
size_t rank_ws_bytes(const GemmLseParams& p, size_t* mask_bytes, size_t* key_bytes) {
  *mask_bytes = align_up((size_t)p.num_m_pairs * p.num_n_tiles, 256);
  *key_bytes = align_up((size_t)p.rows * sizeof(uint32_t), 256);
  return *mask_bytes + *key_bytes + align_up((size_t)p.cols * sizeof(float), 256);
}

}  // namespace
}  // namespace pgica

extern "C" {

int pgica_gemm_lse_workspace_bytes(int64_t rows, int64_t cols, int64_t k, size_t* bytes_host) {
  pgica::GemmLseParams p{};
  int grid = 0;
  return pgica::plan(rows, cols, k, &p, &grid, bytes_host);
}

static int gemm_lse_impl(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale,
                         const int32_t* labels, int64_t diag_offset, float* lse, float* tgt, float* z_out,
                         void* workspace, size_t workspace_bytes, void* stream, float* lse_col = nullptr) {
  using namespace pgica;
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  GemmLseParams p{};
  int grid = 0;
  size_t need = 0;
  rc = plan(rows, cols, k, &p, &grid, &need);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(a && b && lse, "gemm_lse: null operand");
  PGICA_REQUIRE(scale > 0.f && scale == scale, "gemm_lse: scale must be positive (got %g)", (double)scale);
  size_t col_sum_bytes = 0;
  const size_t col_bytes = lse_col ? col_stats_bytes(p, &col_sum_bytes) : 0;
  if (workspace_bytes < need + col_bytes || !workspace) {
    set_error("gemm_lse: workspace too small (%zu < %zu)", workspace_bytes, need + col_bytes);
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  if (lse_col) {
    p.col_sum = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + need);
    p.col_shift = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + need + col_sum_bytes);
    p.cols_pad = (int)align_up((size_t)cols, 32);
  }
  const size_t seg = need / 3;
  p.part_max = reinterpret_cast<float*>(workspace);
  p.part_sum = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + seg);
  p.part_tgt = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + 2 * seg);
  p.num_parts = p.num_n_tiles * epi_groups(lse_col != nullptr);
  p.scale = scale;
  p.labels = labels;
  p.diag_offset = (int)diag_offset;
  p.z_out = z_out;

  CUtensorMap tm_a, tm_b;
  rc = make_tmap_bf16(&tm_a, a, rows, k, k, kBlockM);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_b, b, cols, k, k, kBlockN / 2);
  if (rc != PGICA_OK) return rc;

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = launch_pairs(lse_col ? gemm_lse_kernel<true> : gemm_lse_kernel<false>, grid, block_threads(lse_col != nullptr), st,
                    tm_a, tm_b, p);
  if (rc != PGICA_OK) return rc;
  lse_merge_kernel<<<(unsigned)ceil_div(rows, kMergeRows), kMergeRows * kMergeGroups, 0, st>>>(p, lse, tgt);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  if (lse_col) {
    col_merge_kernel<<<(unsigned)ceil_div(cols, 32), 512, 0, st>>>(p, p.rows_pad / 32, lse_col);
    PGICA_CUDA_OK(cudaGetLastError());
    count_launches(1);
  }
  return PGICA_OK;
}

int pgica_gemm_lse_rowcol_workspace_bytes(int64_t rows, int64_t cols, int64_t k, size_t* bytes_host) {
  pgica::GemmLseParams p{};
  int grid = 0;
  size_t need = 0;
  int rc = pgica::plan(rows, cols, k, &p, &grid, &need);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  size_t sum_bytes = 0;
  *bytes_host = need + pgica::col_stats_bytes(p, &sum_bytes);
  return PGICA_OK;
}

int pgica_gemm_lse_rowcol(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale,
                          const int32_t* labels, int64_t diag_offset, float* lse_row, float* tgt, float* lse_col,
                          void* workspace, size_t workspace_bytes, void* stream) {
  PGICA_REQUIRE(lse_col, "gemm_lse_rowcol: null column output");
  return gemm_lse_impl(a, b, rows, cols, k, scale, labels, diag_offset, lse_row, tgt, nullptr, workspace,
                       workspace_bytes, stream, lse_col);
}

int pgica_gemm_lse(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale,
                   const int32_t* labels, int64_t diag_offset, float* lse, float* tgt, void* workspace,
                   size_t workspace_bytes, void* stream) {
  return gemm_lse_impl(a, b, rows, cols, k, scale, labels, diag_offset, lse, tgt, nullptr, workspace,
                       workspace_bytes, stream);
}

int pgica_retrieval_ranks_workspace_bytes(int64_t rows, int64_t cols, int64_t k, size_t* bytes_host) {
  pgica::GemmLseParams p{};
  int grid = 0;
  size_t lse_bytes = 0, mask_bytes = 0, key_bytes = 0;
  int rc = pgica::plan(rows, cols, k, &p, &grid, &lse_bytes);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  *bytes_host = pgica::rank_ws_bytes(p, &mask_bytes, &key_bytes);
  return PGICA_OK;
}

int pgica_retrieval_ranks(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, const int32_t* col_owner,
                          int32_t* row_rank, int32_t* col_rank, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace pgica;
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  GemmLseParams p{};
  int grid = 0;
  size_t lse_bytes = 0, mask_bytes = 0, key_bytes = 0;
  rc = plan(rows, cols, k, &p, &grid, &lse_bytes);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(a && b && row_rank && col_rank, "retrieval_ranks: null operand");
  const size_t need = rank_ws_bytes(p, &mask_bytes, &key_bytes);
  if (workspace_bytes < need || !workspace) {
    set_error("retrieval_ranks: workspace too small (%zu < %zu)", workspace_bytes, need);
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  RankParams r{};
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  r.col_owner = col_owner;
  r.tile_mask = ws;
  r.pos_key = reinterpret_cast<uint32_t*>(ws + mask_bytes);
  r.pos_col = reinterpret_cast<float*>(ws + mask_bytes + key_bytes);
  r.row_rank = row_rank;
  r.col_rank = col_rank;

  CUtensorMap tm_a, tm_b;
  rc = make_tmap_bf16(&tm_a, a, rows, k, k, kBlockM);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_b, b, cols, k, k, kBlockN / 2);
  if (rc != PGICA_OK) return rc;

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t init_n = std::max<int64_t>((int64_t)(p.num_m_pairs * p.num_n_tiles), rows);
  rank_init_kernel<<<(unsigned)std::min<int64_t>(ceil_div(init_n, 256), 4096), 256, 0, st>>>(p, r, p.num_m_pairs * p.num_n_tiles);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  rank_mark_kernel<<<(unsigned)ceil_div(cols, 256), 256, 0, st>>>(p, r);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  rc = launch_pairs(gemm_rank_kernel<true>, grid, block_threads(true), st, tm_a, tm_b, p, r);
  if (rc != PGICA_OK) return rc;
  return launch_pairs(gemm_rank_kernel<false>, grid, block_threads(true), st, tm_a, tm_b, p, r);
}

int pgica_similarity(const void* a, const void* b, int64_t rows, int64_t cols, int64_t k, float scale, float* sim,
                     float* lse, void* workspace, size_t workspace_bytes, void* stream) {
  PGICA_REQUIRE(sim && lse, "similarity: null output");
  return gemm_lse_impl(a, b, rows, cols, k, scale, nullptr, 0, lse, nullptr, sim, workspace, workspace_bytes, stream);
}

}  // extern "C"
