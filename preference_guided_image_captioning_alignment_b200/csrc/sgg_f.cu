// Dual softmax-gradient GEMM: BOTH products of a backward pass from ONE recomputation of the logits.
//
//   OutX[i, :] = sum_j G(i, j) * Y[j, :]        (DPO: dH, X = hidden, Y = LM-head weight;  NT-Xent: dA)
//   OutY[j, :] = sum_i G(i, j) * X[i, :]        (DPO: dW;                                   NT-Xent: dB)
//   G(i, j) as in sgg.cu (row term and/or column term), z_ij = <X_i, Y_j> recomputed on the tensor cores.
//
// sggx_kernel (sgg_x.cu) runs once per product and therefore recomputes every 128 x 128 tile of logits twice:
// 4 GEMM-units of tensor work for 2 units of result.  Here a tile of G is produced once and consumed twice, 3 units.
// TMEM is what makes that possible and what shapes the kernel: an SM holds 128 x 512 fp32 accumulators, so the
// 148 SMs together hold 74 slices of (128 rows x 1024 columns).  The whole GPU runs ONE persistent cooperative
// grid of CTA PAIRS (2-CTA clusters, tcgen05 cta_group::2: M = 256 instructions whose B operand is split across
// the two shared memories, which halves the operand fill and read traffic per SM — with single-CTA instructions
// the tensor pipe lost 15-25 % to shared-memory bandwidth, profiles/r1_trace_sggf_v1_1cta.log).  A pair takes one
// of three roles for the lifetime of the launch:
//
//   X-holders  (R/2)*S pairs (S = k/512): CTA rho keeps OutX of row block 2rp + rho (512 columns) resident in
//              TMEM for a whole chunk of R row blocks and accumulates OutX[r] += G(r, c) * Y[c] over all c,
//   Y-holders  (Cw/2)*S pairs: CTA rho keeps OutY of column tile 2cp + rho resident for one pass over the chunk's
//              row blocks and accumulates OutY[c] += G(r, c)^T * X[r]  (G^T is the same tile read MN-major),
//   producers  the rest: recompute the 256 x 256 quad Z = X[2rp, 2rp+1] Y[2cp, 2cp+1]^T (CTA rho ends up with
//              the rows of block 2rp + rho), turn it into bf16 G tiles and publish them with a TMA store into an
//              exchange ring in global memory (a few MB, overwritten every few tiles, L2-resident) followed by a
//              release store to a per-slot flag.
//
// Consumers poll the flag (acquire), pull the tile through TMA into shared memory and feed tcgen05.mma; when the
// tile has landed they bump a per-slot counter that lets the producer reuse the slot.  Within a pass the quads are
// produced along diagonals (time step t: row pair (cp + t) mod Rc for column pair cp), so every holder consumes at
// a steady rate and the exchange ring stays short.  Nothing tile-sized beyond that ring ever reaches memory, and no
// reduction through memory is needed: OutX is complete when its chunk ends, OutY when its pass ends (and is
// accumulated in place, fp32, when X needs more than one chunk).  Row blocks / column tiles past the end of X / Y
// (odd counts) are computed from TMA's zero fill and never stored.
//
// Progress: every role walks the quads in the same global production order q.  The lowest-numbered unfinished tile
// can always be produced (its slot's previous tenant has a lower number) and consumed (its consumers have nothing
// older to wait for), so the grid cannot deadlock provided all CTAs are co-resident — hence the cooperative launch.
#include <stdlib.h>

#include "common.h"
#include "sgg_tile.cuh"

#include <mutex>

namespace pgica {
namespace {

constexpr int kBM = 128;
constexpr int kBT = 128;
constexpr int kBK = 64;
constexpr int kNC = 512;                              // output columns per holder CTA (all of its TMEM)
constexpr uint32_t kChunkBytes = 128 * kBK * 2;       // 16 KB: a [128][64] bf16 box
constexpr uint32_t kPBytes = kBM * kBT * 2;           // 32 KB: one G tile
constexpr uint32_t kPStageBytes = 2 * kChunkBytes;    // producer ring slot: X chunk + this CTA's half of the Y chunk
constexpr int kPRing = 6;
constexpr uint32_t kBox64Bytes = 64 * kBK * 2;        // 8 KB: a [64][64] box
constexpr uint32_t kCStageBytes = 4 * kBox64Bytes;    // holder ring slot: 64 operand rows x this CTA's 256 columns
constexpr int kCRing = 4;
constexpr uint32_t kDrainBytes = 32768;                // holder: 4 drain warps x two 4 KB TMA-store buffers
constexpr int kStagesPerTile = kBT / 64;              // 2
// Producer epilogue warps.  With both softmax terms (NT-Xent, k = 512) the epilogue is the producer's bottleneck and a
// lone warp per scheduler issues only ~0.3 instructions per cycle on its dependent FFMA / MUFU chains (ncu stall
// samples, profiles/r2_ncu_ntxent_bwd_stalls.txt): 8 warps, two per scheduler.  With the row term only (the LM head,
// k = 1024) the tensor pipe is the bottleneck and the kernel stays at 4 — 256 threads x 168 registers leave room in
// the register file for the all-reduce kernel that runs beside it (peer_ar.cu); 384 threads would fill it.
constexpr int epi_warps(bool row, bool col) { return col ? 8 : (void(row), 4); }
constexpr int block_threads(bool row, bool col) { return 128 + 32 * epi_warps(row, col); }
// No slack for aligning the dynamic window by hand: the array is declared __align__(1024) (checked on the device),
// which keeps 1.5 KB of the SM's 228 KB free — enough for the 1 KB the hardware reserves per resident CTA, so that a
// small shared-memory-free kernel (the progress-gated peer all-reduce, peer_ar.cu) can run BESIDE this one.
constexpr size_t kSmem = 7 * 32768 + 3 * kBT * 4 + 512;
static_assert(kPRing * kPStageBytes + kPBytes == 7 * 32768, "producer shared-memory plan");
static_assert(2 * kPBytes + kCRing * kCStageBytes + kDrainBytes == 7 * 32768, "holder shared-memory plan");

#ifdef PGICA_TRACE
__device__ long long* g_sggf_trace = nullptr;
#endif

struct SggfParams {
  int mx, my, k;
  int RB2, J2;            // row-block pairs of X, column-tile pairs of Y
  int R2, C2, S;          // row pairs per chunk, column pairs per pass, 512-column splits of k
  int CG;                 // column groups: X-holder (row pair, group g) accumulates only the column pairs cp with cp % CG == g
                          //   (few row blocks: several pairs share the sweep over Y; partial OutX sums are add-reduced)
  int nH, nW, nP, D;      // PAIRS per role; exchange double-slots per producer CTA
  int spread;             // 1: spread an X-holder's quads evenly over a pass (StepOffsets)
  int debug_producers_only;  // diagnostics: holders exit at once, producers publish nothing (results are garbage)
  int outx_bf16, outy_bf16;
  SoftmaxGradStats st;
  void* out_x;
  void* out_y;
  uint32_t* progress;     // optional: progress[s] += 1 (release, gpu scope) whenever a drain warp's stores of a FINAL
  int cp_per_seg;         //   OutY tile of segment s = (column pair / cp_per_seg) are complete; a column pair (256 rows
                          //   of OutY) contributes 8 * S increments.  Lets a co-resident kernel or the host start
                          //   moving finished rows of OutY (the data-parallel all-reduce of dW) while the grid is
                          //   still computing the rest.
  uint32_t* ready;        // [2*nP*D*2] use count + 1 of the tile that is complete in the slot
  uint32_t* done;         // [2*nP*D*2] consumers that have pulled a tile out of the slot, ever
};

// ---- PTX pieces only this kernel uses
// L2 eviction priorities: the exchange ring is a few MB that every tile passes through (keep it: evict_last), the
// output gradients are written once and never read again by this launch (evict_first).  Measured effect on cfg2: DRAM
// traffic 880 -> 825 MB per launch; what remains above the 325 MB of algorithmic bytes is the two-chunk plan itself
// (W streamed once per chunk, dW stored by the first chunk and read-modify-written by the second).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_store_2d_hint(const void* tmap, const void* smem_src, int c0, int c1, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_hint(void* smem_dst, const void* tmap, uint32_t bar_cluster, int c0,
                                                      int c1, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, "
      "{%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1), "l"(pol)
      : "memory");
}
// TMA load into THIS CTA's shared memory whose completion bytes are credited to a barrier that may live in the
// pair's other CTA (`bar_cluster` is a shared::cluster address): how both halves of a cta_group::2 operand report
// to the leader's barrier.
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
// all MMAs issued so far by this thread complete -> one arrival on the same-offset barrier of BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
// fp32 tile shared -> global: plain store, or element-wise add into what is there
__device__ __forceinline__ void tma_reduce_add_2d(const void* tmap, const void* smem_src, int c0, int c1, uint64_t pol) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(pol)
               : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_relaxed_gpu_add(uint32_t* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Spin until *p >= v (monotonic counters); traps instead of hanging if the protocol is broken.
__device__ __forceinline__ void wait_flag_ge(const uint32_t* p, uint32_t v) {
  if (ld_acquire_gpu(p) >= v) return;
  const long long t0 = clock64();
  while (ld_acquire_gpu(p) < v) {
    __nanosleep(40);
    if (clock64() - t0 > PGICA_WATCHDOG_CYCLES) {
      printf("pgica: exchange-flag watchdog (block %d thread %d want %u have %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, v, ld_acquire_gpu(p));
      __trap();
    }
  }
}

// Production order.  A pass covers Rc row pairs x Cc column pairs in Rc time steps; in step t column pair c meets row
// pair (off(c) + t) mod Rc with off(c) = floor(c * Rc / Cc): every Y-holder consumes one quad per step, and the steps
// in which a given X-holder is served are spread evenly over the pass (with off(c) = c they would come in one burst
// of Cc consecutive steps, which the exchange ring would have to absorb).  StepOffsets walks off(c) for c = 0, 1, ...
struct StepOffsets {
  int off, acc, Rc, Cc;
  int step;
  __host__ __device__ StepOffsets(int rc, int cc, int spread) : off(0), acc(0), Rc(rc), Cc(cc), step(spread ? rc : cc) {}
  __host__ __device__ void next() {
    acc += step;
    while (acc >= Cc) {
      acc -= Cc;
      ++off;
    }
  }
  __host__ __device__ int row(int t) const {  // (off + t) mod Rc; off may reach Rc when Cc < Rc is false, hence the loop
    int r = off + t;
    while (r >= Rc) r -= Rc;
    return r;
  }
};

// Visits every quad in production order.  f(q, r0, r, c0, c): sequence number q; the quad covers row pair r0 + r
// (row blocks 2(r0+r), 2(r0+r)+1) and column pair c0 + c.
template <class F>
__host__ __device__ __forceinline__ void for_each_quad(const SggfParams& p, F&& f) {
  int q = 0;
  for (int r0 = 0; r0 < p.RB2; r0 += p.R2) {
    const int Rc = p.R2 < p.RB2 - r0 ? p.R2 : p.RB2 - r0;
    for (int c0 = 0; c0 < p.J2; c0 += p.C2) {
      const int Cc = p.C2 < p.J2 - c0 ? p.C2 : p.J2 - c0;
      for (int t = 0; t < Rc; ++t) {
        StepOffsets so(Rc, Cc, p.spread);
        for (int c = 0; c < Cc; ++c, ++q) {
          f(q, r0, so.row(t), c0, c);
          so.next();
        }
      }
    }
  }
}

// The quads q = first, first + stride, ... of the same production order WITHOUT walking the ones in between: a cursor
// over the (chunk, pass) blocks plus the closed form of StepOffsets (off(c) = floor(c * step / Cc)).  Every producer
// warp used to run for_each_quad over ALL quads and skip the foreign ones — ~240 cycles of loop control per quad,
// i.e. ~9 k cycles per own quad with 36 producers: more than the 8.8 k cycles the MMAs of a k = 1024 quad take, and all
// of it serial in the epilogue warps (profiles/r2_trace_sggf_enumeration_overhead.log: epi_other = quads x 240).
template <class F>
__host__ __device__ __forceinline__ void for_each_own_quad(const SggfParams& p, int first, int stride, F&& f) {
  int r0 = 0, c0 = 0, qbase = 0;
  int Rc = p.R2 < p.RB2 ? p.R2 : p.RB2;
  int Cc = p.C2 < p.J2 ? p.C2 : p.J2;
  for (int q = first;; q += stride) {
    while (q >= qbase + Rc * Cc) {  // advance to the block that holds q
      qbase += Rc * Cc;
      c0 += p.C2;
      if (c0 >= p.J2) {
        c0 = 0;
        r0 += p.R2;
        if (r0 >= p.RB2) return;
        Rc = p.R2 < p.RB2 - r0 ? p.R2 : p.RB2 - r0;
      }
      Cc = p.C2 < p.J2 - c0 ? p.C2 : p.J2 - c0;
    }
    const int ql = q - qbase;
    const int t = ql / Cc, c = ql - t * Cc;
    const int off = p.spread ? (c * Rc) / Cc : c;  // StepOffsets after c steps
    f(q, r0, (off + t) % Rc, c0, c);
  }
}

// Visits, in production order, the pair-tiles one holder pair accumulates (two per quad).  is_y = false: X-holder of
// row pair `idx` (chunk-relative); true: Y-holder of column pair `idx` (pass-relative).  f(q, sel, rp, cp, first,
// period): quad q = (row pair rp, column pair cp), absolute; sel = 0/1 picks the column tile 2cp + sel (X-holder)
// or the row block 2rp + sel (Y-holder); `first` marks the first pair-tile of an accumulation period.  g(period,
// chunk, pass) is called after the last pair-tile of every period that had any.
template <class F, class G>
__host__ __device__ __forceinline__ void for_each_holder_tile(const SggfParams& p, bool is_y, int idx, F&& f, G&& g) {
  int qbase = 0, period = 0;
  const int CG = p.CG > 1 ? p.CG : 1;
  const int xrow = is_y ? 0 : idx / CG, xgrp = is_y ? 0 : idx % CG;  // X-holder slot = (row pair in chunk, column group)
  for (int r0 = 0, chunk = 0; r0 < p.RB2; r0 += p.R2, ++chunk) {
    const int Rc = p.R2 < p.RB2 - r0 ? p.R2 : p.RB2 - r0;
    bool first = true;
    for (int c0 = 0, pass = 0; c0 < p.J2; c0 += p.C2, ++pass) {
      const int Cc = p.C2 < p.J2 - c0 ? p.C2 : p.J2 - c0;
      if (is_y) {
        if (idx < Cc) {
          StepOffsets so(Rc, Cc, p.spread);
          for (int c = 0; c < idx; ++c) so.next();
          for (int t = 0; t < Rc; ++t) {
            const int q = qbase + t * Cc + idx;
            const int r = so.row(t);
            f(q, 0, r0 + r, c0 + idx, t == 0, period);
            f(q, 1, r0 + r, c0 + idx, false, period);
          }
          g(period, chunk, pass);
          ++period;
        }
      } else if (xrow < Rc && !p.spread) {
        // off(c) = c: column pair c meets this row pair in step t iff c = xrow - t (mod Rc) — visited directly (walking
        // all Rc x Cc quads of the pass to find them cost ~240 cycles each, see for_each_own_quad)
        for (int t = 0; t < Rc; ++t) {
          int c = xrow - t;
          if (c < 0) c += Rc;
          for (; c < Cc; c += Rc) {
            if (CG == 1 || (c0 + c) % CG == xgrp) {
              const int q = qbase + t * Cc + c;
              f(q, 0, r0 + xrow, c0 + c, first, period);
              first = false;
              f(q, 1, r0 + xrow, c0 + c, false, period);
            }
          }
        }
      } else if (xrow < Rc) {
        for (int t = 0; t < Rc; ++t) {
          StepOffsets so(Rc, Cc, p.spread);
          for (int c = 0; c < Cc; ++c) {  // column pairs that meet this row pair in step t, increasing
            if (so.row(t) == xrow && (c0 + c) % CG == xgrp) {
              const int q = qbase + t * Cc + c;
              f(q, 0, r0 + xrow, c0 + c, first, period);
              first = false;
              f(q, 1, r0 + xrow, c0 + c, false, period);
            }
            so.next();
          }
        }
      }
      qbase += Rc * Cc;
    }
    if (!is_y && xrow < Rc) {
      g(period, chunk, 0);
      ++period;
    }
  }
}

// kShared (both terms only): the caller guarantees |logit| <= scale (unit-norm rows) and column targets that mirror the
// row targets (NT-Xent).  One exponential e = 2^(z c - c) then serves both softmax terms, P_row = e 2^(c - lse_row) and
// P_col = e 2^(c - lse_col), each factor finite in fp32 because 2 c < 100; and the two one-hots fall on the same
// element, handled outside the inner loop.
template <bool kRow, bool kCol, bool kShared = false>
__global__ void __launch_bounds__(block_threads(kRow, kCol), 1)
sggf_kernel(const __grid_constant__ CUtensorMap tm_x128, const __grid_constant__ CUtensorMap tm_y128,
            const __grid_constant__ CUtensorMap tm_x64, const __grid_constant__ CUtensorMap tm_y64,
            const __grid_constant__ CUtensorMap tm_s, const __grid_constant__ CUtensorMap tm_ox,
            const __grid_constant__ CUtensorMap tm_oy, const SggfParams p) {
  constexpr int kEpiWarps = epi_warps(kRow, kCol), kEpiThreads = 32 * kEpiWarps;
  constexpr int kChunksPerWarp = 16 / kEpiWarps;  // 32-column chunks of a 128-column tile per epilogue warp (4 or 2)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0) {
    if (threadIdx.x == 0) printf("pgica: sggf_kernel dynamic shared memory is not 1024-byte aligned\n");
    __trap();
  }
  float* s_col = reinterpret_cast<float*>(smem + 7 * 32768);
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_col + 3 * kBT);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rho = cluster_ctarank();      // 0 = leader of the pair (issues the MMAs)
  const int pair = (int)blockIdx.x >> 1;
  const bool is_producer = pair >= p.nH + p.nW;
  const int num_kb = p.k / kBK;
  const uint32_t n_consumers = 2u * (uint32_t)p.S;  // CTAs that pull each G tile

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x128);
    tma_prefetch_desc(&tm_y128);
    tma_prefetch_desc(&tm_x64);
    tma_prefetch_desc(&tm_y64);
    tma_prefetch_desc(&tm_s);
    tma_prefetch_desc(&tm_ox);
    tma_prefetch_desc(&tm_oy);
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }

  if (is_producer) {
    // =================================================================================================== producer
    uint8_t* ring = smem;
    uint8_t* staging = smem + kPRing * kPStageBytes;
    uint64_t* full_bar = bars;                 // [kPRing] leader's: both CTAs' halves of a stage have landed (the leader
                                               //          expects the bytes of both, the peer's TMA credits it remotely)
    uint64_t* empty_bar = full_bar + kPRing;   // [kPRing] per CTA (multicast commit)
    uint64_t* zfull_bar = empty_bar + kPRing;  // [2] per CTA (multicast commit)
    uint64_t* zempty_bar = zfull_bar + 2;      // [2] leader's: both CTAs' epilogues have read the Z buffer
    uint64_t* stfull_bar = zempty_bar + 2;
    uint64_t* stfree_bar = stfull_bar + 1;
    if (warp == 1 && lane == 0) {
      for (int i = 0; i < kPRing; ++i) {
        mbar_init(&full_bar[i], 1);
        mbar_init(&empty_bar[i], 1);
      }
      for (int i = 0; i < 2; ++i) {
        mbar_init(&zfull_bar[i], 1);
        mbar_init(&zempty_bar[i], 2 * kEpiThreads);
      }
      mbar_init(stfull_bar, kEpiThreads);
      mbar_init(stfree_bar, 1);
      fence_mbar_init();
    }
    tc_fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const int pp = pair - p.nH - p.nW;             // producer pair number
    const uint32_t pcta = (uint32_t)pp * 2u + rho;  // producer CTA number (owns D double slots of the ring)

    if (warp == 0 || warp == 2) {
      // ---------------------------------------------------------------- TMA loads of this CTA's MMA1 operand halves
      // Two loader warps, one per stage parity: a single warp needs ~500 cycles per stage (barrier wait, expect_tx,
      // two TMA issues) against the ~550 the tensor pipe takes to consume one, which leaves no slack for jitter.
      // (Four loader warps were measured too: no further gain.)
      const int par = warp >> 1;
      int slot = 0;
      uint32_t phase = 0, stage_no = 0;
      const uint32_t lbar0 = mapa_u32(smem_u32(&full_bar[0]), 0);  // the leader's full barriers (shared::cluster)
      LAP_DECL(6);
      for_each_own_quad(p, pp, p.nP, [&](int q, int r0, int r, int c0, int c) {
        const int xrow = (2 * (r0 + r) + (int)rho) * kBM, yrow = (2 * (c0 + c) + (int)rho) * kBT;
        for (int kb = 0; kb < num_kb; ++kb, ++stage_no) {
          if ((int)(stage_no & 1u) == par) {
            LAP(0);
            mbar_wait(&empty_bar[slot], phase ^ 1);
            LAP(1);
            if (elect_one()) {
              const uint32_t lbar = lbar0 + slot * 8;
              if (rho == 0) mbar_expect_tx(&full_bar[slot], 2 * kPStageBytes);
              uint8_t* dst = ring + slot * kPStageBytes;
              tma_load_2d_pair(dst, &tm_x128, lbar, kb * kBK, xrow);
              tma_load_2d_pair(dst + kChunkBytes, &tm_y128, lbar, kb * kBK, yrow);
            }
            __syncwarp();
          }
          if (++slot == kPRing) {
            slot = 0;
            phase ^= 1;
          }
        }
      });
      LAP(0);
      if (lane == 0 && warp == 0) LAP_FLUSH(g_sggf_trace, 4, 2);
    } else if (warp == 1 && rho == 0) {
      // ---------------------------------------------------------------- MMA1 (leader): Z[256 x 256] = X[2rp, 2rp+1] Y[2cp, 2cp+1]^T
      constexpr uint32_t idesc1 = make_idesc_bf16(256, 256, 0, 0);
      const uint64_t desc_k = make_smem_desc(0, 16, 1024);
      int slot = 0;
      uint32_t phase = 0, n = 0;
      LAP_DECL(6);
      for_each_own_quad(p, pp, p.nP, [&](int q, int, int, int, int) {
        const uint32_t buf = n & 1u;
        LAP(0);
        mbar_wait_cluster(&zempty_bar[buf], ((n >> 1) & 1u) ^ 1u);  // both epilogues have read this Z buffer
        LAP(1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * 256u;
        for (int kb = 0; kb < num_kb; ++kb) {
          LAP(0);
          mbar_wait_cluster(&full_bar[slot], phase);
          LAP(2);
          tc_fence_after_sync();
          if (elect_one()) {
            const uint32_t x_addr = smem_u32(ring + slot * kPStageBytes);
            const uint64_t da = desc_k | ((x_addr >> 4) & 0x3FFF);
            const uint64_t db = desc_k | (((x_addr + kChunkBytes) >> 4) & 0x3FFF);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k) umma2_bf16_ss(d_tmem, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
            umma2_commit_both(&empty_bar[slot]);
            if (kb == num_kb - 1) umma2_commit_both(&zfull_bar[buf]);
          }
          __syncwarp();
          if (++slot == kPRing) {
            slot = 0;
            phase ^= 1;
          }
        }
        ++n;
      });
      LAP(0);
      if (lane == 0) LAP_FLUSH(g_sggf_trace, 0, 3);
    } else if (warp == 3) {
      // ---------------------------------------------------------------- exchange: staging -> ring slot -> flag
      uint32_t n = 0, ntile = 0;
      const uint64_t pol_keep = l2_policy_evict_last();
      LAP_DECL(6);
      for_each_own_quad(p, pp, p.nP, [&](int q, int, int, int, int) {
        const uint32_t ds = n % (uint32_t)p.D, use = n / (uint32_t)p.D;
        for (int half = 0; half < 2; ++half) {
          const uint32_t tslot = (pcta * p.D + ds) * 2u + half;
          LAP(0);
          mbar_wait(stfull_bar, ntile & 1u);
          LAP(1);
          if (use > 0 && !p.debug_producers_only) wait_flag_ge(p.done + tslot, n_consumers * use);  // every consumer has pulled the old tile
          LAP(2);
          if (lane == 0 && p.debug_producers_only) mbar_arrive(stfree_bar);
          if (lane == 0 && !p.debug_producers_only) {
            asm volatile("fence.proxy.async.global;" ::: "memory");  // acquire above before the async-proxy write
            tma_store_2d_hint(&tm_s, staging, 0, (int)tslot * kBM, pol_keep);
            tma_store_2d_hint(&tm_s, staging + kChunkBytes, kBK, (int)tslot * kBM, pol_keep);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // staging has been read
            mbar_arrive(stfree_bar);
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the tile is complete in global memory
            asm volatile("fence.proxy.async.global;" ::: "memory");
            st_release_gpu(p.ready + tslot, use + 1u);
          }
          __syncwarp();
          LAP(3);
          ++ntile;
        }
        ++n;
      });
      LAP(0);
      if (lane == 0) LAP_FLUSH(g_sggf_trace, 6, 4);
    } else if (warp >= 4) {
      // ---------------------------------------------------------------- epilogue: this CTA's Z rows -> two G tiles
      // Warp w reads the TMEM lanes of quarter w & 3 (the hardware's lane window of a warp) and, with eight warps, of
      // every 128-column tile the 64 columns of its group (w - 4) >> 2 — one [128][64] box of the staging tile each.
      const int quarter = warp & 3, wg = (warp - 4) >> 2;
      const int et = threadIdx.x - 128;
      const int row_in_blk = quarter * 32 + lane;
      const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
      const uint32_t g_local = smem_u32(staging);
      uint32_t n = 0, ntile = 0;
      LAP_DECL(6);
      for_each_own_quad(p, pp, p.nP, [&](int q, int r0, int r, int c0, int c) {
        const int row = (2 * (r0 + r) + (int)rho) * kBM + row_in_blk;
        float rl, rc;
        int rt;
        load_row_stat<kRow>(p.st, row, row < p.mx, rl, rc, rt);
        const float rs = kShared ? rc * fast_exp2(p.st.c - rl) : 0.f;  // the row's factor of the shared exponential
        const uint32_t buf = n & 1u;
        LAP(0);
        mbar_wait(&zfull_bar[buf], (n >> 1) & 1u);
        LAP(1);
        tc_fence_after_sync();
        for (int half = 0; half < 2; ++half) {
          const int col0 = (2 * (c0 + c) + half) * kBT;
          if (kCol) {
            if (et < kBT) {
              float l, cf;
              int tg;
              load_col_stat<kCol>(p.st, col0 + et, col0 + et < p.my, l, cf, tg);
              stage_col_stat<kShared>(s_col, et, l, cf, tg, p.st.c);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          }
          const int rrel = rt - col0;
          uint32_t gp[kChunksPerWarp * 16];
#pragma unroll
          for (int cl = 0; cl < kChunksPerWarp; ++cl) {
            const int ch = wg * kChunksPerWarp + cl;  // 32-column chunk of the tile
            uint32_t rr[32];
            tmem_ld_32x32(tmem_base + lane_addr + buf * 256u + half * kBT + ch * 32, rr);
            tmem_ld_wait();
            float g[32];
            g_chunk<kRow, kCol, kShared>(rr, p.st.c, rl, rc, rs, row, rrel, s_col, ch, g);
            pack_g_chunk(g, gp + cl * 16);
          }
          if (half == 1) {
            tc_fence_before_sync();
            mbar_arrive_cluster(&zempty_bar[buf], 0);  // tell the leader: this thread has read the Z buffer
          }
          LAP(2);
          mbar_wait(stfree_bar, (ntile & 1u) ^ 1u);  // the exchange warp's TMA store has read the previous tile
          LAP(3);
#pragma unroll
          for (int cl = 0; cl < kChunksPerWarp; ++cl)
            store_g_chunk(g_local, row_in_blk, wg * kChunksPerWarp + cl, gp + cl * 16);
          fence_proxy_async_smem();
          mbar_arrive(stfull_bar);
          ++ntile;
          if (kCol) asm volatile("bar.sync 3, %0;" ::"n"(kEpiThreads) : "memory");  // the column statistics may be overwritten
          LAP(4);
        }
        ++n;
      });
      LAP(0);
      if (et == 0) LAP_FLUSH(g_sggf_trace, 10, 5);
    }
    tc_fence_before_sync();
    __syncthreads();
    cluster_sync_all();  // the pair shares barriers and TMEM commits: nobody leaves early
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    return;
  }

  // ======================================================================================================= holders
  const bool is_y = pair >= p.nH;
  const int hidx = (is_y ? pair - p.nH : pair) / p.S;   // X-holder: (row pair in chunk) * CG + column group; Y-holder: column pair in pass
  const int xrow = hidx / (p.CG > 1 ? p.CG : 1);        // X-holder's row pair in the chunk
  const int split = (is_y ? pair - p.nH : pair) % p.S;  // which 512 output columns
  uint8_t* gbuf = smem;                       // two G tiles
  uint8_t* ring = smem + 2 * kPBytes;         // kCRing operand stages
  uint8_t* drain_stage = ring + kCRing * kCStageBytes;
  uint64_t* full_bar = bars;                  // [kCRing] leader's (expects both CTAs' bytes)
  uint64_t* empty_bar = full_bar + kCRing;    // [kCRing] per CTA
  uint64_t* gfull_bar = empty_bar + kCRing;   // [2] leader's (expects both CTAs' bytes)
  uint64_t* gempty_bar = gfull_bar + 2;       // [2] per CTA
  uint64_t* outfull_bar = gempty_bar + 2;     // per CTA
  uint64_t* outfree_bar = outfull_bar + 1;    // leader's (count 256)
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kCRing; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&gfull_bar[i], 1);
      mbar_init(&gempty_bar[i], 1);
    }
    mbar_init(outfull_bar, 1);
    mbar_init(outfree_bar, 256);
    fence_mbar_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (p.debug_producers_only) {
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    return;
  }
  const CUtensorMap* tm_op = is_y ? &tm_x64 : &tm_y64;  // the other operand of this pair's product
  const int op_col0 = split * kNC + (int)rho * 128;     // this CTA's 128 of each 256-column instruction

  // exchange slot of the tile (row block 2rp + a, column tile 2cp + b) of quad q
  auto tile_slot = [&](int q, uint32_t a, uint32_t b, uint32_t& use) {
    const uint32_t prod = (uint32_t)q % (uint32_t)p.nP, i = (uint32_t)q / (uint32_t)p.nP;
    use = i / (uint32_t)p.D;
    return ((prod * 2u + a) * p.D + i % (uint32_t)p.D) * 2u + b;
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA, G tiles: poll the exchange ring, pull this CTA's tile
    // (its own warp: the flag poll is an L2 round trip per tile and must not hold up the operand loads below)
    uint32_t n = 0;
    const uint64_t pol_keep = l2_policy_evict_last();
    const uint32_t gbar0 = mapa_u32(smem_u32(&gfull_bar[0]), 0);  // the leader's barriers (shared::cluster)
    LAP_DECL(6);
    for_each_holder_tile(
        p, is_y, hidx,
        [&](int q, int sel, int, int, bool, int) {
          // X-holder CTA rho: G(2rp + rho, 2cp + sel);  Y-holder CTA rho: G(2rp + sel, 2cp + rho)
          uint32_t use;
          const uint32_t tslot = is_y ? tile_slot(q, (uint32_t)sel, rho, use) : tile_slot(q, rho, (uint32_t)sel, use);
          const uint32_t gb = n & 1u;
          LAP(0);
          mbar_wait(&gempty_bar[gb], ((n >> 1) & 1u) ^ 1u);  // the MMAs of the pair-tile before last are complete
          LAP(1);
          wait_flag_ge(p.ready + tslot, use + 1u);           // the tile is complete in the ring
          LAP(2);
          if (elect_one()) {
            asm volatile("fence.proxy.async.global;" ::: "memory");  // acquire above before the async-proxy read
            const uint32_t lbar = gbar0 + gb * 8;
            if (rho == 0) mbar_expect_tx(&gfull_bar[gb], 2 * kPBytes);
            tma_load_2d_pair_hint(gbuf + gb * kPBytes, &tm_s, lbar, 0, (int)tslot * kBM, pol_keep);
            tma_load_2d_pair_hint(gbuf + gb * kPBytes + kChunkBytes, &tm_s, lbar, kBK, (int)tslot * kBM, pol_keep);
          }
          __syncwarp();
          ++n;
        },
        [&](int, int, int) {});
    LAP(0);
    if (lane == 0) LAP_FLUSH(g_sggf_trace, 4, 3);
  } else if (warp == 2) {
    // ------------------------------------------------------------------ TMA, operand rows: this CTA's half of X[r] / Y[c]
    // (independent of the producers: runs ahead of the G tiles by the depth of the ring)
    int slot = 0;
    uint32_t phase = 0;
    const uint32_t lbar0 = mapa_u32(smem_u32(&full_bar[0]), 0);
    LAP_DECL(6);
    for_each_holder_tile(
        p, is_y, hidx,
        [&](int, int sel, int rp, int cp, bool, int) {
          const int op_row0 = (is_y ? 2 * rp + sel : 2 * cp + sel) * kBM;
          for (int st = 0; st < kStagesPerTile; ++st) {
            LAP(0);
            mbar_wait(&empty_bar[slot], phase ^ 1);
            LAP(3);
            if (elect_one()) {
              const uint32_t lbar = lbar0 + slot * 8;
              if (rho == 0) mbar_expect_tx(&full_bar[slot], 2 * kCStageBytes);
              uint8_t* dst = ring + slot * kCStageBytes;
#pragma unroll
              for (int b = 0; b < 4; ++b)  // box b: instruction h = b >> 1, 64-column chunk b & 1 of this CTA's 128
                tma_load_2d_pair(dst + b * kBox64Bytes, tm_op, lbar, op_col0 + (b >> 1) * 256 + (b & 1) * kBK,
                                 op_row0 + st * 64);
            }
            __syncwarp();
            if (++slot == kCRing) {
              slot = 0;
              phase ^= 1;
            }
          }
        },
        [&](int, int, int) {});
    LAP(0);
#ifdef PGICA_TRACE
    if (lane == 0 && g_sggf_trace) g_sggf_trace[(size_t)blockIdx.x * kTraceSlots + 7] = lap.acc[3];
#endif
  } else if (warp == 1 && rho == 0) {
    // ------------------------------------------------------------------ MMA2 (leader): Out[256 x 512] += G(^T) * operand rows
    const uint32_t idesc2 = make_idesc_bf16(256, 256, is_y ? 1 : 0, 1);
    const uint64_t desc_ak = make_smem_desc(0, 16, 1024);              // G as A, K-major (X-holder)
    const uint64_t desc_amn = make_smem_desc(0, kChunkBytes, 1024);    // G^T as A: the same tile read MN-major
    const uint64_t desc_b = make_smem_desc(0, kBox64Bytes, 1024);      // operand rows, MN-major, 64-col boxes 8 KB apart
    int slot = 0;
    uint32_t phase = 0, n = 0;
    LAP_DECL(6);
    for_each_holder_tile(
        p, is_y, hidx,
        [&](int q, int sel, int, int, bool first, int period) {
          const uint32_t gb = n & 1u;
          if (first && period > 0) {
            LAP(0);
            mbar_wait_cluster(outfree_bar, (uint32_t)(period - 1) & 1u);  // both accumulators have left TMEM
            LAP(1);
            tc_fence_after_sync();
          }
          LAP(0);
          mbar_wait_cluster(&gfull_bar[gb], (n >> 1) & 1u);
          LAP(2);
          tc_fence_after_sync();
          const uint32_t g_addr = smem_u32(gbuf + gb * kPBytes);
          const uint64_t dg = (is_y ? desc_amn : desc_ak) | ((g_addr >> 4) & 0x3FFF);
          for (int st = 0; st < kStagesPerTile; ++st) {
            LAP(0);
            mbar_wait_cluster(&full_bar[slot], phase);
            LAP(3);
            tc_fence_after_sync();
            if (elect_one()) {
              const uint32_t y_addr = smem_u32(ring + slot * kCStageBytes);
              const uint64_t dy = desc_b | ((y_addr >> 4) & 0x3FFF);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const int ks = st * 4 + kk;  // K step of 16 within the tile's 128
                const uint64_t da = is_y ? dg + ks * (2048 >> 4) : dg + (ks >> 2) * (kChunkBytes >> 4) + (ks & 3) * 2;
                const uint32_t acc = (first && ks == 0) ? 0u : 1u;
#pragma unroll
                for (int h = 0; h < 2; ++h)
                  umma2_bf16_ss(tmem_base + h * 256u, da, dy + kk * (2048 >> 4) + h * (2 * kBox64Bytes >> 4), idesc2, acc);
              }
              umma2_commit_both(&empty_bar[slot]);
              if (st == kStagesPerTile - 1) umma2_commit_both(&gempty_bar[gb]);
            }
            __syncwarp();
            if (++slot == kCRing) {
              slot = 0;
              phase ^= 1;
            }
          }
          if (elect_one()) {
            // both tiles have landed in the pair's shared memory (gfull above): their ring slots may be overwritten.
            // Relaxed and after the MMA issue: a release fence here would stall the issuing thread for an L2 round trip.
            uint32_t use;
            red_relaxed_gpu_add(p.done + (is_y ? tile_slot(q, (uint32_t)sel, 0u, use) : tile_slot(q, 0u, (uint32_t)sel, use)), 1u);
            red_relaxed_gpu_add(p.done + (is_y ? tile_slot(q, (uint32_t)sel, 1u, use) : tile_slot(q, 1u, (uint32_t)sel, use)), 1u);
          }
          __syncwarp();
          ++n;
        },
        [&](int, int, int) {
          if (elect_one()) umma2_commit_both(outfull_bar);
          __syncwarp();
        });
    LAP(0);
    if (lane == 0) LAP_FLUSH(g_sggf_trace, 0, 4);
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------------ drain: accumulator -> OutX / OutY
    const int quarter = warp & 3;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const int out_col0 = split * kNC;
    const uint64_t pol_stream = l2_policy_evict_first();
    const int n_chunks = (p.RB2 + p.R2 - 1) / p.R2;
    int pending_seg = -1;  // segment of the OutY tile whose TMA stores this warp has issued but not yet seen complete
    auto signal_progress = [&](int seg) {
      // TMA (async-proxy) stores complete -> generic-proxy release at GPU scope.  The consumer is a kernel on THIS GPU
      // (peer_ar.cu acquires the counter and relays to the other ranks with its own system-scope release: causality
      // order is transitive); a system-scope release here cost 1.8 us per drain on the Y-holders' critical path.
      asm volatile("fence.proxy.async.global;" ::: "memory");
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p.progress + seg), "r"(1u) : "memory");
    };
    LAP_DECL(6);
    for_each_holder_tile(
        p, is_y, hidx, [&](int, int, int, int, bool, int) {},
        [&](int period, int chunk, int pass) {
          const int blk = 2 * (is_y ? pass * p.C2 + hidx : chunk * p.R2 + xrow) + (int)rho;
          const bool bf16 = (is_y ? p.outy_bf16 : p.outx_bf16) != 0;
          const bool accumulate = is_y ? chunk > 0 : p.CG > 1;  // OutY over chunks / OutX over column groups (zeroed by the host)
          LAP(0);
          mbar_wait(outfull_bar, (uint32_t)period & 1u);
          LAP(1);
          tc_fence_after_sync();
          // The accumulator leaves through a swizzled staging buffer and TMA stores (TMA add-reductions when OutY is
          // accumulated over chunks): full 128-byte lines instead of 32 scattered 16-byte stores per instruction, and
          // the rows past the end of the matrix are clipped by the tensor map.  One box = 32 rows x 128 bytes:
          // 32 fp32 columns, or 64 bf16 columns.
          const CUtensorMap* tm_o = is_y ? &tm_oy : &tm_ox;
          uint8_t* stg = drain_stage + quarter * 8192;
          const int row0 = blk * kBM + quarter * 32;
          const int cols_per_box = bf16 ? 64 : 32;
          // The stores of the previous period had a whole period to complete; waiting for them HERE (not at the end of
          // their own drain) keeps a drain as short as its shared-memory traffic even when the destination is a peer
          // GPU, and still orders a tile's plain store before the add-reduction a later chunk makes into it.
          if (lane == 0) {
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            if (pending_seg >= 0) signal_progress(pending_seg);  // the previous period's tile is complete in memory
          }
          __syncwarp();
          pending_seg = (is_y && p.progress != nullptr && chunk == n_chunks - 1) ? (pass * p.C2 + hidx) / p.cp_per_seg : -1;
#pragma unroll 1
          for (int bx = 0; bx < kNC / cols_per_box; ++bx) {
            uint32_t rr[32];
            if (bf16) {
              uint32_t r2[32];
              tmem_ld_32x32(tmem_base + lane_addr + bx * 64, rr);
              tmem_ld_32x32(tmem_base + lane_addr + bx * 64 + 32, r2);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) rr[i] = pack_bf16x2(__uint_as_float(rr[2 * i]), __uint_as_float(rr[2 * i + 1]));
#pragma unroll
              for (int i = 0; i < 16; ++i) rr[16 + i] = pack_bf16x2(__uint_as_float(r2[2 * i]), __uint_as_float(r2[2 * i + 1]));
            } else {
              tmem_ld_32x32(tmem_base + lane_addr + bx * 32, rr);
              tmem_ld_wait();
            }
            if (bx >= 2) {
              if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");  // this buffer's last store has read it
              __syncwarp();
            }
            const uint32_t sb = smem_u32(stg + (bx & 1) * 4096);
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4)
              st_smem_v4(sb + sw128_offset(lane, c4), rr[c4 * 4], rr[c4 * 4 + 1], rr[c4 * 4 + 2], rr[c4 * 4 + 3]);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (accumulate)
                tma_reduce_add_2d(tm_o, stg + (bx & 1) * 4096, out_col0 + bx * cols_per_box, row0, pol_stream);
              else
                tma_store_2d_hint(tm_o, stg + (bx & 1) * 4096, out_col0 + bx * cols_per_box, row0, pol_stream);
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
          }
          tc_fence_before_sync();
          mbar_arrive_cluster(outfree_bar, 0);  // tell the leader: this CTA's accumulator may be overwritten
          LAP(2);
        });
    if (lane == 0) {
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the last period's stores are complete
      if (pending_seg >= 0) signal_progress(pending_seg);
    }
    __syncwarp();
    if (threadIdx.x == 128) LAP_FLUSH(g_sggf_trace, 10, 3);
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// ------------------------------------------------------------------------------------------------- host side
struct Plan {
  int R2, C2, nH, nW, nP;  // pairs
  double cost;
  int CG;                  // column groups of the X-holders (1 unless x has few row blocks)
};

// Time model in units of one 256 x 256 x 16 pair instruction at the rate the holders sustain (~140 cycles): a holder
// pair spends 16 per pair-tile (two per quad), a drain of the 128 x 512 accumulator costs about 90, a producer pair
// what per_quad below says.  The slowest role sets the pace of a chunk.
//
// Column groups (allow_groups): an X-holder pair sweeps ALL column pairs of its row pair, 32 instructions each —
// 6300 for the GPT-2 vocabulary however few rows x has (the compacted Stage-2 batches of the trainer have 2-4 row
// blocks).  When all of x fits one chunk with pairs to spare, CG X-holder pairs share a row pair's sweep (column pair
// cp goes to group cp % CG) and add-reduce their partial OutX at the end.
Plan choose_plan(int RB2, int J2, int k, int npairs, bool single_chunk, bool allow_groups = false,
                 bool both_terms = false) {
  const int S = k / kNC;
  // a producer pair spends per quad the longer of its MMAs (k/16 instructions, ~1.1x with the TMA waits that remain —
  // measured after round 2 removed the schedule walk from the producer warps, profiles/r2_dual_ab2.log) and of its
  // epilogue (256 x 256 elements over two CTAs: ~5 k cycles with one exponential per element, ~8 k with two)
  const double epilogue = both_terms ? 58.0 : 36.0;
  const double mma = 1.1 * k / 16.0;
  const double per_quad = mma > epilogue ? mma : epilogue, drain = 90.0;
  Plan best{0, 0, 0, 0, 0, 1e300, 1};
  for (int R2 = single_chunk ? RB2 : 1; R2 <= RB2 && R2 * S <= npairs - S - 1; ++R2) {
    const int max_groups = (allow_groups && R2 >= RB2) ? 16 : 1;
    for (int CG = 1; CG <= max_groups && CG <= J2; ++CG) {
      const int nH = R2 * S * CG;
      if (nH > npairs - S - 1) break;
      for (int C2 = 1; C2 * S <= npairs - nH - 1 && C2 <= J2; ++C2) {
        const int nW = C2 * S, nP = npairs - nH - nW;
        const int passes = (J2 + C2 - 1) / C2;
        double total = 0;
        for (int r0 = 0; r0 < RB2; r0 += R2) {
          const int Rc = RB2 - r0 < R2 ? RB2 - r0 : R2;
          const double tH = 32.0 * ((J2 + CG - 1) / CG) + drain;
          const double tW = passes * (32.0 * Rc + drain);
          const double tP = (double)(((long)J2 * Rc + nP - 1) / nP) * per_quad;
          double t = tH > tW ? tH : tW;
          if (tP > t) t = tP;
          total += t + per_quad + 64;  // pipeline fill / drain of a chunk
        }
        if (total < best.cost) best = Plan{R2, C2, nH, nW, nP, total, CG};
      }
    }
  }
  return best;
}

int plan_override(Plan* pl, int npairs, int S) {
  // options sggf_plan_r2 / sggf_plan_c2 pin the role split in pairs (tuning / tests)
  const int R2 = (int)get_option(kOptSggfPlanR2), C2 = (int)get_option(kOptSggfPlanC2);
  if (R2 < 1 || C2 < 1) return 0;
  if (R2 * S + C2 * S >= npairs) return 0;
  pl->R2 = R2;
  pl->C2 = C2;
  pl->CG = 1;
  pl->nH = R2 * S;
  pl->nW = C2 * S;
  pl->nP = npairs - pl->nH - pl->nW;
  return 1;
}

constexpr int kSlotsPerProducer = 4;  // double slots (two G tiles each) per producer CTA

template <bool kRow, bool kCol, bool kShared = false>
int resident_pairs(int* out) {
  // the shared-memory opt-in is a per-device attribute of the function, the occupancy a per-device number
  static int cached[64] = {0};
  static std::mutex mu;
  int dev = 0;
  PGICA_CUDA_OK(cudaGetDevice(&dev));
  PGICA_REQUIRE(dev >= 0 && dev < 64, "softmax_grad_gemm_dual: device ordinal %d out of range", dev);
  std::lock_guard<std::mutex> lock(mu);
  if (cached[dev] == 0) {
    auto kern = sggf_kernel<kRow, kCol, kShared>;
    PGICA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * 64);
    cfg.blockDim = dim3(block_threads(kRow, kCol));
    cfg.dynamicSmemBytes = kSmem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    PGICA_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 3) {
      set_error("softmax_grad_gemm_dual: only %d CTA pairs of this kernel fit on the device", n);
      return PGICA_ERR_CUDA;
    }
    cached[dev] = n;
  }
  *out = cached[dev];
  return PGICA_OK;
}

template <bool kRow, bool kCol, bool kShared = false>
int launch(const CUtensorMap& tm_x128, const CUtensorMap& tm_y128, const CUtensorMap& tm_x64,
           const CUtensorMap& tm_y64, const CUtensorMap& tm_s, const CUtensorMap& tm_ox, const CUtensorMap& tm_oy,
           const SggfParams& p, cudaStream_t st) {
  auto kern = sggf_kernel<kRow, kCol, kShared>;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * (p.nH + p.nW + p.nP)));
  cfg.blockDim = dim3(block_threads(kRow, kCol));
  cfg.dynamicSmemBytes = kSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeCooperative;  // all pairs co-resident or the launch fails: the roles wait on each other
  attr[1].val.cooperative = 1;
  cfg.attrs = attr;
  // The roles spin-wait on each other: every pair must be resident, which only a cooperative launch guarantees.  A
  // refused cooperative launch (SMs held by another context, MPS, a concurrent kernel) is therefore an ERROR, not
  // something to retry without the attribute.  Option sggf_coop = 0 selects a plain launch explicitly; it is also
  // the default when a profiler that cannot replay cooperative cluster launches was attached at load time.
  const bool coop = get_option(kOptSggfCoop) != 0;
  cfg.numAttrs = coop ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tm_x128, tm_y128, tm_x64, tm_y64, tm_s, tm_ox, tm_oy, p);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    set_error("softmax_grad_gemm_dual: %slaunch of %u CTAs failed: %s", coop ? "cooperative " : "", cfg.gridDim.x,
              cudaGetErrorString(e));
    return PGICA_ERR_CUDA;
  }
  count_launches(1);
  return PGICA_OK;
}

struct ProgressSpec {
  uint32_t* counters = nullptr;  // device, one uint32 per segment of OutY rows
  int64_t rows_per_segment = 0;  // multiple of 256 (a column pair)
};

template <bool kRow, bool kCol, bool kShared = false>
int plan_and_launch(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, SggfParams p, void* workspace,
                    size_t workspace_bytes, const ProgressSpec& pg, cudaStream_t st) {
  int npairs = 0;
  int rc = resident_pairs<kRow, kCol, kShared>(&npairs);
  if (rc != PGICA_OK) return rc;
  const int S = p.S;
  // a bf16 OutY cannot be accumulated over chunks: all of X must then fit one chunk of X-holders.  One chunk is also
  // taken, when it fits, with a progress counter (the rows of OutY then become final from the first pass on instead
  // of only during the last chunk: the overlapped all-reduce gets the whole launch to hide in) and with option
  // sggf_single_chunk = 1 (W streamed once, OutY written once: 325 MB instead of 825 MB of DRAM traffic on cfg2, for
  // ~2 % more time — measured 1.071 vs 1.051 ms, profiles/r2_dual_ab1.log).
  // column groups need an OutX that can be add-reduced: fp32
  const bool groups_ok = !p.outx_bf16 && get_option(kOptSggfColGroups) != 0;
  Plan pl = choose_plan(p.RB2, p.J2, (int)k, npairs, p.outy_bf16 != 0, groups_ok, kRow && kCol);
  if (pl.R2 < p.RB2 && (pg.counters != nullptr || get_option(kOptSggfSingleChunk) != 0)) {
    const Plan one = choose_plan(p.RB2, p.J2, (int)k, npairs, true, groups_ok, kRow && kCol);
    if (one.R2 >= p.RB2 && one.nP >= 1) pl = one;
  }
  plan_override(&pl, npairs, S);
  PGICA_REQUIRE(pl.R2 >= 1 && pl.nP >= 1, "softmax_grad_gemm_dual: no role split of %d CTA pairs fits %d row blocks%s",
                npairs, 2 * p.RB2, p.outy_bf16 ? " in one chunk (bf16 OutY)" : "");
  PGICA_REQUIRE(!(p.outy_bf16 && p.RB2 > pl.R2),
                "softmax_grad_gemm_dual: a bf16 OutY cannot be accumulated over chunks (x has %d row blocks)", 2 * p.RB2);
  if (pg.counters != nullptr) {
    PGICA_REQUIRE(pg.rows_per_segment > 0 && pg.rows_per_segment % (2 * kBT) == 0,
                  "softmax_grad_gemm_dual: rows_per_segment must be a positive multiple of 256 (got %lld)",
                  (long long)pg.rows_per_segment);
    p.progress = pg.counters;
    p.cp_per_seg = (int)(pg.rows_per_segment / (2 * kBT));
  }
  p.R2 = pl.R2;
  p.C2 = pl.C2;
  p.CG = pl.CG;
  if (const int64_t forced = get_option(kOptSggfColGroups); forced > 1 && !p.outx_bf16 && pl.R2 >= p.RB2 &&
                                                            pl.R2 * S * (int)forced + pl.nW < npairs && forced <= p.J2) {
    p.CG = (int)forced;  // option sggf_col_groups > 1 pins the group count (tests)
    pl.nH = pl.R2 * S * p.CG;
    pl.nP = npairs - pl.nH - pl.nW;
  }
  if (p.CG > 1)  // partial OutX sums of the groups are add-reduced into zeros
    PGICA_CUDA_OK(cudaMemsetAsync(p.out_x, 0, (size_t)mx * k * sizeof(float), st));
  p.nH = pl.nH;
  p.nW = pl.nW;
  p.nP = pl.nP;
  p.D = kSlotsPerProducer;
  p.spread = get_option(kOptSggfSpread) != 0 ? 1 : 0;
  p.debug_producers_only = get_option(kOptSggfProducersOnly) != 0 ? 1 : 0;
  {  // tuning: fewer exchange double-slots per producer CTA (8 was no faster than 4)
    const int v = (int)get_option(kOptSggfSlots);
    if (v >= 1 && v <= kSlotsPerProducer) p.D = v;
  }
  const size_t nslots = (size_t)2 * p.nP * p.D * 2;
  const size_t ring_bytes = nslots * kPBytes;
  const size_t flag_bytes = align_up(nslots * sizeof(uint32_t), 256);
  if (workspace_bytes < ring_bytes + 2 * flag_bytes) {
    set_error("softmax_grad_gemm_dual: workspace too small (%zu < %zu)", workspace_bytes, ring_bytes + 2 * flag_bytes);
    return PGICA_ERR_WORKSPACE_TOO_SMALL;
  }
  uint8_t* w = static_cast<uint8_t*>(workspace);
  p.ready = reinterpret_cast<uint32_t*>(w + ring_bytes);
  p.done = reinterpret_cast<uint32_t*>(w + ring_bytes + flag_bytes);
  PGICA_CUDA_OK(cudaMemsetAsync(p.ready, 0, 2 * flag_bytes, st));
  CUtensorMap tm_x128, tm_y128, tm_x64, tm_y64, tm_s;
  rc = make_tmap_bf16(&tm_x128, x, mx, k, k, 128);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y128, y, my, k, k, 128);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_x64, x, mx, k, k, 64);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y64, y, my, k, k, 64);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_s, workspace, nslots * kBM, kBT, kBT, 128);
  if (rc != PGICA_OK) return rc;
  // the outputs leave through TMA in boxes of 32 rows x 128 bytes
  CUtensorMap tm_ox, tm_oy;
  rc = p.outx_bf16 ? make_tmap_bf16(&tm_ox, p.out_x, mx, k, k, 32) : make_tmap_f32(&tm_ox, p.out_x, mx, k, k, 32);
  if (rc != PGICA_OK) return rc;
  rc = p.outy_bf16 ? make_tmap_bf16(&tm_oy, p.out_y, my, k, k, 32) : make_tmap_f32(&tm_oy, p.out_y, my, k, k, 32);
  if (rc != PGICA_OK) return rc;
  return launch<kRow, kCol, kShared>(tm_x128, tm_y128, tm_x64, tm_y64, tm_s, tm_ox, tm_oy, p, st);
}

}  // namespace

bool sggf_supported(int64_t mx, int64_t my, int64_t k) {
  // option sgg_fused = 0 falls back to one launch per product (sgg_x.cu)
  if (get_option(kOptSggFused) == 0) return false;
  return k % kNC == 0 && k / kNC <= 4 && mx >= 1 && my >= 1;
}

// true when x fits one chunk of X-holders, i.e. OutY is written once and may therefore be bf16
bool sggf_single_chunk(int64_t mx, int64_t my, int64_t k) {
  int npairs = 0;
  if (k % kNC != 0 || k / kNC > 4 || resident_pairs<true, false>(&npairs) != PGICA_OK) return false;
  const int RB2 = (int)((ceil_div(mx, kBM) + 1) / 2), J2 = (int)((ceil_div(my, kBT) + 1) / 2);
  Plan pl = choose_plan(RB2, J2, (int)k, npairs, true);
  return pl.R2 >= RB2 && pl.nP >= 1;
}

// Role split the planner picks for `npairs` resident CTA pairs (host arithmetic only; no device needed).
void sggf_plan(int64_t mx, int64_t my, int64_t k, int npairs, int single_chunk, int out[6]) {
  const int RB2 = (int)((ceil_div(mx, kBM) + 1) / 2), J2 = (int)((ceil_div(my, kBT) + 1) / 2);
  const Plan pl = choose_plan(RB2, J2, (int)k, npairs, (single_chunk & 1) != 0, (single_chunk & 2) != 0);
  out[5] = pl.CG;
  out[0] = pl.R2;
  out[1] = pl.C2;
  out[2] = pl.nH;
  out[3] = pl.nW;
  out[4] = pl.nP;
}

// Host replay of the kernel's schedule (the very enumerators the device code runs), for the CPU test-suite:
// role 0 = producers' view: out gets (q, row pair, column pair) per quad; role 1 / 2 = X- / Y-holder `idx`: out gets
// (q, sel, row pair, column pair, first, period) per pair-tile.  Returns the number of records (written up to `cap`).
int64_t sggf_schedule(int RB2, int J2, int R2, int C2, int spread, int role, int idx, int32_t* out, int64_t cap) {
  SggfParams p{};
  p.CG = spread >> 8;  // bits 8.. of `spread` carry the column-group count for the host replay (0 / 1 = none)
  spread &= 1;
  p.RB2 = RB2;
  p.J2 = J2;
  p.R2 = R2;
  p.C2 = C2;
  p.spread = spread;
  int64_t n = 0;
  if (role == 0) {
    // the producers' view, from the cursor the device code runs, cross-checked against the plain walk over all quads
    for_each_own_quad(p, 0, 1, [&](int q, int r0, int r, int c0, int c) {
      if (n < cap) {
        out[3 * n] = q;
        out[3 * n + 1] = r0 + r;
        out[3 * n + 2] = c0 + c;
      }
      ++n;
    });
    int64_t m = 0;
    bool same = true;
    for_each_quad(p, [&](int q, int r0, int r, int c0, int c) {
      if (m < cap && m < n) same &= out[3 * m] == q && out[3 * m + 1] == r0 + r && out[3 * m + 2] == c0 + c;
      ++m;
    });
    if (!same || m != n) return -2;
  } else {
    for_each_holder_tile(
        p, role == 2, idx,
        [&](int q, int sel, int rp, int cp, bool first, int period) {
          if (n < cap) {
            int32_t* o = out + 6 * n;
            o[0] = q;
            o[1] = sel;
            o[2] = rp;
            o[3] = cp;
            o[4] = first ? 1 : 0;
            o[5] = period;
          }
          ++n;
        },
        [&](int, int, int) {});
  }
  return n;
}

size_t sggf_workspace_bytes() {
  // exchange ring for the largest producer count (72 of 74 resident pairs) + flags
  const size_t nslots = (size_t)2 * 72 * kSlotsPerProducer * 2;
  return nslots * (size_t)kPBytes + 2 * align_up(nslots * sizeof(uint32_t), 256);
}

int sggf_dispatch(const void* x, const void* y, int64_t mx, int64_t my, int64_t k, const SoftmaxGradStats& stats,
                  void* out_x, int out_x_is_bf16, void* out_y, int out_y_is_bf16, void* workspace,
                  size_t workspace_bytes, cudaStream_t st, uint32_t* progress = nullptr, int64_t rows_per_segment = 0,
                  bool shared_exponential = false) {
  PGICA_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 255u) == 0,
                "softmax_grad_gemm_dual: workspace missing or not 256-byte aligned");
  ProgressSpec sc;
  sc.counters = progress;
  sc.rows_per_segment = rows_per_segment;
  const int RB = (int)ceil_div(mx, kBM), J = (int)ceil_div(my, kBT);
  PGICA_REQUIRE((int64_t)RB * J < (1ll << 30), "softmax_grad_gemm_dual: problem too large");
  SggfParams p{};
  p.mx = (int)mx;
  p.my = (int)my;
  p.k = (int)k;
  p.RB2 = (RB + 1) / 2;
  p.J2 = (J + 1) / 2;
  p.S = (int)(k / kNC);
  p.outx_bf16 = out_x_is_bf16;
  p.outy_bf16 = out_y_is_bf16;
  p.st = stats;
  p.out_x = out_x;
  p.out_y = out_y;
  const bool row = stats.r_lse != nullptr, col = stats.c_lse != nullptr;
  if (shared_exponential) {
    // see sggf_kernel: |logit| <= scale, 2 scale log2(e) < 100, mirrored targets — promised by the caller (heads.cu)
    PGICA_REQUIRE(row && col && stats.r_tgt && stats.c_tgt && bounded_logits(stats.c),
                  "softmax_grad_gemm_dual: shared exponential misused");
    return plan_and_launch<true, true, true>(x, y, mx, my, k, p, workspace, workspace_bytes, sc, st);
  }
  return with_terms(row, col, [&](auto r, auto c) {
    return plan_and_launch<decltype(r)::value, decltype(c)::value>(x, y, mx, my, k, p, workspace, workspace_bytes, sc,
                                                                    st);
  });
}

}  // namespace pgica

#ifdef PGICA_TRACE
extern "C" int pgica_debug_set_sggf_trace(void* buf) {
  long long* p = static_cast<long long*>(buf);
  return cudaMemcpyToSymbol(pgica::g_sggf_trace, &p, sizeof(p)) == cudaSuccess ? 0 : -1;
}
#endif

namespace pgica {
void sggf_plan(int64_t mx, int64_t my, int64_t k, int npairs, int single_chunk, int out[6]);
int64_t sggf_schedule(int RB2, int J2, int R2, int C2, int spread, int role, int idx, int32_t* out, int64_t cap);
}
extern "C" int64_t pgica_debug_dual_schedule(int row_pairs, int col_pairs, int row_pairs_per_chunk, int col_pairs_per_pass,
                                             int spread, int role, int idx, int32_t* out_host, int64_t capacity) {
  if (row_pairs < 1 || col_pairs < 1 || row_pairs_per_chunk < 1 || col_pairs_per_pass < 1 || role < 0 || role > 2 ||
      idx < 0 || !out_host || capacity < 0 || (spread >> 8) > 64)
    return -1;
  return pgica::sggf_schedule(row_pairs, col_pairs, row_pairs_per_chunk, col_pairs_per_pass, spread, role, idx, out_host,
                              capacity);
}
extern "C" int pgica_softmax_grad_gemm_dual_plan(int64_t mx, int64_t my, int64_t k, int npairs, int flags,
                                                 int32_t* plan_host) {
  const int single_chunk = flags;
  PGICA_REQUIRE(plan_host && mx > 0 && my > 0 && k > 0 && k % 512 == 0 && k / 512 <= 4 && npairs >= 3,
                "softmax_grad_gemm_dual_plan: bad argument");
  int out[6];
  pgica::sggf_plan(mx, my, k, npairs, single_chunk, out);
  for (int i = 0; i < 6; ++i) plan_host[i] = out[i];
  return PGICA_OK;
}

extern "C" int pgica_softmax_grad_gemm_dual_workspace_bytes(int64_t mx, int64_t my, int64_t k, size_t* bytes_host) {
  PGICA_REQUIRE(bytes_host, "workspace query: null result pointer");
  (void)mx;
  (void)my;
  (void)k;
  *bytes_host = pgica::sggf_workspace_bytes();
  return PGICA_OK;
}

namespace {
// Arguments both dual entry points take; `name` prefixes the error message.
int check_dual_args(const char* name, const void* x, const void* y, int64_t mx, int64_t my, int64_t k, float scale,
                    const float* r_lse, const float* r_coef, const float* c_lse, const float* c_coef, void* out_x,
                    void* out_y) {
  using namespace pgica;
  int rc = pgica_device_check();
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(x && y && out_x && out_y, "%s: null operand", name);
  PGICA_REQUIRE(mx > 0 && my > 0 && k > 0, "%s: bad shape (mx %lld my %lld k %lld)", name, (long long)mx, (long long)my,
                (long long)k);
  PGICA_REQUIRE(k % kNC == 0 && k / kNC <= 4, "%s: k must be 512, 1024, 1536 or 2048 (got %lld)", name, (long long)k);
  PGICA_REQUIRE(mx < (1ll << 30) && my < (1ll << 30), "%s: dimension too large", name);
  const bool row = r_lse != nullptr, col = c_lse != nullptr;
  PGICA_REQUIRE(row || col, "%s: need row statistics, column statistics or both", name);
  PGICA_REQUIRE(!row || r_coef, "%s: r_coef missing", name);
  PGICA_REQUIRE(!col || c_coef, "%s: c_coef missing", name);
  PGICA_REQUIRE(scale > 0.f, "%s: scale must be positive", name);
  return PGICA_OK;
}
}  // namespace

extern "C" int pgica_softmax_grad_gemm_dual(const void* x, const void* y, int64_t mx, int64_t my, int64_t k,
                                            float scale, const float* r_lse, const float* r_coef,
                                            const int32_t* r_tgt, const float* c_lse, const float* c_coef,
                                            const int32_t* c_tgt, void* out_x, int out_x_is_bf16, void* out_y,
                                            int out_y_is_bf16, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace pgica;
  const int rc = check_dual_args("softmax_grad_gemm_dual", x, y, mx, my, k, scale, r_lse, r_coef, c_lse, c_coef, out_x,
                                 out_y);
  if (rc != PGICA_OK) return rc;
  return sggf_dispatch(x, y, mx, my, k, {scale * kLog2e, r_lse, r_coef, r_tgt, c_lse, c_coef, c_tgt}, out_x,
                       out_x_is_bf16, out_y, out_y_is_bf16, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int pgica_softmax_grad_gemm_dual_progress(const void* x, const void* y, int64_t mx, int64_t my, int64_t k,
                                                     float scale, const float* r_lse, const float* r_coef,
                                                     const int32_t* r_tgt, const float* c_lse, const float* c_coef,
                                                     const int32_t* c_tgt, void* out_x, int out_x_is_bf16, void* out_y,
                                                     int out_y_is_bf16, uint32_t* progress, int64_t rows_per_segment,
                                                     int32_t* increments_per_256_rows_host, void* workspace,
                                                     size_t workspace_bytes, void* stream) {
  using namespace pgica;
  const int rc = check_dual_args("softmax_grad_gemm_dual_progress", x, y, mx, my, k, scale, r_lse, r_coef, c_lse,
                                 c_coef, out_x, out_y);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(progress, "softmax_grad_gemm_dual_progress: null progress counters");
  if (increments_per_256_rows_host) *increments_per_256_rows_host = 8 * (int32_t)(k / kNC);  // 2 CTAs x S splits x 4 drain warps
  return sggf_dispatch(x, y, mx, my, k, {scale * kLog2e, r_lse, r_coef, r_tgt, c_lse, c_coef, c_tgt}, out_x,
                       out_x_is_bf16, out_y, out_y_is_bf16, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream), progress, rows_per_segment);
}
