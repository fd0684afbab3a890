// Persistent cluster form of the softmax-gradient GEMM (see sgg.cu for the maths).
//
// The C CTAs of a thread-block cluster own the C 256-column slices of one 128-row block of Out (resident in TMEM)
// and SHARE the recomputed G tiles, so the logits of a (128 x 128) tile are recomputed once per cluster.  Tile j
// is produced by CTA (j mod C): MMA1 -> Z in TMEM -> epilogue warps -> bf16 G tile.  How the tile reaches the other
// CTAs is the difference to sgg_cluster.cu: distributed shared memory moves ~20 B/cycle/SM on B200 (measured,
// tools/ubench.cu), so a 32 KB tile broadcast to 3 peers occupies the producer for ~5000 cycles and needs a
// dedicated 32 KB landing slot per producer in every CTA.  Here the producer writes the tile once with a TMA store
// into a small per-cluster exchange ring in global memory (S tiles x 32 KB per cluster, a few MB in total, reused
// every S tiles and therefore L2-resident), signals the cluster with mbarrier arrives, and every CTA pulls the tile
// through its ordinary TMA operand ring like any other operand.  No tile-sized matrix is ever materialised: the
// exchange ring holds at most S tiles per cluster at any time.  What this buys:
//   * the 4 x 32 KB landing slots disappear: the operand ring grows from 3 to 6 stages of 32 KB,
//   * the exchange latency drops from ~8000 to ~3000 cycles and no longer gates on "slot free in every CTA",
//   * the kernel can be persistent (clusters loop over row blocks), which matters for dW with its 393 row blocks.
// MMA1 runs with N = 256 (two G tiles at once: a 128 x N x 16 tcgen05.mma with shared-memory operands costs
// N/2 + 43 cycles, so N = 256 reaches 75 % of the tensor peak where N = 128 reaches 60 %).  A round = C such
// 256-wide tiles = 2C G tiles; a CTA issues MMA1 for its tile of round r, then the MMA2s of the 2C tiles of round
// r-1.  Between a Z tile being complete and its G tiles being needed lie a whole MMA2 phase and the next MMA1
// (~20000 cycles); the epilogue + exchange need ~10000, and the slack costs no shared memory because finished tiles
// wait in the exchange ring.
#include "common.h"
#include "sgg_tile.cuh"

#include <mutex>

namespace pgica {
namespace {

constexpr int kBM = 128;
constexpr int kBT = 128;
constexpr int kBD = 256;
constexpr int kBK = 64;
constexpr uint32_t kChunkBytes = 128 * kBK * 2;   // 16 KB: a [128][64] bf16 box
constexpr uint32_t kQ0BoxBytes = 32 * kBK * 2;    // 4 KB: a [32][64] bf16 box (rows 0..31 of a Y tile, MMA2 operand)
constexpr uint32_t kQ1BoxBytes = 96 * kBK * 2;    // 12 KB: a [96][64] bf16 box (rows 32..127)
constexpr uint32_t kPBytes = kBM * kBT * 2;       // 32 KB: one G tile
constexpr int kBT2 = 2 * kBT;                     // MMA1 covers two G tiles at once (N = 256: 75 % vs 60 % of peak)
constexpr uint32_t kStageBytes = kChunkBytes + 2 * kChunkBytes;  // 48 KB ring slot: X chunk + 256-row Y chunk
constexpr int kRing = 4;
constexpr int kXSlots = 16;  // exchange-ring depth in tiles (two rounds of a 4-CTA cluster)
constexpr int kThreads = 256;
constexpr uint32_t kTmemOut = 0, kTmemZ = 256;  // Out [0,256), Z [256,512) (single buffer, 256 columns)
constexpr size_t kSmem = 1024 + kRing * kStageBytes + kPBytes + 3 * kBT * 4 + 512;

#ifdef PGICA_TRACE
__device__ long long* g_sggx_trace = nullptr;
#endif

struct SggxParams {
  int mx, my, k, num_tiles, passes, num_items, ldo, out_bf16, prefetch_y;
  SoftmaxGradStats st;
  void* out;
};

// ---- PTX pieces only this kernel uses
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// tcgen05.commit that arrives on the same-offset barrier of every CTA in `mask`
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

template <int C, bool kRow, bool kCol>
__global__ void __launch_bounds__(kThreads, 1)
sggx_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_y,
            const __grid_constant__ CUtensorMap tm_y32, const __grid_constant__ CUtensorMap tm_y96,
            const __grid_constant__ CUtensorMap tm_s, const SggxParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* ring = smem;
  uint8_t* staging = smem + kRing * kStageBytes;  // this CTA's freshly produced G tile, source of the TMA store
  float* s_col = reinterpret_cast<float*>(staging + kPBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_col + 3 * kBT);
  uint64_t* empty_bar = full_bar + kRing;
  uint64_t* zfull_bar = empty_bar + kRing;   // [1] (+1 spare)
  uint64_t* zempty_bar = zfull_bar + 2;      // [1] (+1 spare)
  uint64_t* gready_bar = zempty_bar + 2;     // [kXSlots] tile in exchange slot s is complete in global memory
  uint64_t* gdone_bar = gready_bar + kXSlots;  // [kXSlots] every CTA has finished MMA2 on the tile in slot s
  uint64_t* outfull_bar = gdone_bar + kXSlots;
  uint64_t* outfree_bar = outfull_bar + 1;
  uint64_t* stfull_bar = outfree_bar + 1;   // staging holds a complete G tile (128 epilogue arrivals)
  uint64_t* stfree_bar = stfull_bar + 1;    // the TMA store has read staging: it may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stfree_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t q = cluster_ctarank();
  const int cluster_id = blockIdx.x / C;
  const int num_clusters = gridDim.x / C;
  const int num_kb = (p.k + kBK - 1) / kBK;
  const int J = p.num_tiles;       // G tiles (128 rows of Y each)
  const int J2 = (J + 1) / 2;      // MMA1 tiles (256 rows of Y each)
  const int rounds = (J2 + C - 1) / C;
  // This cluster's items (row block, pass), and its rounds numbered straight through all of them ("global rounds"):
  // MMA1 of global round R is followed by the MMA2s of global round R-1, across item boundaries too, so the tensor
  // pipe never idles while an Out slice is drained or the first Z tile of an item is turned into G.
  const int n_my = (p.num_items - cluster_id + num_clusters - 1) / num_clusters;
  const int T = n_my * rounds;
  const int xrow0 = cluster_id * kXSlots * kBM;  // first row of this cluster's exchange ring in the scratch matrix

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_y);
    tma_prefetch_desc(&tm_y32);
    tma_prefetch_desc(&tm_y96);
    tma_prefetch_desc(&tm_s);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kRing; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&zfull_bar[i], 1);
      mbar_init(&zempty_bar[i], 128);
    }
    for (int i = 0; i < kXSlots; ++i) {
      mbar_init(&gready_bar[i], 1);
      mbar_init(&gdone_bar[i], C);
    }
    mbar_init(outfull_bar, 1);
    mbar_init(outfree_bar, 128);
    mbar_init(stfull_bar, 128);
    mbar_init(stfree_bar, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // every CTA's barriers exist before anyone arrives on a peer's
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (whole warp, one elected lane)
    int slot = 0;
    uint32_t phase = 0;
    auto advance = [&]() {
      if (++slot == kRing) {
        slot = 0;
        phase ^= 1;
      }
    };
    LAP_DECL(9);
    for (int R = 0; R <= T; ++R) {
      {
        const int it = R / rounds, r = R - it * rounds;
        const int m_blk = (cluster_id + it * num_clusters) / p.passes;
        const int own2 = r * C + (int)q;
        if (R < T && own2 < J2) {
          // A large Y (the LM-head weight in dH) streams from HBM: one cluster in eight pulls the tile this CTA
          // needs two rounds from now into L2, so that nobody's ring stalls on a DRAM round trip.
          const int ahead = own2 + 2 * C;
          const bool pf = p.prefetch_y && ahead < J2 && (((own2 / C) ^ cluster_id) & 7) == 0;
          for (int kb = 0; kb < num_kb; ++kb) {
            LAP(0);
            mbar_wait(&empty_bar[slot], phase ^ 1);
            LAP(1);
            if (elect_one()) {
              mbar_expect_tx(&full_bar[slot], kStageBytes);
              uint8_t* dst = ring + slot * kStageBytes;
              tma_load_2d(dst, &tm_x, &full_bar[slot], kb * kBK, m_blk * kBM);
              tma_load_2d(dst + kChunkBytes, &tm_y, &full_bar[slot], kb * kBK, own2 * kBT2);
              tma_load_2d(dst + 2 * kChunkBytes, &tm_y, &full_bar[slot], kb * kBK, own2 * kBT2 + kBT);
              if (pf) {
                tma_prefetch_2d(&tm_y, kb * kBK, ahead * kBT2);
                tma_prefetch_2d(&tm_y, kb * kBK, ahead * kBT2 + kBT);
              }
            }
            __syncwarp();
            advance();
          }
        }
      }
      if (R >= 1) {
        {
          const int itp = (R - 1) / rounds, rp = (R - 1) - itp * rounds;
          const int item_p = cluster_id + itp * num_clusters;
          const int out_col0 = ((item_p - (item_p / p.passes) * p.passes) * C + (int)q) * kBD;
          const int gbase = itp * J;  // exchange-ring sequence number of tile 0 of that item
          const int t_end = min((rp + 1) * 2 * C, J);
          for (int t = rp * 2 * C; t < t_end; ++t) {
            const int g = gbase + t;
            const int xs = g % kXSlots;
            LAP(0);
            mbar_wait_cluster(&gready_bar[xs], (uint32_t)(g / kXSlots) & 1u);  // tile is complete in global memory
            LAP(3);
            mbar_wait(&empty_bar[slot], phase ^ 1);
            LAP(2);
            if (elect_one()) {
              // order the acquire above (generic proxy) before the async-proxy read of the tile below
              asm volatile("fence.proxy.async.global;" ::: "memory");
              // slot A: the G tile (32 KB) + rows 0..31 of Y[tile t, out_col0 .. +256) as four [32][64] boxes (16 KB)
              mbar_expect_tx(&full_bar[slot], kStageBytes);
              uint8_t* dst = ring + slot * kStageBytes;
              tma_load_2d(dst, &tm_s, &full_bar[slot], 0, xrow0 + xs * kBM);
              tma_load_2d(dst + kChunkBytes, &tm_s, &full_bar[slot], kBK, xrow0 + xs * kBM);
#pragma unroll
              for (int i = 0; i < 4; ++i)
                tma_load_2d(dst + kPBytes + i * kQ0BoxBytes, &tm_y32, &full_bar[slot], out_col0 + i * kBK, t * kBT);
            }
            __syncwarp();
            advance();
            LAP(0);
            mbar_wait(&empty_bar[slot], phase ^ 1);
            LAP(2);
            if (elect_one()) {
              // slot B: rows 32..127 of the same Y tile as four [96][64] boxes (48 KB)
              mbar_expect_tx(&full_bar[slot], kStageBytes);
              uint8_t* dst = ring + slot * kStageBytes;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                tma_load_2d(dst + i * kQ1BoxBytes, &tm_y96, &full_bar[slot], out_col0 + i * kBK, t * kBT + 32);
            }
            __syncwarp();
            advance();
          }
        }
      }
    }
    LAP(0);
    if (lane == 0) LAP_FLUSH(g_sggx_trace, 0, 4);
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, one elected lane)
    constexpr uint32_t idesc1 = make_idesc_bf16(kBM, kBT2, 0, 0);
    constexpr uint32_t idesc2 = make_idesc_bf16(kBM, kBD, 0, 1);
    const uint64_t desc_k = make_smem_desc(0, 16, 1024);              // K-major operand, start address 0
    const uint64_t desc_mn32 = make_smem_desc(0, kQ0BoxBytes, 1024);  // MN-major operand: 64-column chunks 4 KB apart
    const uint64_t desc_mn96 = make_smem_desc(0, kQ1BoxBytes, 1024);  // ... 12 KB apart
    constexpr uint16_t kAllCtas = (uint16_t)((1u << C) - 1u);
    int slot = 0;
    uint32_t phase = 0;
    auto advance = [&]() {
      if (++slot == kRing) {
        slot = 0;
        phase ^= 1;
      }
    };
    uint32_t zuse = 0;  // own MMA1 tiles issued so far (Z is a single 256-column buffer)
    LAP_DECL(9);
    for (int R = 0; R <= T; ++R) {
      {
        const int own2 = (R % rounds) * C + (int)q;
        if (R < T && own2 < J2) {
          LAP(0);
          mbar_wait(zempty_bar, (zuse & 1u) ^ 1u);  // the epilogue has read the previous Z tile out of TMEM
          LAP(1);
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + kTmemZ;
          for (int kb = 0; kb < num_kb; ++kb) {
            LAP(0);
            mbar_wait(&full_bar[slot], phase);
            LAP(2);
            tc_fence_after_sync();
            if (elect_one()) {
              const uint32_t x_addr = smem_u32(ring + slot * kStageBytes);
              const uint64_t da = desc_k | ((x_addr >> 4) & 0x3FFF);
              const uint64_t db = desc_k | (((x_addr + kChunkBytes) >> 4) & 0x3FFF);
#pragma unroll
              for (int k = 0; k < kBK / 16; ++k) umma_bf16_ss(d_tmem, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
              umma_commit(&empty_bar[slot]);
              if (kb == num_kb - 1) umma_commit(zfull_bar);
            }
            __syncwarp();
            advance();
          }
          ++zuse;
        }
      }
      if (R >= 1) {
        {
          const int itp = (R - 1) / rounds, rp = (R - 1) - itp * rounds;
          const int gbase = itp * J;
          const int t_end = min((rp + 1) * 2 * C, J);
          for (int t = rp * 2 * C; t < t_end; ++t) {
            if (t == 0 && itp > 0) {
              // the previous item's Out slice must have left TMEM before this item starts accumulating
              LAP(0);
              mbar_wait(outfree_bar, (uint32_t)(itp - 1) & 1u);
              LAP(1);
              tc_fence_after_sync();
            }
            LAP(0);
            mbar_wait(&full_bar[slot], phase);  // slot A: the G tile + the first 32 rows of the Y tile
            LAP(3);
            tc_fence_after_sync();
            const int aslot = slot;
            const uint32_t g_addr = smem_u32(ring + slot * kStageBytes);
            const uint64_t dg = desc_k | ((g_addr >> 4) & 0x3FFF);
            if (elect_one()) {
              const uint64_t dy = desc_mn32 | (((g_addr + kPBytes) >> 4) & 0x3FFF);
#pragma unroll
              for (int ks = 0; ks < 2; ++ks)  // K = 16 vocab rows per step, N = 256
                umma_bf16_ss(tmem_base + kTmemOut, dg + ks * 2, dy + ks * (16 * 128 >> 4), idesc2, (t | ks) != 0 ? 1u : 0u);
            }
            __syncwarp();
            advance();
            LAP(0);
            mbar_wait(&full_bar[slot], phase);  // slot B: rows 32..127 of the Y tile
            LAP(4);
            tc_fence_after_sync();
            if (elect_one()) {
              const uint32_t y_addr = smem_u32(ring + slot * kStageBytes);
              const uint64_t dy = desc_mn96 | ((y_addr >> 4) & 0x3FFF);
#pragma unroll
              for (int ks = 2; ks < 8; ++ks)
                umma_bf16_ss(tmem_base + kTmemOut, dg + (ks >> 2) * (kChunkBytes >> 4) + (ks & 3) * 2,
                             dy + (ks - 2) * (16 * 128 >> 4), idesc2, 1u);
              umma_commit(&empty_bar[slot]);
              umma_commit(&empty_bar[aslot]);
              // every CTA of the cluster learns that this CTA is done with exchange slot (gbase + t) % kXSlots
              umma_commit_mcast(&gdone_bar[(gbase + t) % kXSlots], kAllCtas);
            }
            __syncwarp();
            advance();
          }
          if (rp == rounds - 1) {  // that was the last round of an item: its Out slice is complete
            if (elect_one()) umma_commit(outfull_bar);
            __syncwarp();
          }
        }
      }
    }
    LAP(0);
    if (lane == 0) LAP_FLUSH(g_sggx_trace, 4, 5);
  } else if (warp == 3) {
    // ------------------------------------------------------------------ exchange warp
    // Takes each finished G tile from the staging buffer to the cluster: TMA store into the exchange ring, wait for
    // the store to complete, release it to every CTA.  Runs beside the epilogue warps, so the ~3000 cycles of store
    // completion + fences are off their critical path (they matter when k is small and the epilogue is the pace).
    uint32_t ntile = 0;
    LAP_DECL(9);
    for (int R = 0; R < T; ++R) {
      const int it = R / rounds, r = R - it * rounds;
      const int own2 = r * C + (int)q;
      if (own2 >= J2) continue;
      for (int half = 0; half < 2; ++half) {
        const int t = 2 * own2 + half;
        if (t >= J) break;
        const int g = it * J + t;
        const int xs = g % kXSlots;
        const int use = g / kXSlots;
        LAP(0);
        mbar_wait(stfull_bar, ntile & 1u);
        LAP(1);
        if (use > 0) mbar_wait_cluster(&gdone_bar[xs], (uint32_t)(use - 1) & 1u);  // nobody still reads slot xs
        LAP(2);
        if (lane == 0) {
          tma_store_2d(&tm_s, staging, 0, xrow0 + xs * kBM);
          tma_store_2d(&tm_s, staging + kChunkBytes, kBK, xrow0 + xs * kBM);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // staging has been read
          mbar_arrive(stfree_bar);
          asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the tile is complete in global memory
          // async-proxy writes ordered before one cluster-scope release fence, then relaxed arrives
          asm volatile("fence.proxy.async.global;" ::: "memory");
          asm volatile("fence.acq_rel.cluster;" ::: "memory");
#pragma unroll
          for (int c = 0; c < C; ++c)
            asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(
                             mapa_u32(smem_u32(&gready_bar[xs]), (uint32_t)c))
                         : "memory");
        }
        __syncwarp();
        LAP(3);
        ++ntile;
      }
    }
    LAP(0);
    if (lane == 0) LAP_FLUSH(g_sggx_trace, 18, 4);
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: Z -> G for this CTA's own tiles
    const int quarter = warp & 3;
    const int et = threadIdx.x - 128;
    const int row_in_blk = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t g_local = smem_u32(staging);
    uint32_t zuse = 0, ntile = 0;
    LAP_DECL(9);
    // Out slice of item number `itd` of this cluster: TMEM -> global, then hand TMEM back to the MMA warp
    auto drain_out = [&](int itd) {
      const int item_d = cluster_id + itd * num_clusters;
      const int m_blk_d = item_d / p.passes;
      const int ocol0 = ((item_d - m_blk_d * p.passes) * C + (int)q) * kBD;
      const int row_d = m_blk_d * kBM + row_in_blk;
      LAP(0);
      mbar_wait(outfull_bar, (uint32_t)itd & 1u);
      LAP(5);
      tc_fence_after_sync();
#pragma unroll 1
      for (int ch = 0; ch < kBD / 32; ++ch) {
        uint32_t rr[32];
        tmem_ld_32x32(tmem_base + lane_addr + kTmemOut + ch * 32, rr);
        tmem_ld_wait();
        const int col = ocol0 + ch * 32;
        if (row_d < p.mx) store_out_chunk<false>(p.out, p.out_bf16, p.ldo, row_d, col, p.k, rr);
      }
      tc_fence_before_sync();
      mbar_arrive(outfree_bar);
    };
    int row = 0;
    float rl = 0.f, rc = 0.f, nl = 0.f, nc = 0.f;
    int rt = -1, nt = -1, gbase = 0;
    auto load_col = [&](int j, float& l, float& cf, int& tg) {
      const int col = j * kBT + et;
      load_col_stat<kCol>(p.st, col, j < J && col < p.my, l, cf, tg);
    };
    for (int R = 0; R < T; ++R) {
      const int it = R / rounds, r = R - it * rounds;
      if (r == 0) {  // a new item: its row block's statistics
        const int m_blk = (cluster_id + it * num_clusters) / p.passes;
        row = m_blk * kBM + row_in_blk;
        gbase = it * J;
        load_row_stat<kRow>(p.st, row, row < p.mx, rl, rc, rt);
        load_col(2 * (int)q, nl, nc, nt);  // column statistics of the first G tile this CTA produces
      }
      {
        const int own2 = r * C + (int)q;
        if (own2 < J2) {

        LAP(0);
        mbar_wait(zfull_bar, zuse & 1u);
        ++zuse;
        LAP(1);
        tc_fence_after_sync();
        for (int half = 0; half < 2; ++half) {
          const int t = 2 * own2 + half;  // G tile index
          if (t >= J) break;
          const bool last_half = (half == 1) || (t + 1 >= J);
          if (kCol) {
            stage_col_stat<false>(s_col, et, nl, nc, nt, p.st.c);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            load_col((half == 0 && t + 1 < J) ? t + 1 : 2 * (own2 + C), nl, nc, nt);  // next G tile of this CTA
          }
          const int rrel = rt - t * kBT;
          uint32_t gp[kBT / 2];  // this thread's row of the G tile as bf16 pairs
#pragma unroll
          for (int ch = 0; ch < kBT / 32; ++ch) {
            uint32_t rr[32];
            tmem_ld_32x32(tmem_base + lane_addr + kTmemZ + half * kBT + ch * 32, rr);
            tmem_ld_wait();
            float g[32];
            g_chunk<kRow, kCol>(rr, p.st.c, rl, rc, 0.f, row, rrel, s_col, ch, g);
            pack_g_chunk(g, gp + ch * 16);
          }
          if (last_half) {
            tc_fence_before_sync();
            mbar_arrive(zempty_bar);  // the Z tile has been read: the next MMA1 of this CTA may overwrite it
          }
          LAP(2);
          mbar_wait(stfree_bar, (ntile & 1u) ^ 1u);  // the exchange warp's TMA store has read the previous tile
          LAP(3);
#pragma unroll
          for (int ch = 0; ch < kBT / 32; ++ch) store_g_chunk(g_local, row_in_blk, ch, gp + ch * 16);
          fence_proxy_async_smem();  // generic-proxy writes -> visible to the async proxy (the TMA store reads them)
          mbar_arrive(stfull_bar);   // hand the tile to the exchange warp
          ++ntile;
          if (kCol) asm volatile("bar.sync 3, 128;" ::: "memory");  // the column statistics may be overwritten
          LAP(4);
        }
        }
      }
      // the MMA2s of the previous item's last round were issued right after this round's MMA1: drain that item now
      if (r == 0 && it > 0) drain_out(it - 1);
    }
    drain_out(n_my - 1);
    LAP(0);
    if (et == 0) LAP_FLUSH(g_sggx_trace, 9, 9);
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // no CTA may exit while a peer can still arrive on its barriers
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

template <int C, bool kRow, bool kCol>
int max_clusters(int* out) {
  static int cached_dev[64] = {0};
  static std::mutex mu;
  int dev = 0;
  PGICA_CUDA_OK(cudaGetDevice(&dev));
  PGICA_REQUIRE(dev >= 0 && dev < 64, "softmax_grad_gemm: device ordinal %d out of range", dev);
  std::lock_guard<std::mutex> lock(mu);
  int& cached = cached_dev[dev];
  if (cached == 0) {
    auto kern = sggx_kernel<C, kRow, kCol>;
    PGICA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(C * 64));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kSmem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    PGICA_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n <= 0) {
      set_error("softmax_grad_gemm: no %d-CTA cluster of this kernel fits on the device", C);
      return PGICA_ERR_CUDA;
    }
    cached = n;
  }
  *out = cached;
  return PGICA_OK;
}

template <int C, bool kRow, bool kCol>
int launch(const CUtensorMap& tm_x, const CUtensorMap& tm_y, const CUtensorMap& tm_y32, const CUtensorMap& tm_y96,
           const void* scratch,
           size_t scratch_bytes, const SggxParams& p, cudaStream_t st) {
  int resident = 0;
  int rc = max_clusters<C, kRow, kCol>(&resident);
  if (rc != PGICA_OK) return rc;
  const int64_t by_ws = (int64_t)(scratch_bytes / ((size_t)kXSlots * kPBytes));
  int64_t clusters = p.num_items < resident ? p.num_items : resident;
  if (by_ws < clusters) clusters = by_ws;
  PGICA_REQUIRE(clusters >= 1, "softmax_grad_gemm: exchange workspace too small (%zu bytes)", scratch_bytes);
  CUtensorMap tm_s;
  rc = make_tmap_bf16(&tm_s, scratch, (uint64_t)clusters * kXSlots * kBM, kBT, kBT, 128);
  if (rc != PGICA_OK) return rc;
  auto kern = sggx_kernel<C, kRow, kCol>;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(clusters * C));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PGICA_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tm_x, tm_y, tm_y32, tm_y96, tm_s, p));
  count_launches(1);
  return PGICA_OK;
}

}  // namespace

#ifdef PGICA_TRACE
extern "C" int pgica_debug_set_sggx_trace(void* buf) {
  long long* p = static_cast<long long*>(buf);
  return cudaMemcpyToSymbol(g_sggx_trace, &p, sizeof(p)) == cudaSuccess ? 0 : -1;
}
#endif

// Upper bound of the exchange workspace any launch of this kernel uses (64 resident clusters x ring).
size_t sggx_workspace_bytes() { return (size_t)64 * kXSlots * kPBytes; }

// Called by pgica_softmax_grad_gemm when k is a multiple of 256*C.  Returns PGICA_OK or an error code.
int sggx_dispatch(int cluster, const void* x, const void* y, int64_t mx, int64_t my, int64_t k,
                  const SoftmaxGradStats& stats, void* out, int out_is_bf16, void* workspace, size_t workspace_bytes,
                  cudaStream_t st) {
  PGICA_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 127u) == 0,
                "softmax_grad_gemm: exchange workspace missing or not 128-byte aligned");
  SggxParams p{};
  p.mx = (int)mx;
  p.my = (int)my;
  p.k = (int)k;
  p.num_tiles = (int)ceil_div(my, kBT);
  p.passes = (int)(k / (kBD * cluster));
  const int64_t items = ceil_div(mx, kBM) * p.passes;
  PGICA_REQUIRE(items < (1ll << 24) && items * p.num_tiles < (1ll << 31), "softmax_grad_gemm: problem too large");
  p.num_items = (int)items;
  p.ldo = (int)k;
  p.out_bf16 = out_is_bf16;
  p.prefetch_y = (my * k * 2 > (int64_t)(32 << 20)) ? 1 : 0;  // only an operand that cannot sit in L2
  p.st = stats;
  p.out = out;
  CUtensorMap tm_x, tm_y, tm_y32, tm_y96;
  int rc = make_tmap_bf16(&tm_x, x, mx, k, k, 128);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y, y, my, k, k, 128);
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y32, y, my, k, k, 32);  // MMA2 operand, rows 0..31 of a tile (shares a slot with G)
  if (rc != PGICA_OK) return rc;
  rc = make_tmap_bf16(&tm_y96, y, my, k, k, 96);  // MMA2 operand, rows 32..127 (a slot of its own)
  if (rc != PGICA_OK) return rc;
  if (cluster == 2 || cluster == 4)
    return with_terms(stats.r_lse != nullptr, stats.c_lse != nullptr, [&](auto r, auto c) {
      constexpr bool kRow = decltype(r)::value, kCol = decltype(c)::value;
      return cluster == 2 ? launch<2, kRow, kCol>(tm_x, tm_y, tm_y32, tm_y96, workspace, workspace_bytes, p, st)
                          : launch<4, kRow, kCol>(tm_x, tm_y, tm_y32, tm_y96, workspace, workspace_bytes, p, st);
    });
  set_error("softmax_grad_gemm: unsupported cluster size %d", cluster);
  return PGICA_ERR_INVALID_ARGUMENT;
}

}  // namespace pgica
