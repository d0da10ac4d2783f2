// sdw_gemm2.cu — persistent 2-CTA (cta_group::2) variant of the implicit-GEMM kernel.
//
// Why: a 128 x BN tile moves (128 + BN) * 128 B of operands per 64-deep K block for 2 * 128 * BN * 64 FLOP —
// 64-71 FLOP per L2 byte, which caps the whole chip near 40 % of tensor peak (profiles/r01_ncu_gemm_v1.md: LTS 33 % at
// tensor 34 %).  A CTA pair computes a 256 x BN tile with ONE tcgen05.mma.cta_group::2 (M = 256): each CTA stages its
// own 128 activation rows and only HALF of the weight tile, so operand bytes per FLOP drop by ~1.6-2x, and the
// accumulators of two consecutive tiles double-buffer in TMEM so the epilogue of tile i overlaps the mainloop of
// tile i+1 (persistent grid: one cluster per SM pair, static round-robin over tiles, N fastest so an activation tile leaves DRAM once).
//
//   warp 0 (both CTAs)  : TMA producer — own A tile [128 x 64] + own half of B [BN/2 x 64]; completion bytes are
//                         signalled on the LEADER's full barrier (cta_group::2 TMA, mapa'd barrier address).
//   warp 1 (leader)     : MMA issuer, 4 x UMMA(M=256, N=BN, K=16) per K block; tcgen05.commit multicast frees the
//                         smem stage in both CTAs / publishes the accumulator to both epilogues.
//   warp 2 (both CTAs)  : residual producer of the TMA epilogue (one thread; [128 x 32] chunks, two ring slots per chunk
//                         group c % EW).
//   warps 4.. (both)    : epilogue on the CTA's own 128 rows, EW = 2 or 4 warps per TMEM lane quarter (sdw_gemm_epi.cuh),
//                         then a remote arrive on the leader's tmem_empty barrier.
//
// Mainloop flavours (all in this kernel; chosen per GEMM by plan_gemm, sdw_gemm.cu):
//   per-tap      one activation box per (tap, channel chunk)              every conv / linear (the original form)
//   TR = 1       tap reuse: one (8+2)-row box per (channel chunk, kx) feeds the three ky taps      3x3 stride-1 convs
// (two more flavours were built, measured slower and removed again: the activation rows of an M pair kept resident
//  across its N tiles, and 4-CTA clusters with the activation tile TMA-multicast to two CTA pairs — profiles/
//  r01_epi_bench_a_stationary.txt, r01_gemm_shapes_cluster4_multicast.txt.)
// EW = epilogue warps per TMEM lane quarter.  EW = 2 (384 threads) everywhere; EW = 4 (640 threads, registers
// re-balanced with setmaxnreg) for the short-K GEMMs, whose tile time is set by the epilogue — ncu: the MMA issuer
// spins on tmem_empty and the TMA producer on the full ring while two epilogue warps per scheduler run at 0.44 IPC
// (profiles/r02_ncu_epilogue_shortk.md).
// Shared memory is carved at run time: [barriers 1 KB | operand ring | epilogue buffers]; the planner sizes the ring
// from what the chosen epilogue (classic: 16 KB, TMA: 40-72 KB, with 16 warps up to 112 KB) leaves of the 227 KB.
#include "sdw_gemm_epi.cuh"
#include "sdw_internal.h"
#include "sdw_ptx.cuh"

namespace sdw {

// warpgroup 0: producer, MMA, residual producer (+1 idle warp); then EW warpgroups of epilogue warps
template <int EW> struct G2Threads { static constexpr int value = 128 + 128 * EW; };
// EW = 4: the CTA's register pool is what it was launched with, 640 threads x 96 = 61440 (setmaxnreg.inc blocks until the
// pool has room — asking for 112 hung the kernel): 128 * 56 + 512 * 104 = 60416
static constexpr int G2_REGS_ROLE = 56, G2_REGS_EPI = 104;
static_assert(128 * G2_REGS_ROLE + 512 * G2_REGS_EPI <= 640 * 96, "setmaxnreg budget of the 640-thread kernel");
static constexpr int G2_A_STAGE = 128 * 64 * 2;

// NSUB = accumulators per activation tile: NSUB = 2 computes a 256 x (2*BN) tile per CTA pair — the A tile is pulled
// from L2 once for twice the columns (the kernel is L2->SM bandwidth bound: profiles/r01_mma_eff_vs_blockN.txt) at the
// price of single-buffered TMEM (2 * 2 * 160 > 512 columns), so it is used for long-K problems (3x3 convs) only.
//
// TR = 1 (tap reuse, 3x3 stride-1 convs on 16 x 8-pixel tiles): the kernel is bound by the operand bytes an SM ingests
// per K block (~41 B/clk/SM: profiles/r01_gemm_shapes_cluster4_multicast.txt), and the three ky taps of one kx read
// the same pixels shifted by whole image rows.  One TMA box of (8 + 2) rows x 16 px x 64 ch per (channel chunk, kx)
// therefore serves three taps: tap ky's A operand is the same shared-memory tile entered 16 rows (2 KB, swizzle-atom
// aligned) further down, so a pipeline stage is 20 KB of A + 3 weight tiles instead of 3 x 16 KB of A + 3 weight tiles.
static constexpr int G2_TR_BW = 16, G2_TR_BH = 8;
static constexpr int G2_A_STAGE_TR = (G2_TR_BH + 2) * G2_TR_BW * 128;
template <int BN, int NSUB, int TR = 0>
struct Gemm2Cfg {
  static constexpr int BH = BN / 2;
  static constexpr int B_SUB = BH * 128;           // one CTA's half of one BN-wide weight tile
  static constexpr int A_STAGE = TR ? G2_A_STAGE_TR : G2_A_STAGE;
  static constexpr int TAPS = TR ? 3 : 1;          // taps per pipeline stage
  static constexpr int B_STAGE = TAPS * NSUB * B_SUB;
  static constexpr int NBUF = (2 * NSUB * BN <= 512) ? 2 : 1;  // accumulator buffers in TMEM
  static constexpr int ACC_COLS = NSUB * BN;
  static constexpr int TMEM_COLS = NBUF * ACC_COLS <= 256 ? 256 : 512;
  // shared memory: [barriers 1 KB][nstages x A][nstages x B][epilogue buffers]; the planner sizes nstages from what the
  // chosen epilogue leaves (sdw_internal.h: G2_*), so the carve-up below is a run-time one
  static constexpr int MAX_STAGES = 8;
  static constexpr int SMEM_BYTES = G2_SMEM_DYN;
};

template <int BN, int NSUB, int EW, int TR = 0>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2Threads<EW>::value, 1)
    gemm2_tc_kernel(const __grid_constant__ GemmKParams p) {
  static_assert(EW == 2 || (EW == 4 && NSUB == 1), "four epilogue warps per lane quarter: TMA epilogue, one accumulator");
  constexpr int CL = 2;
  using Cfg = Gemm2Cfg<BN, NSUB, TR>;
  constexpr int A_STAGE = Cfg::A_STAGE;
  constexpr int NBUF = Cfg::NBUF;
  const int STAGES = p.nstages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty_bar = full_bar + Cfg::MAX_STAGES;
  uint64_t* tmem_full = empty_bar + Cfg::MAX_STAGES;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;               // [2]  (leader's copy is the one in use)
  uint64_t* res_full = tmem_empty + 2;                // [8]  residual ring (TMA epilogue): 2 * EW slots in use
  uint64_t* res_empty = res_full + 8;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(res_empty + 8);
  uint8_t* smem_a = smem + G2_BAR_BYTES;
  uint8_t* smem_b = smem_a + STAGES * A_STAGE;
  // epilogue buffers.  classic: 2 KB per warp; TMA: output slabs (EW = 2: two 2 KB slabs per warp, EW = 4: one),
  // 1 KB bias copy per warp, residual ring
  uint8_t* epi_stage = smem_b + STAGES * Cfg::B_STAGE;
  uint8_t* epi_bias = epi_stage + G2_EPI_OUT;
  uint8_t* res_ring = epi_bias + (EW / 2) * G2_EPI_BIAS;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // rank in the CTA pair (cluster of two)
  constexpr uint32_t lead_rank = 0;         // cluster rank of the pair's leader
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x / CL;
  const int nclusters = gridDim.x / CL;
  const int n_groups = p.n_tiles;
  const int total_tiles = p.m_pairs * n_groups;
  const int num_kb = TR ? 3 * p.kchunks : p.ntaps * p.kchunks;  // pipeline stages per tile

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.mapA[0]);
    tma_prefetch_desc(&p.mapB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 8 * EW);  // 4 * EW epilogue warps x 2 CTAs
    }
    for (int r = 0; r < 2 * EW; ++r) {
      mbar_init(&res_full[r], 1);
      mbar_init(&res_empty[r], 4);  // the four warps (one per TMEM lane quarter) of the chunk's group
    }
    if (p.epi_tma) {
      tma_prefetch_desc(&p.mapOut);
      if (p.resid) tma_prefetch_desc(&p.mapRes);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_ptr_smem, Cfg::TMEM_COLS);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  // (compute-sanitizer racecheck reports tcgen05.alloc's shared-memory write of the TMEM address against the read below
  // as a hazard — with or without an extra bar.sync here: it does not model the tensor-core unit's write; the cluster
  // barrier orders the two.  profiles/r02_sanitizer_racecheck.md)
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  auto tile_coords = [&](int t, int& x0, int& y0, int& b0, int& n0) {
    // N fastest: the n_tiles column tiles of one M pair run on neighbouring clusters at the same time, so the
    // activation tile is fetched from DRAM once and re-read from L2 (the whole weight matrix is L2-resident anyway)
    const int m_pair = fast_div(t, p.mg_ng);
    const int n_tile = t - m_pair * n_groups;
    const int m_tile = m_pair * 2 + static_cast<int>(rank);
    const int tb = fast_div(m_tile, p.mg_twh);
    const int rem = m_tile - tb * (p.tiles_w * p.tiles_h);
    const int th = fast_div(rem, p.mg_tw);
    const int tw = rem - th * p.tiles_w;
    x0 = tw * p.bw;
    y0 = th * p.bh;
    b0 = tb * p.bb;
    n0 = n_tile * (NSUB * BN);
  };

  // i-th tile of this cluster: t = cluster_id + i * nclusters (N fastest across clusters)
  auto tile_index = [&](int i, int& t) {
    t = cluster_id + i * nclusters;
    return t < total_tiles;
  };

  // EW = 4: registers re-balanced inside the two branches (they only meet again at the teardown) — the role warps need
  // few, the 16 epilogue warps take the rest
  if (warp < 4) {
  if (EW == 4) reg_dealloc<G2_REGS_ROLE>();
  if (warp == 0) {
    // =========================== TMA producer (both CTAs) ==========================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int t;
      for (int i = 0; tile_index(i, t); ++i) {
        int x0, y0, b0, n0;
        tile_coords(t, x0, y0, b0, n0);
        int tap = 0, kc = 0;  // per-tap mainloop: (tap, channel chunk) of K block kb, advanced without a division
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_expect_tx(&full_bar[stage], 2 * (A_STAGE + Cfg::B_STAGE));
          const uint32_t bar = mapa_rank(smem_u32(&full_bar[stage]), lead_rank);
          if (TR) {
            // stage = (channel chunk kc, column tap kx): one (bh+2)-row box + the weight tiles of taps (ky, kx), ky = 0..2
            const int kx = tap;  // tap reuse: `tap` counts the column tap kx = 0..2 of channel chunk kc
            tma_load_4d_2sm(&p.mapA[0], bar, smem_a + stage * A_STAGE, kc * 64, x0 + kx - 1, y0 - 1, b0);
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
              for (int sub = 0; sub < NSUB; ++sub)
                tma_load_4d_2sm(&p.mapB, bar, smem_b + stage * Cfg::B_STAGE + (ky * NSUB + sub) * Cfg::B_SUB,
                                ((ky * 3 + kx) * p.kchunks + kc) * 64, n0 + sub * BN + static_cast<int>(rank) * Cfg::BH, 0,
                                0);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
            if (++tap == 3) {
              tap = 0;
              ++kc;
            }
            continue;
          }
          tma_load_4d_2sm(&p.mapA[p.tap_map[tap]], bar, smem_a + stage * A_STAGE, kc * 64, x0 + p.tap_dx[tap],
                          y0 + p.tap_dy[tap], b0);
#pragma unroll
          for (int sub = 0; sub < NSUB; ++sub)
            tma_load_4d_2sm(&p.mapB, bar, smem_b + stage * Cfg::B_STAGE + sub * Cfg::B_SUB, kb * 64,
                            n0 + sub * BN + static_cast<int>(rank) * Cfg::BH, p.b_batched ? y0 : 0,
                            p.b_batched ? b0 : 0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
          if (++kc == p.kchunks) {
            kc = 0;
            ++tap;
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only) =======================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(256, BN);
      int stage = 0;
      uint32_t phase = 0;
      int t;
      for (int it = 0; tile_index(it, t); ++it) {
        const int a = it % NBUF;
        mbar_wait(&tmem_empty[a], ((it / NBUF) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_acc = tmem_base + a * Cfg::ACC_COLS;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = make_desc_k_sw128(smem_u32(smem_a + stage * A_STAGE));
          const uint64_t db = make_desc_k_sw128(smem_u32(smem_b + stage * Cfg::B_STAGE));
          if (TR) {
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
#pragma unroll
                for (int sub = 0; sub < NSUB; ++sub)
                  umma_f16_ss_2cta(tmem_acc + sub * BN, da + ky * ((G2_TR_BW * 128) >> 4) + 2 * k,
                                   db + (ky * NSUB + sub) * (Cfg::B_SUB >> 4) + 2 * k, idesc, (kb | ky | k) != 0 ? 1u : 0u);
              }
            }
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
#pragma unroll
              for (int sub = 0; sub < NSUB; ++sub)
                umma_f16_ss_2cta(tmem_acc + sub * BN, da + 2 * k, db + sub * (Cfg::B_SUB >> 4) + 2 * k, idesc,
                                 (kb | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit_2cta(&empty_bar[stage], 0b11);  // frees the stage in both CTAs
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_2cta(&tmem_full[a], 0b11);
      }
    }
  } else if (warp == 2) {
    // =========================== residual producer (TMA epilogue, both CTAs) =========
    // [128 rows x 32 columns] chunks of this CTA's residual tile, in chunk order; runs ahead of the epilogue by up to two
    // chunks per chunk group (2 * EW slots), across tile boundaries
    if (NSUB == 1 && p.epi_tma && p.resid && lane == 0) {
      uint32_t kq = 0;  // fills issued per chunk group, mod 4, two bits each
      int t;
      for (int i = 0; tile_index(i, t); ++i) {
        int x0, y0, b0, n0;
        tile_coords(t, x0, y0, b0, n0);
        const int nch = (max(0, min(BN, p.N - n0)) + 31) >> 5;
        for (int c = 0; c < nch; ++c) {
          const uint32_t g = static_cast<uint32_t>(c) & (EW - 1);  // chunk group: slots {g, g + EW}, filled alternately
          const uint32_t k = (kq >> (2 * g)) & 3u;
          kq = (kq & ~(3u << (2 * g))) | (((k + 1) & 3u) << (2 * g));
          const uint32_t slot = g + EW * (k & 1);
          mbar_wait(&res_empty[slot], ((k >> 1) & 1) ^ 1);
          mbar_expect_tx(&res_full[slot], G2_RES_STAGE);
          tma_load_4d(&p.mapRes, &res_full[slot], res_ring + slot * G2_RES_STAGE, n0 + c * 32, x0, y0, b0);
        }
      }
    }
  }
  } else {
    // =========================== epilogue (both CTAs, own 128 rows) ==================
    if (EW == 4) reg_alloc<G2_REGS_EPI>();
    EpiTmaState est;
    int t;
    for (int it = 0; tile_index(it, t); ++it) {
      int x0, y0, b0, n0;
      tile_coords(t, x0, y0, b0, n0);
      const int a = it % NBUF;
      // the EW warps of a lane quarter interleave 32-column chunks: EW times the loads / stores / math in flight
      if (EW == 4 || (NSUB == 1 && p.epi_tma)) {
        gemm_epilogue_tma<BN, EW>(p, tmem_base + a * Cfg::ACC_COLS, warp, lane, x0, y0, b0, n0, &tmem_full[a], (it / NBUF) & 1,
                                  (warp - 4) >> 2, epi_stage + (warp - 4) * (EW == 4 ? 2048 : 4096),
                                  reinterpret_cast<float*>(epi_bias + (warp - 4) * 1024), res_ring, res_full, res_empty, est);
      } else if (EW == 2) {
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub)
          gemm_epilogue<BN>(p, tmem_base + a * Cfg::ACC_COLS + sub * BN, warp, lane, x0, y0, b0, n0 + sub * BN,
                            &tmem_full[a], (it / NBUF) & 1, (warp - 4) >> 2, 2, epi_stage + (warp - 4) * 2048);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_rank(smem_u32(&tmem_empty[a]), lead_rank));
    }
    if (p.epi_tma && lane == 0) bulk_wait_group<0>();  // every output slab has reached global memory
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int NSUB, int EW, int TR>
static int launch2(const GemmLaunch& l, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    SDW_CUDA_OK(cudaFuncSetAttribute(gemm2_tc_kernel<BN, NSUB, EW, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Gemm2Cfg<BN, NSUB, TR>::SMEM_BYTES));
    attr = true;
  }
  gemm2_tc_kernel<BN, NSUB, EW, TR><<<l.grid, G2Threads<EW>::value, Gemm2Cfg<BN, NSUB, TR>::SMEM_BYTES, stream>>>(l.p);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// instantiations: BLOCK_N 128 / 160 / 192 / 256 x {per-tap, tap reuse} with one accumulator, 160 x 2 accumulators
// (per-tap); the wide epilogue (EW = 4) for the per-tap kernels with one accumulator (the short-K linears / 1x1 convs)
int launch_gemm2(const GemmLaunch& l, cudaStream_t stream) {
  const int key = l.bn * 1000 + l.nsub * 100 + l.ew * 10 + (l.tr ? 1 : 0);
  switch (key) {
    case 128120: return launch2<128, 1, 2, 0>(l, stream);
    case 160120: return launch2<160, 1, 2, 0>(l, stream);
    case 192120: return launch2<192, 1, 2, 0>(l, stream);
    case 256120: return launch2<256, 1, 2, 0>(l, stream);
    case 128140: return launch2<128, 1, 4, 0>(l, stream);
    case 160140: return launch2<160, 1, 4, 0>(l, stream);
    case 192140: return launch2<192, 1, 4, 0>(l, stream);
    case 256140: return launch2<256, 1, 4, 0>(l, stream);
    case 160220: return launch2<160, 2, 2, 0>(l, stream);
    case 128121: return launch2<128, 1, 2, 1>(l, stream);
    case 160121: return launch2<160, 1, 2, 1>(l, stream);
    case 192121: return launch2<192, 1, 2, 1>(l, stream);
    case 256121: return launch2<256, 1, 2, 1>(l, stream);
    default: break;
  }
  set_error("no CTA-pair kernel for this BLOCK_N / accumulators / epilogue width / tap reuse combination");
  return 1;
}

}  // namespace sdw
