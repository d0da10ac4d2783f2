// sdw_attn.cu — fused (flash) attention on tcgen05 for the UNet's self- and cross-attention
// (the SDPA inside `BasicTransformerBlock`, reached from stable_diffusion_pipeline.py:418).
//
//   O[b, q, h*d:(h+1)*d] = softmax(Q_h K_h^T * d^-1/2) V_h          per (batch b, head h), fp16 in / fp16 out
//
// Nothing but Q, K, V^T tiles and the O tile touches HBM.  Two kernels:
//
// attn_pp_kernel  (head dim <= 64, more than one KV tile: every self-attention of SD-1.x at 64x64 / SD-2.1)
//   Persistent CTA, one per SM, working on TWO 128-query tiles (A, B) of one (b, h) at a time against a shared K / V^T
//   ring.  Warp roles: TMA producer; one MMA-issuing warp per query tile; one softmax warpgroup per query tile (thread =
//   query row).  Per KV tile and query tile:  S = Q K^T (M=128, N=128, fp32 in TMEM)  ->  the softmax warpgroup pulls the
//   whole score row into registers with ONE pass of tcgen05.ld and immediately hands the S columns back (s_free), so
//   S_{j+1} is computed while the exponentials of tile j run — the S -> softmax -> P -> PV hand-off that capped the
//   one-tile kernel at 62 % MUFU occupancy (profiles/r01_ncu_attn_lazy.md) is off the critical path; row max first, then
//   exponentials against a lazily updated reference max (O is rescaled in TMEM only when a row max moves by more than
//   2^8), P written back to tensor memory as fp16 pairs and O += P V issued as a TS-mode MMA.  The two warpgroups share each
//   scheduler's MUFU pipe (one ex2 per score, 16 / clk / SM — the bound of this kernel at head dim 40), so one tile's
//   exponentials fill the other's TMEM-load / row-max / barrier gaps.  Registers are re-balanced with setmaxnreg (softmax
//   224, rest 48), and one exponential pair in four is evaluated on the FMA pipe (Cody-Waite + degree-3 polynomial), which
//   takes a quarter of the load off the MUFU.  Self-attention 64x64, d = 40, batch 60: 2249 us (0.33 of the burst tensor
//   peak, 1.26x the all-MUFU exponential floor) against 2383 us with every exponential on the MUFU and 2991 us for the
//   one-tile kernel (profiles/r02_attn_ab_matrix.txt, r02_attn_softmax_loop_ab_same_box.txt).  Single-KV-tile (cross)
//   attention with >= 2 query tiles runs here too (155.6 vs 193.1 us at 64x64, 77 keys).
//
// attn_fwd_kernel  (everything else: single-KV-tile cross attention with a query-tile loop, head dims 80 / 160)
//   One CTA = one 128-query tile of one (b, h) (several tiles in turn when all keys fit one KV tile):
//   warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 online softmax (thread = query row) with the same lazy
//   reference max; P in tensor memory (TS-mode PV) for head dims <= 80, in shared memory for 160.
// Ordering is carried by mbarriers only.
#include "sdw_internal.h"
#include "sdw_ptx.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace sdw {

static constexpr int ATT_THREADS = 192;
static constexpr int ATT_BQ = 128;

struct alignas(64) AttnKParams {
  CUtensorMap mapQ, mapK, mapV;
  int Nq, Nk, d, heads;
  int dk_steps;          // ceil(d / 16)
  float scale_log2e;     // d^-1/2 * log2(e)
  __half* out;
  int64_t out_ld;
  int qt_per_cta;        // attn_fwd_kernel: query tiles per CTA (> 1 only when all keys fit one KV tile)
  int qpairs, total_work;  // attn_pp_kernel: 256-row query blocks per (b, h); work items = B * heads * qpairs
  long long* dbg;        // attn_pp_kernel: optional clock64 trace of CTA 0 (tools/attn_trace.py), else nullptr
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 2^t for two values on the FMA pipe (Cody-Waite: floor by a round-down magic add, degree-3 minimax polynomial on the
// fraction — relative error 7.5e-5, a sixth of the fp16 rounding P gets anyway — exponent spliced in with one integer
// multiply-add per value).  Takes a share of the exponentials off the MUFU pipe, which bounds this kernel.
__device__ __forceinline__ void ex2_poly2(float t0, float t1, float& e0, float& e1) {
  t0 = fmaxf(t0, -126.f);
  t1 = fmaxf(t1, -126.f);
  const uint64_t magic = pk2(12582912.f, 12582912.f);
  const uint64_t t = pk2(t0, t1);
  uint64_t xr;
  asm("add.rm.f32x2 %0, %1, %2;" : "=l"(xr) : "l"(t), "l"(magic));
  uint64_t fl, f;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(fl) : "l"(xr), "l"(magic));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(f) : "l"(t), "l"(fl));
  uint64_t q = fma2(f, pk2(0.0780244991f, 0.0780244991f), pk2(0.2260671854f, 0.2260671854f));
  q = fma2(q, f, pk2(0.6958335042f, 0.6958335042f));
  q = fma2(q, f, pk2(0.9999251962f, 0.9999251962f));
  float q0, q1, r0, r1;
  upk2(q, q0, q1);
  upk2(xr, r0, r1);
  e0 = __int_as_float(__float_as_int(r0) * 8388608 + __float_as_int(q0));
  e1 = __int_as_float(__float_as_int(r1) * 8388608 + __float_as_int(q1));
}

// =============================================================================================
// attn_pp_kernel
// =============================================================================================
// Variants of this kernel that were built, measured on a B200 and removed again (evidence: profiles/r02_attn_*.txt,
// DESIGN.md §4): two softmax threads per query row (four warps per scheduler: 2941 vs 2633 us at batch 60), a token that
// makes the MUFU bursts of the two query tiles alternate (2558 vs 2528 us), a double-buffered-score version with BKV = 96
// and P written in place (3411 us), exponentials partly on the FMA pipe on top of it (3449 / 3720 us); on the shipped
// two-tile kernel, same box, cycles under ncu (profiles/r02_attn_softmax_loop_ab_same_box.txt): the row max fused into
// the exponential pass (4.69 M vs 4.43 M cycles) and PV_{j-1} awaited only after the first chunk's exponentials (4.57 M).
// What did pay: one exponential pair in four as a degree-3 polynomial on the FMA pipe (4.18 M cycles, 2249 us).
template <int DVP>
struct PPCfg {
  static constexpr int ST = 4;                       // K / V^T ring depth
  static constexpr int THREADS = 384;                // warpgroup 0: warp 0 TMA, warp 1 MMA(A), warp 2 MMA(B), warp 3 idle;
                                                     // warpgroup 1: softmax of query tile A; warpgroup 2: of query tile B
  static constexpr int Q_BYTES = ATT_BQ * 128;       // one 128 x 64 fp16 tile, SWIZZLE_128B
  static constexpr int K_STAGE = 128 * 128;          // BKV = 128 keys x 64 (zero-filled head dim) fp16
  static constexpr int V_STAGE = 2 * DVP * 128;      // V^T: two 64-key boxes of DVP rows
  static constexpr int SMEM = 2 * Q_BYTES + ST * (K_STAGE + V_STAGE) + 1024 + 512;
  // tensor memory (512 columns, one CTA per SM): S_A S_B | P_A P_B | O_A O_B
  static constexpr int S_COL = 0, P_COL = 256, O_COL = 384;
  static constexpr int REGS_SOFTMAX = 224, REGS_OTHER = 48;
  static_assert(DVP <= 64 && DVP % 16 == 0, "head dim <= 64");
  static_assert(128 * REGS_OTHER + 256 * REGS_SOFTMAX <= 65536 - 1024, "register file (an exact fit hung setmaxnreg.inc on hardware: keep slack)");
};


// TRACE: compile the clock64 stamps in (tools/attn_trace.py); the shipped instantiation carries no trace code — with the
// stamps merely predicated off the kernel was 8 % slower
template <int DVP, int TRACE>
__global__ void __launch_bounds__(PPCfg<DVP>::THREADS, 1) attn_pp_kernel(const __grid_constant__ AttnKParams p) {
  using Cfg = PPCfg<DVP>;
  constexpr int ST = Cfg::ST, BKV = 128;
  constexpr int NCH = BKV / 32;                     // 32-column chunks of a score row
  constexpr uint32_t GROUP = 128;                   // softmax threads per query tile
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* q_smem = smem;                          // [2][Q_BYTES]
  uint8_t* k_smem = q_smem + 2 * Cfg::Q_BYTES;     // [ST][K_STAGE]
  uint8_t* v_smem = k_smem + ST * Cfg::K_STAGE;    // [ST][V_STAGE]
  uint64_t* bars = reinterpret_cast<uint64_t*>(v_smem + ST * Cfg::V_STAGE);
  uint64_t* q_full = bars;            // [2] TMA -> MMA(X)
  uint64_t* q_empty = q_full + 2;     // [2] MMA(X) commit -> TMA: every S of this work item has completed
  uint64_t* kv_full = q_empty + 2;    // [ST] TMA -> both MMA warps
  uint64_t* kv_empty = kv_full + ST;  // [ST] PV_A(j) and PV_B(j) commits (count 2) -> TMA
  uint64_t* s_full = kv_empty + ST;   // [2] MMA(X) commit -> softmax(X)
  uint64_t* s_free = s_full + 2;      // [2] softmax(X) (GROUP) -> MMA(X): the score rows sit in registers
  uint64_t* p_ready = s_free + 2;     // [2] softmax(X) (GROUP) -> MMA(X): P_j is in tensor memory
  uint64_t* pv_done = p_ready + 2;    // [2] MMA(X) commit -> softmax(X): P columns / O accumulator free
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(pv_done + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (p.Nk + BKV - 1) / BKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.mapQ);
    tma_prefetch_desc(&p.mapK);
    tma_prefetch_desc(&p.mapV);
    for (int x = 0; x < 2; ++x) {
      mbar_init(&q_full[x], 1);
      mbar_init(&q_empty[x], 1);
      mbar_init(&s_full[x], 1);
      mbar_init(&s_free[x], GROUP);
      mbar_init(&p_ready[x], GROUP);
      mbar_init(&pv_done[x], 1);
    }
    for (int s = 0; s < ST; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 2);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;

  if (warp < 4) {
    reg_dealloc<Cfg::REGS_OTHER>();
    if (warp == 0) {
      // ============================ TMA producer ============================================
      if (elect_one_sync()) {  // one lane, and ptxas knows it: no per-instruction uniformity loops around tcgen05.mma
        int kvc = 0, wi = 0;
        for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++wi) {
          const int qp = w % p.qpairs, head = (w / p.qpairs) % p.heads, b = w / (p.qpairs * p.heads);
          for (int x = 0; x < 2; ++x) {
            if (wi > 0) mbar_wait(&q_empty[x], (wi - 1) & 1);
            mbar_expect_tx(&q_full[x], Cfg::Q_BYTES);
            tma_load_4d(&p.mapQ, &q_full[x], q_smem + x * Cfg::Q_BYTES, 0, qp * 2 * ATT_BQ + x * ATT_BQ, head, b);
          }
          for (int j = 0; j < ntiles; ++j, ++kvc) {
            const int s = kvc % ST;
            mbar_wait(&kv_empty[s], ((kvc / ST) & 1) ^ 1);
            mbar_expect_tx(&kv_full[s], Cfg::K_STAGE + Cfg::V_STAGE);
            tma_load_4d(&p.mapK, &kv_full[s], k_smem + s * Cfg::K_STAGE, 0, j * BKV, head, b);
            tma_load_4d(&p.mapV, &kv_full[s], v_smem + s * Cfg::V_STAGE, j * BKV, 0, head, b);
            tma_load_4d(&p.mapV, &kv_full[s], v_smem + s * Cfg::V_STAGE + DVP * 128, j * BKV + 64, 0, head, b);
          }
        }
      }
    } else if (warp <= 2) {
      // ============================ MMA issuer of query tile X ===============================
      if (elect_one_sync()) {  // one lane, and ptxas knows it: no per-instruction uniformity loops around tcgen05.mma
        const int X = warp - 1;
        constexpr uint32_t idesc_s = make_idesc_f16(ATT_BQ, BKV);
        constexpr uint32_t idesc_o = make_idesc_f16(ATT_BQ, DVP);
        const uint32_t q_addr = smem_u32(q_smem + X * Cfg::Q_BYTES);
        const uint32_t t_s = tmem + Cfg::S_COL + X * 128;
        const uint32_t t_p = tmem + Cfg::P_COL + X * 64;
        const uint32_t t_o = tmem + Cfg::O_COL + X * 64;
        int kvc = 0, gt = 0, wi = 0;  // KV tiles consumed (ring position), tiles of THIS pipeline, work items
        auto issue_s = [&](int kv) {
          const int s = kv % ST;
          mbar_wait(&kv_full[s], (kv / ST) & 1);
          tc_fence_after();
          const uint32_t k_addr = smem_u32(k_smem + s * Cfg::K_STAGE);
          for (int ks = 0; ks < p.dk_steps; ++ks)
            umma_f16_ss(t_s, make_desc_k_sw128(q_addr + ks * 32), make_desc_k_sw128(k_addr + ks * 32), idesc_s,
                        ks != 0 ? 1u : 0u);
          umma_commit(&s_full[X]);
        };
        for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++wi) {
          mbar_wait(&q_full[X], wi & 1);
          tc_fence_after();
          if (gt > 0) {  // the last score tile of the previous work item has been pulled into registers
            mbar_wait(&s_free[X], (gt - 1) & 1);
            tc_fence_after();
          }
          issue_s(kvc);
          for (int j = 0; j < ntiles; ++j) {
            if (j + 1 < ntiles) {
              mbar_wait(&s_free[X], (gt + j) & 1);
              tc_fence_after();
              issue_s(kvc + j + 1);
            } else {
              umma_commit(&q_empty[X]);  // every S of this work item has been issued: Q may be refilled once they complete
            }
            mbar_wait(&p_ready[X], (gt + j) & 1);
            tc_fence_after();
            const int s = (kvc + j) % ST;
            const uint32_t v_addr = smem_u32(v_smem + s * Cfg::V_STAGE);
#pragma unroll
            for (int ks = 0; ks < BKV / 16; ++ks) {
              const uint64_t db = make_desc_k_sw128(v_addr + (ks >> 2) * (DVP * 128) + (ks & 3) * 32);
              umma_f16_ts(t_o, t_p + ks * 8, db, idesc_o, (j | ks) != 0 ? 1u : 0u);
            }
            umma_commit(&pv_done[X]);
            umma_commit(&kv_empty[s]);
          }
          kvc += ntiles;
          gt += ntiles;
        }
      }
    }
  } else {
    // ============================ softmax / correction / epilogue of query tile X ==============
    reg_alloc<Cfg::REGS_SOFTMAX>();
    const int X = (warp >> 2) - 1;   // query tile
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t t_s = tmem + lane_base + Cfg::S_COL + X * 128;
    const uint32_t t_p = tmem + lane_base + Cfg::P_COL + X * 64;
    const uint32_t t_o = tmem + lane_base + Cfg::O_COL + X * 64;
    const float sl2 = p.scale_log2e;
    const bool trace = TRACE && p.dbg != nullptr && blockIdx.x == 0 && r == 0;
    constexpr float LAZY_LOG2 = 8.f;
    int gt = 0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
      const int qp = w % p.qpairs, head = (w / p.qpairs) % p.heads, b = w / (p.qpairs * p.heads);
      float m_ref = -INFINITY, l_run = 0.f;
      for (int j = 0; j < ntiles; ++j, ++gt) {
        long long ts0 = 0, ts1 = 0, ts2 = 0, ts3 = 0;
        if (trace) ts0 = clock64();
        mbar_wait(&s_full[X], gt & 1);
        tc_fence_after();
        if (trace) ts1 = clock64();
        // ---- this thread's score columns into registers, then give the S columns back -----------
        uint32_t v[NCH][32];
#pragma unroll
        for (int c = 0; c < NCH; ++c) tmem_ld_32x32(t_s + c * 32, v[c]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&s_free[X]);
        if (trace) ts2 = clock64();
        const int kv0 = j * BKV;
        if (kv0 + BKV > p.Nk) {  // ragged last tile: keys >= Nk do not exist
#pragma unroll
          for (int i = 0; i < BKV; ++i)
            if (kv0 + i >= p.Nk) v[i >> 5][i & 31] = 0xff800000u;  // -inf
        }
        // ---- row max, lazy reference update ------------------------------------------------------
        float m_t;
        {
          float mx[NCH];
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            float a0 = __uint_as_float(v[c][0]), a1 = __uint_as_float(v[c][1]);
#pragma unroll
            for (int i = 2; i < 32; i += 2) {
              a0 = fmaxf(a0, __uint_as_float(v[c][i]));
              a1 = fmaxf(a1, __uint_as_float(v[c][i + 1]));
            }
            mx[c] = fmaxf(a0, a1);
          }
          m_t = mx[0];
#pragma unroll
          for (int c = 1; c < NCH; ++c) m_t = fmaxf(m_t, mx[c]);
        }
        bool pv_waited = (j == 0);  // tile 0: the epilogue of the previous work item has waited for its last PV
        if (j == 0) {
          m_ref = m_t;
        } else if (__any_sync(0xffffffffu, (m_t - m_ref) * sl2 > LAZY_LOG2)) {
          // exact online-softmax step for this warp's rows: new reference, O and l rescaled (rare after the first tiles)
          const float m_new = fmaxf(m_ref, m_t);
          const float alpha = ex2f((m_ref - m_new) * sl2);
          m_ref = m_new;
          l_run *= alpha;
          mbar_wait(&pv_done[X], (gt - 1) & 1);  // PV_{j-1} has completed: O is stable, the P columns are free
          tc_fence_after();
          pv_waited = true;
#pragma unroll
          for (int c = 0; c < DVP / 16; ++c) {
            uint32_t o[16];
            tmem_ld_32x16(t_o + c * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x16(t_o + c * 16, o);
          }
          tmem_st_wait();
        }
        if (trace) ts3 = clock64();
        // ---- exponentials against the reference max, P -> tensor memory chunk by chunk.  One pair in four goes through
        //      the FMA pipe: same box, batch 60: 4.18 M cycles against 4.43 M with every exponential on the MUFU
        //      (profiles/r02_attn_softmax_loop_ab_same_box.txt) ----------------------------------------------------------
        const float mb = m_ref * sl2;
        const uint64_t sl2_2 = pk2(sl2, sl2), nmb_2 = pk2(-mb, -mb);
        uint64_t sm2[4] = {pk2(0.f, 0.f), pk2(0.f, 0.f), pk2(0.f, 0.f), pk2(0.f, 0.f)};
        if (!pv_waited) {
          mbar_wait(&pv_done[X], (gt - 1) & 1);  // PV_{j-1} has read P_{j-1}: the P columns may be overwritten
          tc_fence_after();
        }
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          uint32_t pkc[16];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float t0, t1, t2, t3, e0, e1, e2, e3;
            upk2(fma2(pk2(__uint_as_float(v[c][i]), __uint_as_float(v[c][i + 1])), sl2_2, nmb_2), t0, t1);
            upk2(fma2(pk2(__uint_as_float(v[c][i + 2]), __uint_as_float(v[c][i + 3])), sl2_2, nmb_2), t2, t3);
            e0 = ex2f(t0);
            e1 = ex2f(t1);
            if ((i >> 2) % 4 == 3) {
              ex2_poly2(t2, t3, e2, e3);  // this pair on the FMA pipe
            } else {
              e2 = ex2f(t2);
              e3 = ex2f(t3);
            }
            sm2[(i >> 1) & 3] = add2(sm2[(i >> 1) & 3], pk2(e0, e1));
            sm2[((i >> 1) + 1) & 3] = add2(sm2[((i >> 1) + 1) & 3], pk2(e2, e3));
            pkc[i >> 1] = pack_h2(e0, e1);
            pkc[(i >> 1) + 1] = pack_h2(e2, e3);
          }
          tmem_st_32x16(t_p + c * 16, pkc);  // row = lane, column k = keys (2k, 2k+1) as an fp16 pair (TS-mode A layout)
        }
        float sum_t;
        {
          float s0, s1, s2, s3, s4, s5, s6, s7;
          upk2(sm2[0], s0, s1);
          upk2(sm2[1], s2, s3);
          upk2(sm2[2], s4, s5);
          upk2(sm2[3], s6, s7);
          sum_t = ((s0 + s1) + (s2 + s3)) + ((s4 + s5) + (s6 + s7));
        }
        l_run += sum_t;
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&p_ready[X]);
        if (trace) {
          long long* o = p.dbg + (static_cast<long long>(X) * 4096 + (gt & 4095)) * 8;
          o[0] = ts0; o[1] = ts1; o[2] = ts2; o[3] = ts3; o[4] = ts3; o[5] = ts3; o[6] = clock64();
        }
      }
      // ---- epilogue: O / l -> fp16 ------------------------------------------------------------
      mbar_wait(&pv_done[X], (gt - 1) & 1);
      tc_fence_after();
      const float inv_l = 1.f / l_run;
      const int row = qp * 2 * ATT_BQ + X * ATT_BQ + r;
      __half* orow = p.out + (static_cast<int64_t>(b) * p.Nq + row) * p.out_ld + head * p.d;
      const bool vec_ok = ((p.out_ld & 7) == 0) && ((p.d & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
#pragma unroll
      for (int c = 0; c < DVP / 16; ++c) {
        uint32_t o[16];
        tmem_ld_32x16(t_o + c * 16, o);
        tmem_ld_wait();
        if (row < p.Nq) {
#pragma unroll
          for (int h8 = 0; h8 < 2; ++h8) {
            const int dd = c * 16 + h8 * 8;
            if (dd >= p.d) break;
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(o[h8 * 8 + i]) * inv_l;
            if (vec_ok && dd + 8 <= p.d) {
              uint4 u;
              u.x = pack_h2(f[0], f[1]);
              u.y = pack_h2(f[2], f[3]);
              u.z = pack_h2(f[4], f[5]);
              u.w = pack_h2(f[6], f[7]);
              *reinterpret_cast<uint4*>(orow + dd) = u;
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (dd + i < p.d) orow[dd + i] = __float2half_rn(f[i]);
            }
          }
        }
      }
      // the next work item's first PV overwrites O (accumulate = 0) only after this tile's next p_ready, which every
      // softmax thread of the tile signals after this read-out: no separate "O free" barrier is needed
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// =============================================================================================
// attn_fwd_kernel
// =============================================================================================
// SB = number of S accumulator buffers: 2 (double-buffered, one CTA per SM) or 1 (TMEM 256 columns and <= 113 KB of
// shared memory, so TWO CTAs share an SM)
// PT = 1: P stays in tensor memory (BKV / 2 extra columns, fp16 pairs) and PV runs as a TS-mode MMA: no P tile in
// shared memory, no generic->async proxy fence, half the shared-memory traffic per KV tile.
template <int DKA, int DVP, int BKV, int ST, int SB, int PT>
struct AttnCfg {
  static constexpr int Q_BYTES = DKA * ATT_BQ * 128;
  static constexpr int K_STAGE = DKA * BKV * 128;
  static constexpr int V_STAGE = (BKV / 64) * DVP * 128;
  static constexpr int P_BYTES = PT ? 0 : (BKV / 64) * ATT_BQ * 128;
  static constexpr int SMEM = Q_BYTES + P_BYTES + ST * (K_STAGE + V_STAGE) + 1024 + 256;
  static constexpr int P_COL = SB * BKV;                       // PT: P_j as packed fp16 pairs
  static constexpr int NEED = SB * BKV + DVP + (PT ? BKV / 2 : 0);
  static constexpr int TMEM_COLS = NEED <= 128 ? 128 : (NEED <= 256 ? 256 : 512);
  static constexpr int NCTA = SMEM <= 64 * 1024 && TMEM_COLS <= 128 ? 3 : (SMEM <= 114 * 1024 && TMEM_COLS <= 256 ? 2 : 1);  // CTAs per SM
  static constexpr int O_COL = SB * BKV + (PT ? BKV / 2 : 0);
  static_assert(NEED <= TMEM_COLS, "TMEM budget");
};

template <int DKA, int DVP, int BKV, int ST, int SB, int PT>
__global__ void __launch_bounds__(ATT_THREADS, AttnCfg<DKA, DVP, BKV, ST, SB, PT>::NCTA)
    attn_fwd_kernel(const __grid_constant__ AttnKParams p) {
  using Cfg = AttnCfg<DKA, DVP, BKV, ST, SB, PT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* q_smem = smem;
  uint8_t* p_smem = q_smem + Cfg::Q_BYTES;
  uint8_t* k_smem = p_smem + Cfg::P_BYTES;
  uint8_t* v_smem = k_smem + ST * Cfg::K_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(v_smem + ST * Cfg::V_STAGE);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;
  uint64_t* kv_empty = kv_full + ST;
  uint64_t* s_full = kv_empty + ST;  // [2]
  uint64_t* p_ready = s_full + 2;
  uint64_t* pv_done = p_ready + 1;
  uint64_t* q_empty = pv_done + 1;  // query-tile loop: Q smem free (S of this tile issued and complete)
  uint64_t* o_free = q_empty + 1;   //                  O accumulator read out by the epilogue
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(o_free + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = blockIdx.y, b = blockIdx.z;
  const int ntiles = (p.Nk + BKV - 1) / BKV;
  // query tiles of this CTA; tile t of the CTA is tile (g0 + j) of every barrier's phase sequence (nqt > 1 => ntiles == 1)
  const int qt_first = blockIdx.x * p.qt_per_cta;
  const int nqt = min(p.qt_per_cta, (p.Nq + ATT_BQ - 1) / ATT_BQ - qt_first);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.mapQ);
    tma_prefetch_desc(&p.mapK);
    tma_prefetch_desc(&p.mapV);
    mbar_init(q_full, 1);
    for (int s = 0; s < ST; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    mbar_init(&s_full[0], 1);
    mbar_init(&s_full[1], 1);
    mbar_init(p_ready, 128);
    mbar_init(pv_done, 1);
    mbar_init(q_empty, 1);
    mbar_init(o_free, 128);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;

  if (warp == 0) {
    // ============================ TMA producer ============================================
    if (elect_one_sync()) {
      for (int t = 0; t < nqt; ++t) {
        const int q0 = (qt_first + t) * ATT_BQ;
        if (t > 0) mbar_wait(q_empty, (t - 1) & 1);
        mbar_expect_tx(q_full, Cfg::Q_BYTES);
#pragma unroll
        for (int a = 0; a < DKA; ++a) tma_load_4d(&p.mapQ, q_full, q_smem + a * (ATT_BQ * 128), a * 64, q0, head, b);
        if (t > 0) continue;  // single KV tile: K / V^T stay resident
        for (int j = 0; j < ntiles; ++j) {
          const int s = j % ST;
          mbar_wait(&kv_empty[s], ((j / ST) & 1) ^ 1);
          mbar_expect_tx(&kv_full[s], Cfg::K_STAGE + Cfg::V_STAGE);
          const int kv0 = j * BKV;
#pragma unroll
          for (int a = 0; a < DKA; ++a)
            tma_load_4d(&p.mapK, &kv_full[s], k_smem + s * Cfg::K_STAGE + a * (BKV * 128), a * 64, kv0, head, b);
#pragma unroll
          for (int a = 0; a < BKV / 64; ++a)
            tma_load_4d(&p.mapV, &kv_full[s], v_smem + s * Cfg::V_STAGE + a * (DVP * 128), kv0 + a * 64, 0, head, b);
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ================================================
    if (elect_one_sync()) {
      constexpr uint32_t idesc_s = make_idesc_f16(ATT_BQ, BKV);
      constexpr uint32_t idesc_o = make_idesc_f16(ATT_BQ, DVP);
      const uint32_t q_addr = smem_u32(q_smem);
      const uint32_t p_addr = smem_u32(p_smem);
      int g0 = 0;  // tiles issued by earlier query tiles of this CTA
      auto issue_s = [&](int j) {
        const int s = j % ST;
        mbar_wait(&kv_full[s], (j / ST) & 1);
        tc_fence_after();
        const uint32_t k_addr = smem_u32(k_smem + s * Cfg::K_STAGE);
        const uint32_t ts = tmem + ((g0 + j) % SB) * BKV;
        for (int ks = 0; ks < p.dk_steps; ++ks) {
          const uint64_t da = make_desc_k_sw128(q_addr + (ks >> 2) * (ATT_BQ * 128) + (ks & 3) * 32);
          const uint64_t db = make_desc_k_sw128(k_addr + (ks >> 2) * (BKV * 128) + (ks & 3) * 32);
          umma_f16_ss(ts, da, db, idesc_s, ks != 0 ? 1u : 0u);
        }
        umma_commit(&s_full[(g0 + j) % SB]);
      };
      for (int t = 0; t < nqt; ++t) {
        g0 = t * ntiles;
        mbar_wait(q_full, t & 1);
        tc_fence_after();
        issue_s(0);
        if (SB == 2 && ntiles > 1) issue_s(1);
        if (nqt > 1) umma_commit(q_empty);  // Q smem may be refilled once S of this (only) KV tile has completed
        if (t > 0) {
          mbar_wait(o_free, (t - 1) & 1);  // the previous query tile's epilogue has read O out
          tc_fence_after();
        }
        for (int j = 0; j < ntiles; ++j) {
          mbar_wait(p_ready, (g0 + j) & 1);
          tc_fence_after();
          // single S buffer: the softmax has consumed S_j (p_ready), so S_{j+1} goes first and overlaps PV_j
          if (SB == 1 && j + 1 < ntiles) issue_s(j + 1);
          const int s = j % ST;
          const uint32_t v_addr = smem_u32(v_smem + s * Cfg::V_STAGE);
#pragma unroll
          for (int ks = 0; ks < BKV / 16; ++ks) {
            const uint64_t db = make_desc_k_sw128(v_addr + (ks >> 2) * (DVP * 128) + (ks & 3) * 32);
            if (PT) {
              umma_f16_ts(tmem + Cfg::O_COL, tmem + Cfg::P_COL + ks * 8, db, idesc_o, (j | ks) != 0 ? 1u : 0u);
            } else {
              const uint64_t da = make_desc_k_sw128(p_addr + (ks >> 2) * (ATT_BQ * 128) + (ks & 3) * 32);
              umma_f16_ss(tmem + Cfg::O_COL, da, db, idesc_o, (j | ks) != 0 ? 1u : 0u);
            }
          }
          umma_commit(pv_done);
          umma_commit(&kv_empty[s]);
          if (SB == 2 && j + 2 < ntiles) issue_s(j + 2);
        }
      }
    }
  } else {
    // ============================ softmax / correction / epilogue ============================
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t t_o = tmem + lane_base + Cfg::O_COL;
    const float sl2 = p.scale_log2e;
    uint8_t* p_row = p_smem + r * 128;
    const int sw = r & 7;
    for (int t = 0; t < nqt; ++t) {
      const int q0 = (qt_first + t) * ATT_BQ;
      const int g0 = t * ntiles;
      float m_run = -INFINITY, l_run = 0.f;

      // Two softmax paths per KV tile (the "lazy rescale" idea):
      //  fast : exponentials are taken against the row's REFERENCE max m_run (the true running max as of the last slow
      //         tile) instead of this tile's max, so nothing depends on a whole-row reduction: 32-column TMEM loads are
      //         software-pipelined against the MUFU / FMA work of the previous chunk, and O is never rescaled.  P values
      //         may exceed 1, by at most 2^LAZY_LOG2 — harmless in fp16 P / fp32 sums since every term shares m_run.
      //  slow : the exact online-softmax update (true max, O rescale in TMEM).  Taken for tile 0, for ragged tiles, and
      //         — warp-uniformly — whenever any row's tile max exceeds its reference by more than 2^LAZY_LOG2
      //         (S_j is still intact in TMEM, so the tile is simply re-read).
      constexpr float LAZY_LOG2 = 8.f;
      uint32_t pk[BKV / 2];  // P_j of this row, packed fp16 pairs

      for (int j = 0; j < ntiles; ++j) {
        mbar_wait(&s_full[(g0 + j) % SB], ((g0 + j) / SB) & 1);
        tc_fence_after();
        const uint32_t t_s = tmem + lane_base + ((g0 + j) % SB) * BKV;
        const int kv0 = j * BKV;
        const bool ragged = kv0 + BKV > p.Nk;
        bool need_slow = (j == 0) || ragged;
        bool p_stored = false;  // PT: the fast path has already put P_j into tensor memory
        float alpha = 1.f;

        if (!need_slow) {
          // ---------------- fast path: chunk-pipelined, reference max ----------------
          const float mb = m_run * sl2;
          const uint64_t sl2_2 = pk2(sl2, sl2), nmb_2 = pk2(-mb, -mb);
          uint64_t sm2[2] = {pk2(0.f, 0.f), pk2(0.f, 0.f)};
          float mx[2] = {-INFINITY, -INFINITY};
          uint32_t va[32], vb[32];
          tmem_ld_32x32(t_s, va);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < BKV / 32; ++c) {
            uint32_t(&cur)[32] = (c & 1) ? vb : va;
            uint32_t(&nxt)[32] = (c & 1) ? va : vb;
            if (c + 1 < BKV / 32) tmem_ld_32x32(t_s + (c + 1) * 32, nxt);  // in flight while this chunk is exponentiated
            uint32_t pkc[16];
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              const float x0 = __uint_as_float(cur[i]), x1 = __uint_as_float(cur[i + 1]);
              mx[0] = fmaxf(mx[0], x0);
              mx[1] = fmaxf(mx[1], x1);
              float t0, t1;
              upk2(fma2(pk2(x0, x1), sl2_2, nmb_2), t0, t1);
              const float e0 = ex2f(t0), e1 = ex2f(t1);
              sm2[(i >> 1) & 1] = add2(sm2[(i >> 1) & 1], pk2(e0, e1));
              if (PT) pkc[i >> 1] = pack_h2(e0, e1);
              else pk[c * 16 + (i >> 1)] = pack_h2(e0, e1);
            }
            if (PT) {
              // P chunks go to tensor memory as they are produced (the store overlaps the next chunk's exponentials and
              // the row never holds all 64 packed registers); the P columns are free once PV_{j-1} has completed
              if (c == 0 && j > 0) {
                mbar_wait(pv_done, (g0 + j - 1) & 1);
                tc_fence_after();
              }
              tmem_st_32x16(tmem + lane_base + Cfg::P_COL + c * 16, pkc);
            }
            if (c + 1 < BKV / 32) tmem_ld_wait();
          }
          const float m_t = fmaxf(mx[0], mx[1]);
          need_slow = __any_sync(0xffffffffu, (m_t - m_run) * sl2 > LAZY_LOG2);
          p_stored = PT && !need_slow;
          if (!need_slow) {
            float s0, s1, s2, s3;
            upk2(sm2[0], s0, s1);
            upk2(sm2[1], s2, s3);
            l_run += (s0 + s1) + (s2 + s3);
          }
        }
        if (need_slow) {
          // ---------------- slow path: exact online softmax ----------------
          float v[BKV];
          {
            uint32_t vu[BKV / 32][32];
#pragma unroll
            for (int c = 0; c < BKV / 32; ++c) tmem_ld_32x32(t_s + c * 32, vu[c]);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < BKV; ++i) v[i] = __uint_as_float(vu[i / 32][i % 32]);
          }
          if (ragged) {
#pragma unroll
            for (int i = 0; i < BKV; ++i)
              if (kv0 + i >= p.Nk) v[i] = -INFINITY;
          }
          float mx[4] = {v[0], v[1], v[2], v[3]};
#pragma unroll
          for (int i = 4; i < BKV; ++i) mx[i & 3] = fmaxf(mx[i & 3], v[i]);
          const float m_t = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
          const float m_new = fmaxf(m_run, m_t);
          alpha = ex2f((m_run - m_new) * sl2);
          const float mb = m_new * sl2;
          const uint64_t sl2_2 = pk2(sl2, sl2), nmb_2 = pk2(-mb, -mb);
          uint64_t sm2[2] = {pk2(0.f, 0.f), pk2(0.f, 0.f)};
#pragma unroll
          for (int i = 0; i < BKV; i += 2) {
            float t0, t1;
            upk2(fma2(pk2(v[i], v[i + 1]), sl2_2, nmb_2), t0, t1);
            const float e0 = ex2f(t0), e1 = ex2f(t1);
            sm2[(i >> 1) & 1] = add2(sm2[(i >> 1) & 1], pk2(e0, e1));
            pk[i >> 1] = pack_h2(e0, e1);
          }
          float s0, s1, s2, s3;
          upk2(sm2[0], s0, s1);
          upk2(sm2[1], s2, s3);
          l_run = fmaf(l_run, alpha, (s0 + s1) + (s2 + s3));
          m_run = m_new;
        }
        if (j > 0) {
          // P smem and the O accumulator are free once PV_{j-1} has completed
          mbar_wait(pv_done, (g0 + j - 1) & 1);
          tc_fence_after();
          if (need_slow && __any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll
            for (int c = 0; c < DVP / 16; ++c) {
              uint32_t o[16];
              tmem_ld_32x16(t_o + c * 16, o);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
              tmem_st_32x16(t_o + c * 16, o);
            }
            tmem_st_wait();
          }
        }
        if (PT) {
          // P_j -> tensor memory: row = this thread's lane, column c = keys (2c, 2c+1) as an fp16 pair (the TS-mode A layout)
          if (!p_stored) {
            const uint32_t t_p = tmem + lane_base + Cfg::P_COL;
#pragma unroll
            for (int c = 0; c < BKV / 32; ++c) {
              uint32_t w[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) w[i] = pk[c * 16 + i];
              tmem_st_32x16(t_p + c * 16, w);
            }
          }
          tmem_st_wait();
        } else {
          // P_j -> shared memory, K-major SWIZZLE_128B: 16-byte chunk c of row r lives at chunk (c ^ (r & 7))
#pragma unroll
          for (int c8 = 0; c8 < BKV / 8; ++c8) {
            uint4 u;
            u.x = pk[c8 * 4 + 0];
            u.y = pk[c8 * 4 + 1];
            u.z = pk[c8 * 4 + 2];
            u.w = pk[c8 * 4 + 3];
            *reinterpret_cast<uint4*>(p_row + (c8 >> 3) * (ATT_BQ * 128) + (((c8 & 7) ^ sw) << 4)) = u;
          }
          fence_proxy_async_smem();
        }
        tc_fence_before();
        mbar_arrive(p_ready);
      }
      // ---- epilogue: O / l -> fp16 ------------------------------------------------------------
      mbar_wait(pv_done, (g0 + ntiles - 1) & 1);
      tc_fence_after();
      const float inv_l = 1.f / l_run;
      const int row = q0 + r;
      __half* orow = p.out + (static_cast<int64_t>(b) * p.Nq + row) * p.out_ld + head * p.d;
      const bool vec_ok = ((p.out_ld & 7) == 0) && ((p.d & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
#pragma unroll
      for (int c = 0; c < DVP / 16; ++c) {
        uint32_t o[16];
        tmem_ld_32x16(t_o + c * 16, o);
        tmem_ld_wait();
        if (row < p.Nq) {
#pragma unroll
          for (int h8 = 0; h8 < 2; ++h8) {
            const int dd = c * 16 + h8 * 8;
            if (dd >= p.d) break;
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(o[h8 * 8 + i]) * inv_l;
            if (vec_ok && dd + 8 <= p.d) {
              uint4 u;
              u.x = pack_h2(f[0], f[1]);
              u.y = pack_h2(f[2], f[3]);
              u.z = pack_h2(f[4], f[5]);
              u.w = pack_h2(f[6], f[7]);
              *reinterpret_cast<uint4*>(orow + dd) = u;
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (dd + i < p.d) orow[dd + i] = __float2half_rn(f[i]);
            }
          }
        }
      }
      if (nqt > 1) {  // O has been read out: the MMA warp may start the next query tile's PV
        tc_fence_before();
        mbar_arrive(o_free);
      }
    }  // query tiles
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, Cfg::TMEM_COLS);
  }
}

// =============================================================================================
// host
// =============================================================================================
// variants: 0..3 attn_fwd_kernel, head dim <= 16 / 32 / 48 / 64 (BKV 128, P in TMEM, two CTAs per SM)
//           4    attn_fwd_kernel, head dim <= 80  (BKV 64, P in TMEM)
//           5    attn_fwd_kernel, head dim <= 160 (BKV 64, double-buffered S, P in shared memory)
//           8..11 attn_pp_kernel, head dim <= 16 / 32 / 48 / 64, more than one KV tile
struct AttnLaunchImpl {
  AttnKParams p;
  dim3 grid;
  int variant;
};

template <int DKA, int DVP, int BKV, int ST, int SB, int PT>
static int attn_set_attr() {
  SDW_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel<DKA, DVP, BKV, ST, SB, PT>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, AttnCfg<DKA, DVP, BKV, ST, SB, PT>::SMEM));
  return 0;
}
template <int DVP, int TRACE>
static cudaError_t pp_launch_one(const AttnKParams& p, dim3 grid, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_pp_kernel<DVP, TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         PPCfg<DVP>::SMEM);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  attn_pp_kernel<DVP, TRACE><<<grid, PPCfg<DVP>::THREADS, PPCfg<DVP>::SMEM, stream>>>(p);
  return cudaGetLastError();
}

static bool g_attn_init = false;
static int attn_init() {
  if (g_attn_init) return 0;
  if (int e = attn_set_attr<1, 16, 128, 2, 1, 1>()) return e;
  if (int e = attn_set_attr<1, 32, 128, 2, 1, 1>()) return e;
  if (int e = attn_set_attr<1, 48, 128, 2, 1, 1>()) return e;
  if (int e = attn_set_attr<1, 64, 128, 2, 1, 1>()) return e;
  if (int e = attn_set_attr<2, 80, 64, 2, 1, 1>()) return e;
  if (int e = attn_set_attr<3, 160, 64, 3, 2, 0>()) return e;
  g_attn_init = true;
  return 0;
}

bool attn_supported(int d) { return d % 8 == 0 && d >= 8 && d <= 160; }

static long long* g_attn_dbg = nullptr;
void attention_set_trace(long long* buf) { g_attn_dbg = buf; }

static int variant_for(int d, int Nk, int Nq) {
  const int cls = d <= 16 ? 0 : (d <= 32 ? 1 : (d <= 48 ? 2 : 3));
  // single-KV-tile (cross) attention with >= 2 query tiles goes through the two-tile kernel as well: 64x64, 77 keys,
  // batch 60: 155.6 us against 193.1 us for the query-tile loop of attn_fwd_kernel (same box)
  if (d <= 64) return (Nk > 128 || Nq >= 256) ? 8 + cls : cls;
  return d <= 80 ? 4 : 5;
}

int plan_attention(const AttnDesc& a, AttnLaunch* L) {
  SDW_REQUIRE(attn_supported(a.d), "flash attention supports head dims 8..160 (multiples of 8)");
  SDW_REQUIRE(a.q && a.k && a.vt && a.out, "null operand");
  SDW_REQUIRE(a.Nq > 0 && a.Nk > 0 && a.heads > 0 && a.B > 0, "empty attention");
  static_assert(sizeof(AttnLaunchImpl) <= sizeof(AttnLaunch::storage), "AttnLaunch storage too small");
  AttnLaunchImpl* I = reinterpret_cast<AttnLaunchImpl*>(L->storage);
  std::memset(I, 0, sizeof(*I));
  I->variant = variant_for(a.d, a.Nk, a.Nq);
  const bool pp = I->variant >= 8;
  const int bkv = (I->variant == 4 || I->variant == 5) ? 64 : 128;
  const int dvp_tab[12] = {16, 32, 48, 64, 80, 160, 0, 0, 16, 32, 48, 64};
  const int dvp = dvp_tab[I->variant];
  AttnKParams& p = I->p;
  p.Nq = a.Nq; p.Nk = a.Nk; p.d = a.d; p.heads = a.heads;
  p.dk_steps = (a.d + 15) / 16;
  p.scale_log2e = (1.f / std::sqrt(static_cast<float>(a.d))) * 1.4426950408889634f;
  p.out = a.out; p.out_ld = a.out_ld;
  p.dbg = nullptr;
  const int qtiles = (a.Nq + ATT_BQ - 1) / ATT_BQ;
  if (pp) {
    p.qt_per_cta = 2;
    p.qpairs = (qtiles + 1) / 2;
    const int64_t total = static_cast<int64_t>(a.B) * a.heads * p.qpairs;
    SDW_REQUIRE(total < (int64_t(1) << 31), "attention too large");
    p.total_work = static_cast<int>(total);
    I->grid = dim3(static_cast<unsigned>(std::min<int64_t>(total, 148)), 1, 1);
  } else {
    // cross attention (all keys in one KV tile): several query tiles per CTA, as long as >= ~3 waves of CTAs remain
    int qt = 1;
    if (a.Nk <= bkv) {
      qt = 8;  // cross attention 64x64, d = 40: 153 -> 119 us (profiles/r01_attn_bench_qtile_loop.txt)
      while (qt > 1 && static_cast<int64_t>((qtiles + qt - 1) / qt) * a.heads * a.B < 148 * 2 * 3) qt >>= 1;
      qt = std::max(1, std::min(qt, qtiles));
    }
    p.qt_per_cta = qt;
    I->grid = dim3((qtiles + qt - 1) / qt, a.heads, a.B);
  }
  {
    uint64_t dims[4] = {static_cast<uint64_t>(a.d), static_cast<uint64_t>(a.Nq), static_cast<uint64_t>(a.heads),
                        static_cast<uint64_t>(a.B)};
    uint64_t str[4] = {1, static_cast<uint64_t>(a.q_ld), static_cast<uint64_t>(a.d),
                       static_cast<uint64_t>(a.Nq) * a.q_ld};
    uint32_t box[4] = {64, ATT_BQ, 1, 1};
    if (int e = encode_map(&p.mapQ, a.q, 4, dims, str, box)) return e;
  }
  {
    uint64_t dims[4] = {static_cast<uint64_t>(a.d), static_cast<uint64_t>(a.Nk), static_cast<uint64_t>(a.heads),
                        static_cast<uint64_t>(a.B)};
    uint64_t str[4] = {1, static_cast<uint64_t>(a.k_ld), static_cast<uint64_t>(a.d),
                       static_cast<uint64_t>(a.Nk) * a.k_ld};
    uint32_t box[4] = {64, static_cast<uint32_t>(bkv), 1, 1};
    if (int e = encode_map(&p.mapK, a.k, 4, dims, str, box)) return e;
  }
  {
    uint64_t dims[4] = {static_cast<uint64_t>(a.Nk), static_cast<uint64_t>(a.d), static_cast<uint64_t>(a.heads),
                        static_cast<uint64_t>(a.B)};
    uint64_t str[4] = {1, static_cast<uint64_t>(a.vt_ld), static_cast<uint64_t>(a.d) * a.vt_ld,
                       static_cast<uint64_t>(a.heads) * a.d * a.vt_ld};
    uint32_t box[4] = {64, static_cast<uint32_t>(dvp), 1, 1};
    if (int e = encode_map(&p.mapV, a.vt, 4, dims, str, box)) return e;
  }
  return 0;
}

// planner introspection (host only): {variant, query tiles per CTA, grid.x, grid.y, grid.z}
void attention_plan_info(const AttnLaunch& L, int out[5]) {
  const AttnLaunchImpl* I = reinterpret_cast<const AttnLaunchImpl*>(L.storage);
  out[0] = I->variant;
  out[1] = I->p.qt_per_cta;
  out[2] = static_cast<int>(I->grid.x);
  out[3] = static_cast<int>(I->grid.y);
  out[4] = static_cast<int>(I->grid.z);
}

template <int DKA, int DVP, int BKV, int ST, int SB, int PT>
static cudaError_t launch_fwd(const AttnLaunchImpl* I, cudaStream_t stream) {
  attn_fwd_kernel<DKA, DVP, BKV, ST, SB, PT><<<I->grid, ATT_THREADS, AttnCfg<DKA, DVP, BKV, ST, SB, PT>::SMEM, stream>>>(I->p);
  return cudaGetLastError();
}
template <int DVP>
static cudaError_t launch_pp(const AttnLaunchImpl* I, cudaStream_t stream) {
  AttnKParams p = I->p;
  p.dbg = g_attn_dbg;
  if (p.dbg) return pp_launch_one<DVP, 1>(p, I->grid, stream);
  return pp_launch_one<DVP, 0>(p, I->grid, stream);
}

int launch_attention(const AttnLaunch& L, cudaStream_t stream) {
  if (int e = attn_init()) return e;
  const AttnLaunchImpl* I = reinterpret_cast<const AttnLaunchImpl*>(L.storage);
  switch (I->variant) {
    case 0: SDW_CUDA_OK((launch_fwd<1, 16, 128, 2, 1, 1>(I, stream))); break;
    case 1: SDW_CUDA_OK((launch_fwd<1, 32, 128, 2, 1, 1>(I, stream))); break;
    case 2: SDW_CUDA_OK((launch_fwd<1, 48, 128, 2, 1, 1>(I, stream))); break;
    case 3: SDW_CUDA_OK((launch_fwd<1, 64, 128, 2, 1, 1>(I, stream))); break;
    case 4: SDW_CUDA_OK((launch_fwd<2, 80, 64, 2, 1, 1>(I, stream))); break;
    case 5: SDW_CUDA_OK((launch_fwd<3, 160, 64, 3, 2, 0>(I, stream))); break;
    case 8: SDW_CUDA_OK(launch_pp<16>(I, stream)); break;
    case 9: SDW_CUDA_OK(launch_pp<32>(I, stream)); break;
    case 10: SDW_CUDA_OK(launch_pp<48>(I, stream)); break;
    case 11: SDW_CUDA_OK(launch_pp<64>(I, stream)); break;
    default: set_error("bad attention variant"); return 1;
  }
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace sdw
