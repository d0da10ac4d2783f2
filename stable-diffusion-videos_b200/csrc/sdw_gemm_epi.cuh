// sdw_gemm_epi.cuh — the fused epilogue shared by the 1-CTA and 2-CTA tcgen05 implicit-GEMM kernels:
// TMEM accumulator (thread = output row) -> alpha / bias / time-embedding row / SiLU or LeakyReLU / residual /
// scaled second residual / GEGLU / per-head V^T scatter -> fp16 global stores.
#pragma once
#include "sdw_internal.h"
#include "sdw_ptx.cuh"

namespace sdw {

__device__ __forceinline__ void store8(__half* dst, const float* v, bool vec_ok, int nvalid) {
  if (vec_ok && nvalid >= 8) {
    uint4 u;
    u.x = pack_h2(v[0], v[1]);
    u.y = pack_h2(v[2], v[3]);
    u.z = pack_h2(v[4], v[5]);
    u.w = pack_h2(v[6], v[7]);
    *reinterpret_cast<uint4*>(dst) = u;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < nvalid) dst[j] = __float2half_rn(v[j]);
  }
}
__device__ __forceinline__ void load8(const __half* src, float* v, bool vec_ok, int nvalid) {
  if (vec_ok && nvalid >= 8) {
    uint4 u = *reinterpret_cast<const uint4*>(src);
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 f = __half22float2(h[j]);
      v[2 * j] = f.x;
      v[2 * j + 1] = f.y;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (j < nvalid) ? __half2float(src[j]) : 0.f;
  }
}


// ---------------------------------------------------------------------------------------------
// fast paths: everything column-uniform is hoisted, 16-byte vector I/O only (the first version of this
// epilogue spent ~750 SASS instructions per 32-column chunk on generic address / predicate math and was
// the bottleneck of every short-K GEMM — see profiles/r01_ncu_gemm_linear_v1.txt).
// FLAGS: 1 bias, 2 per-sample row vector (time embedding), 4 residual, 8 SiLU, 16 alpha != 1, 32 LeakyReLU(0.2)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float leaky02(float x) { return x > 0.f ? x : 0.2f * x; }

__device__ __forceinline__ void add8(float* o, const float* __restrict__ src) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(src));
  const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 1);
  o[0] += a.x; o[1] += a.y; o[2] += a.z; o[3] += a.w;
  o[4] += b.x; o[5] += b.y; o[6] += b.z; o[7] += b.w;
}

// V^T scatter of one 32-column chunk (columns >= vt_col0): out element (b, head, dd, tok)
__device__ __forceinline__ void epi_vt_chunk(const GemmKParams& p, const uint32_t (&v)[32], int n, int64_t pix_in) {
  const int64_t bq = pix_in / p.vt_ntok;
  const int tok = static_cast<int>(pix_in - bq * p.vt_ntok);
  int cc = n - p.vt_col0;
  int head = cc / p.vt_d;
  int dd = cc - head * p.vt_d;
  __half* base = p.vt + (bq * p.vt_heads) * p.vt_d * p.vt_ld + tok;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    if (n + j < p.N) {
      float a = __uint_as_float(v[j]) * p.alpha;
      if (p.bias) a += __ldg(&p.bias[n + j]);
      base[(static_cast<int64_t>(head) * p.vt_d + dd) * p.vt_ld] = __float2half_rn(a);
    }
    if (++dd == p.vt_d) {
      dd = 0;
      ++head;
    }
  }
}

// Coalescing stage: the row-owner layout (thread = output row) would move 16 B per lane to / from 32 different cache
// lines per instruction.  Instead each warp bounces a 32-row x 64-byte chunk through 2 KB of shared memory
// (XOR-swizzled, conflict-free both ways) and talks to global memory with 4 lanes per row: 8 full 64-byte row
// segments per instruction.  "Coalesced layout": lane l, slot it <-> (row = it*8 + l/4, 16-byte piece = l%4).
struct EpiRows {
  int32_t out[4];  // element offsets of rows it*8 + lane/4 in the output (or -1); the planner guarantees < 2^31
  int32_t res[4];  // ... in the residual (or -1)
};
__device__ __forceinline__ void epi_rows_init(EpiRows& R, int lane, int64_t out_off, int64_t res_off) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int row = it * 8 + (lane >> 2);
    R.out[it] = __shfl_sync(0xffffffffu, static_cast<int32_t>(out_off), row);
    R.res[it] = __shfl_sync(0xffffffffu, static_cast<int32_t>(res_off), row);
  }
}
// w[j8]: this lane's row, 8 fp16 columns each (j8 < npieces valid) -> coalesced global stores
__device__ __forceinline__ void staged_store32(uint8_t* stage, int lane, const uint4 (&w)[4], int npieces,
                                               bool row_ok, const EpiRows& R, __half* out, int col) {
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int j8 = 0; j8 < 4; ++j8)
    if (j8 < npieces && row_ok) *reinterpret_cast<uint4*>(stage + lane * 64 + ((j8 ^ sw) << 4)) = w[j8];
  __syncwarp();
  const int piece = lane & 3;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int row = it * 8 + (lane >> 2);
    if (R.out[it] >= 0 && piece < npieces) {
      const uint4 u = *reinterpret_cast<const uint4*>(stage + row * 64 + ((piece ^ ((row >> 1) & 3)) << 4));
      *reinterpret_cast<uint4*>(out + R.out[it] + col + piece * 8) = u;
    }
  }
  __syncwarp();
}
// direct (row-owner) residual load, used when no stage buffer exists (1-CTA kernel)
template <int FLAGS>
__device__ __forceinline__ void epi_res_load(uint4 (&rs)[4], int n, int nvalid, bool row_ok, const __half* res_row) {
  if (FLAGS & 4) {
#pragma unroll
    for (int j8 = 0; j8 < 4; ++j8)
      if (j8 * 8 < nvalid && row_ok) rs[j8] = *reinterpret_cast<const uint4*>(res_row + n + j8 * 8);
  }
}

template <int BN, int FLAGS>
__device__ __forceinline__ void epi_fast(const GemmKParams& p, uint32_t taddr, int n0, bool row_ok, int64_t pix_in,
                                         __half* out_row, const __half* res_row, const float* rowvec, int chunk0,
                                         int chunk_step, uint8_t* stage, int lane, int64_t out_off, uint4 (&g)[4]) {
  const int nmax = min(BN, p.N - n0);  // valid columns of this tile (multiple of 8)
  const bool vt_mode = p.mode == GEMM_QKV_VT;
  EpiRows R;
  const bool stage_st = stage && p.stage_stores;
  if (stage_st) epi_rows_init(R, lane, row_ok ? out_off : -1, -1);
  // residual of the NEXT chunk in flight (row-owner layout; its first chunk was issued before the TMEM-full wait and
  // the whole row segment was prefetched into L2 — see gemm_epilogue)
  int c = chunk0;
#pragma unroll 1
  for (; c * 32 < nmax; c += chunk_step) {
    const int n = n0 + c * 32;
    const int npieces = min(4, (nmax - c * 32) >> 3);
    const bool vt_chunk = vt_mode && n >= p.vt_col0;
    uint4 rs[4];
    if ((FLAGS & 4) && !vt_chunk) {
#pragma unroll
      for (int j8 = 0; j8 < 4; ++j8) rs[j8] = g[j8];
    }
    if (vt_chunk) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      tmem_ld_wait();
      if (row_ok) epi_vt_chunk(p, v, n, pix_in);
    } else {
      uint4 w[4];
#pragma unroll
      for (int half = 0; half < 2; ++half) {  // 16 accumulator columns at a time: small live register set
        uint32_t v[16];
        tmem_ld_32x16(taddr + c * 32 + half * 16, v);
        if (half == 0) {
          // the next chunk's residual does not depend on the accumulator: issue it before the TMEM wait
          const int cn = c + chunk_step;
          if ((FLAGS & 4) && cn * 32 < nmax) {
            epi_res_load<FLAGS>(g, n0 + cn * 32, nmax - cn * 32, row_ok, res_row);
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int j8 = half * 2 + q;
          if (j8 < npieces) {
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              o[j] = __uint_as_float(v[q * 8 + j]);
              if (FLAGS & 16) o[j] *= p.alpha;
            }
            if (FLAGS & 1) add8(o, p.bias + n + j8 * 8);
            if (FLAGS & 2) add8(o, rowvec + n + j8 * 8);
            if (FLAGS & 8) {
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = silu_f(o[j]);
            }
            if (FLAGS & 32) {
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = leaky02(o[j]);
            }
            if (FLAGS & 4) {
              const __half2* h = reinterpret_cast<const __half2*>(&rs[j8]);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 f = __half22float2(h[j]);
                o[2 * j] += f.x;
                o[2 * j + 1] += f.y;
              }
            }
            w[j8].x = pack_h2(o[0], o[1]);
            w[j8].y = pack_h2(o[2], o[3]);
            w[j8].z = pack_h2(o[4], o[5]);
            w[j8].w = pack_h2(o[6], o[7]);
          }
        }
      }
      if (stage_st) {
        staged_store32(stage, lane, w, npieces, row_ok, R, p.out, n);
      } else if (row_ok) {
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8)
          if (j8 < npieces) *reinterpret_cast<uint4*>(out_row + n + j8 * 8) = w[j8];
      }
    }
  }
}

// GEGLU: packed columns [32 value | 32 gate] pairs -> 32 outputs a * gelu(g)
template <int BN>
__device__ __forceinline__ void epi_geglu(const GemmKParams& p, uint32_t taddr, int n0, bool row_ok, __half* out_row,
                                          bool vec_out, int chunk0, int chunk_step, uint8_t* stage, int lane,
                                          int64_t out_off) {
  EpiRows R;
  const bool stage_st = stage && p.stage_stores && vec_out;
  if (stage_st) epi_rows_init(R, lane, row_ok ? out_off : -1, -1);
#pragma unroll 1
  for (int c = chunk0; c < BN / 64; c += chunk_step) {
    const int n = n0 + c * 64;
    if (n >= p.N) break;
    uint4 w[4];
#pragma unroll
    for (int half = 0; half < 2; ++half) {  // 16 + 16 columns at a time keeps the live register set small
      uint32_t va[16], vg[16];
      tmem_ld_32x16(taddr + c * 64 + half * 16, va);
      tmem_ld_32x16(taddr + c * 64 + 32 + half * 16, vg);
      tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int j8 = half * 2 + q;
        float a[8], g[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          a[j] = __uint_as_float(va[q * 8 + j]) * p.alpha;
          g[j] = __uint_as_float(vg[q * 8 + j]) * p.alpha;
        }
        if (p.bias) {
          add8(a, p.bias + n + j8 * 8);
          add8(g, p.bias + n + 32 + j8 * 8);
        }
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          upk2(geglu2(pk2(0.5f * a[2 * j], 0.5f * a[2 * j + 1]), g[2 * j], g[2 * j + 1]), o[2 * j], o[2 * j + 1]);
        w[j8].x = pack_h2(o[0], o[1]);
        w[j8].y = pack_h2(o[2], o[3]);
        w[j8].z = pack_h2(o[4], o[5]);
        w[j8].w = pack_h2(o[6], o[7]);
      }
    }
    if (stage_st) {
      staged_store32(stage, lane, w, 4, row_ok, R, p.out, n / 2);
    } else if (row_ok) {
#pragma unroll
      for (int j8 = 0; j8 < 4; ++j8) {
        if (vec_out) {
          *reinterpret_cast<uint4*>(out_row + n / 2 + j8 * 8) = w[j8];
        } else {
          const __half* h = reinterpret_cast<const __half*>(&w[j8]);
#pragma unroll
          for (int j = 0; j < 8; ++j) out_row[n / 2 + j8 * 8 + j] = h[j];
        }
      }
    }
  }
}

// warp = absolute warp index of an epilogue warp (its TMEM lane quarter is warp & 3); tmem_acc = accumulator base.
template <int BN>
__device__ __forceinline__ void gemm_epilogue(const GemmKParams& p, uint32_t tmem_acc, int warp, int lane, int x0,
                                              int y0, int b0, int n0, uint64_t* tmem_full_bar, uint32_t full_parity = 0,
                                              int chunk0 = 0, int chunk_step = 1, uint8_t* stage = nullptr) {
  const int quarter = warp & 3;  // TMEM lane quarter this warp may read
  const int r = quarter * 32 + lane;
  const int lx = r & (p.bw - 1);  // bw, bh, bb are powers of two
  const int ly = (r >> p.lg_bw) & (p.bh - 1);
  const int lb = r >> (p.lg_bw + p.lg_bh);
  const int x = x0 + lx, y = y0 + ly, b = b0 + lb;
  const bool row_ok = (x < p.W) && (y < p.H) && (b < p.B);
  const int64_t pix_in = (static_cast<int64_t>(b) * p.H + y) * p.W + x;  // lattice-linear index
  const int oyy = y * p.os + p.oy, oxx = x * p.os + p.ox;
  const int64_t out_off = static_cast<int64_t>(b) * p.o_sB + oyy * p.o_sH + oxx * p.o_sW;
  const int64_t res_off = static_cast<int64_t>(b) * p.r_sB + oyy * p.r_sH + oxx * p.r_sW;
  const bool vec_out = (((p.o_sW | p.o_sH | p.o_sB) & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
  const bool vec_res = p.resid && (((p.r_sW | p.r_sH | p.r_sB) & 7) == 0) &&
                       ((reinterpret_cast<uintptr_t>(p.resid) & 15) == 0);
  const float* rowvec = p.rowvec ? p.rowvec + static_cast<int64_t>(b) * p.rowvec_ld : nullptr;
  __half* out_row = p.out + out_off;
  const __half* res_row = p.resid ? p.resid + res_off : nullptr;
  const __half* res2_row = p.resid2 ? p.resid2 + res_off : nullptr;
  const bool vec_res2 = p.resid2 && (((p.r_sW | p.r_sH | p.r_sB) & 7) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.resid2) & 15) == 0);

  const bool fast = vec_out && (!p.resid || vec_res) && !p.resid2 && ((p.N & 7) == 0) &&
                    (!p.bias || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0) &&
                    (!p.rowvec || ((reinterpret_cast<uintptr_t>(p.rowvec) & 15) == 0 && (p.rowvec_ld & 3) == 0));
  // the residual does not depend on the accumulator: while the mainloop of this tile is still running, pull this
  // row's residual segment into L2 and issue the first chunk's loads (their latency hides behind the TMEM-full wait)
  uint4 g[4];
  if (fast && p.resid && p.mode != GEMM_GEGLU && row_ok) {
    const int nmax = min(BN, p.N - n0);
    for (int cb = 0; cb < nmax * 2; cb += 128)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const uint8_t*>(res_row + n0) + cb));
    if (chunk0 * 32 < nmax) epi_res_load<4>(g, n0 + chunk0 * 32, nmax - chunk0 * 32, true, res_row);
  }

  mbar_wait(tmem_full_bar, full_parity);
  tc_fence_after();
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(quarter * 32) << 16);

  if (p.mode == GEMM_GEGLU) {
    epi_geglu<BN>(p, taddr, n0, row_ok, out_row, vec_out, chunk0, chunk_step, stage, lane, out_off);
    return;
  }
  if (fast) {
    const int flags = (p.bias ? 1 : 0) | (p.rowvec ? 2 : 0) | (p.resid ? 4 : 0) | (p.act == 1 ? 8 : 0) |
                      (p.alpha != 1.f ? 16 : 0) | (p.act == 2 ? 32 : 0);
    switch (flags) {
      case 0: epi_fast<BN, 0>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      case 1: epi_fast<BN, 1>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      case 3: epi_fast<BN, 3>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      case 5: epi_fast<BN, 5>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      case 16: epi_fast<BN, 16>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      // Real-ESRGAN: conv + LeakyReLU, and the dense-block exit 0.2 * (acc + b) + x (bias pre-scaled)
      case 33: epi_fast<BN, 33>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      case 21: epi_fast<BN, 21>(p, taddr, n0, row_ok, pix_in, out_row, res_row, rowvec, chunk0, chunk_step, stage, lane, out_off, g); return;
      default: break;
    }
  }
  // ---- generic path (unaligned views, odd N, rarely used flag combinations) --------------------
#pragma unroll 1
  for (int c = chunk0; c < BN / 32; c += chunk_step) {
    const int n = n0 + c * 32;
    if (n >= p.N) break;
    uint32_t v[32];
    tmem_ld_32x32(taddr + c * 32, v);
    tmem_ld_wait();
    if (!row_ok) continue;
    if (p.mode == GEMM_QKV_VT && n >= p.vt_col0) {
      epi_vt_chunk(p, v, n, pix_in);
      continue;
    }
#pragma unroll
    for (int j8 = 0; j8 < 4; ++j8) {
      const int nn = n + j8 * 8;
      const int nvalid = min(8, p.N - nn);
      if (nvalid <= 0) continue;
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float a = __uint_as_float(v[j8 * 8 + j]) * p.alpha;
        if (j < nvalid) {
          if (p.bias) a += __ldg(&p.bias[nn + j]);
          if (rowvec) a += __ldg(&rowvec[nn + j]);
        }
        if (p.act == 1) a = silu_f(a);
        else if (p.act == 2) a = leaky02(a);
        o[j] = a;
      }
      if (p.resid) {
        float rr[8];
        load8(res_row + nn, rr, vec_res, nvalid);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] += rr[j];
      }
      if (res2_row) {
        float rr[8];
        load8(res2_row + nn, rr, vec_res2, nvalid);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(o[j], p.res2_scale, rr[j]);
      }
      store8(out_row + nn, o, vec_out, nvalid);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA epilogue (2-CTA kernel, short-K GEMMs).  The classic epilogue above keeps every global access on the warp's
// critical path: bias and residual loads behind each TMEM wait, 16-byte row-owner stores to 32 cache lines per
// instruction.  With five K blocks per tile that chain, not the MMA, set the tile time (profiles/r01_ncu_epilogue_shortk.md:
// 8.6 us per 256 x 160 tile against a 1.7 us operand-ingest floor).  Here
//   * the bias slice of the tile is copied to shared memory once per tile (before the accumulator is awaited),
//   * the residual tile arrives in [128 rows x 32 columns] chunks filled by TMA from a producer thread that runs ahead
//     across tiles: two ring slots per chunk group c % EW (consumers: the 4 warps — one per lane quarter — of the group),
//   * each warp writes its 32-row x 32-column output slab to shared memory (64B-swizzled, conflict-free) and one lane
//     hands it to a TMA store; rows / columns outside the tensor are clipped by the tensor map.
// State carried across tiles: `res_k` (residual chunks consumed = ring position of the warp's group) and `nstore` (output slab).
// ---------------------------------------------------------------------------------------------
struct EpiTmaState {
  uint32_t res_k = 0;   // residual chunks this warp has consumed (its group's ring position)
  uint32_t nstore = 0;
};

// EW = warps per TMEM lane quarter (2 or 4); warp `cpar` of a quarter takes the 32-column chunks c = cpar, cpar + EW, ...
// EW = 2: two output slabs per warp (the store of chunk i overlaps the math of chunk i + 1); EW = 4: one slab per warp
// (a warp has one or two chunks per tile; the overlap comes from the other three warps of its quarter).
template <int BN, int EW>
__device__ __forceinline__ void gemm_epilogue_tma(const GemmKParams& p, uint32_t tmem_acc, int warp, int lane, int x0,
                                                  int y0, int b0, int n0, uint64_t* tmem_full_bar, uint32_t full_parity,
                                                  int cpar, uint8_t* out_stage, float* bias_s, const uint8_t* res_ring,
                                                  uint64_t* res_full, uint64_t* res_empty, EpiTmaState& st) {
  const int quarter = warp & 3;
  const int nmax = max(0, min(BN, p.N - n0));  // valid accumulator columns (multiple of 8)
  const bool geglu = p.mode == GEMM_GEGLU;
  // ---- bias slice -> shared memory (GEGLU: value columns carry the 0.5 of GELU) ----
  __syncwarp();
#pragma unroll
  for (int i = lane * 4; i < BN; i += 128) {
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias && i < nmax) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + i));
    if (p.rowvec && i < nmax) {  // time-embedding row, the same for every sample (rowvec_ld == 0: planner-checked)
      const float4 r4 = __ldg(reinterpret_cast<const float4*>(p.rowvec + n0 + i));
      b4.x += r4.x; b4.y += r4.y; b4.z += r4.z; b4.w += r4.w;
    }
    if (geglu && (i & 32) == 0) {
      b4.x *= 0.5f; b4.y *= 0.5f; b4.z *= 0.5f; b4.w *= 0.5f;
    }
    *reinterpret_cast<float4*>(bias_s + i) = b4;
  }
  __syncwarp();
  // this warp's 32-row slab of the tile in lattice coordinates
  const int row0 = quarter * 32;
  const int sx = x0 + (row0 & (p.bw - 1)), sy = y0 + ((row0 >> p.lg_bw) & (p.bh - 1)), sb = b0 + (row0 >> (p.lg_bw + p.lg_bh));
  const int sw = (lane >> 1) & 3;  // 64B-swizzle phase of this thread's row (slab and ring bases are 512B aligned)

  mbar_wait(tmem_full_bar, full_parity);
  tc_fence_after();
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(quarter * 32) << 16);
  const uint64_t alpha2 = pk2(p.alpha, p.alpha);

  if (geglu) {
    const uint64_t alpha_h = pk2(0.5f * p.alpha, 0.5f * p.alpha);
#pragma unroll 1
    for (int c = cpar; c * 64 < nmax; c += EW) {
      uint8_t* ob = out_stage + (EW == 2 ? (st.nstore & 1) * 2048 : 0);
      if (lane == 0) bulk_wait_group_read<EW == 2 ? 1 : 0>();  // the slab about to be overwritten has left shared memory
      __syncwarp();
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t va[16], vg[16];
        tmem_ld_32x16(taddr + c * 64 + half * 16, va);
        tmem_ld_32x16(taddr + c * 64 + 32 + half * 16, vg);
        tmem_ld_wait();
        const float* ba = bias_s + c * 64 + half * 16;
        const float* bg = ba + 32;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint32_t w[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int e = q * 8 + 2 * j;
            const float2 bav = *reinterpret_cast<const float2*>(ba + e);
            const float2 bgv = *reinterpret_cast<const float2*>(bg + e);
            const uint64_t ah = fma2(pk2(__uint_as_float(va[e]), __uint_as_float(va[e + 1])), alpha_h, pk2(bav.x, bav.y));
            float g0, g1;
            upk2(fma2(pk2(__uint_as_float(vg[e]), __uint_as_float(vg[e + 1])), alpha2, pk2(bgv.x, bgv.y)), g0, g1);
            float o0, o1;
            upk2(geglu2(ah, g0, g1), o0, o1);
            w[j] = pack_h2(o0, o1);
          }
          *reinterpret_cast<uint4*>(ob + lane * 64 + (((half * 2 + q) ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(&p.mapOut, ob, (n0 >> 1) + c * 32, sx, sy, sb);
        bulk_commit_group();
      }
      ++st.nstore;
    }
    return;
  }

  const int nch = (nmax + 31) >> 5;
  const int act = p.act;
  const bool vt_mode = p.mode == GEMM_QKV_VT;
#pragma unroll 1
  for (int c = cpar; c < nch; c += EW) {
    uint8_t* ob = out_stage + (EW == 2 ? (st.nstore & 1) * 2048 : 0);
    if (lane == 0) bulk_wait_group_read<EW == 2 ? 1 : 0>();
    __syncwarp();
    if (vt_mode && n0 + c * 32 >= p.vt_col0) {
      // V columns leave transposed: slab[row = column of this chunk][token = lane] (32 x 64 B, unswizzled), one TMA
      // store into V^T (token contiguous).  A warp-wide 2-byte store row is 64 contiguous bytes: conflict-free.
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t v[16];
        tmem_ld_32x16(taddr + c * 32 + half * 16, v);
        tmem_ld_wait();
        const float* bs = bias_s + c * 32 + half * 16;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float o = fmaf(__uint_as_float(v[j]), p.alpha, bs[j]);
          *reinterpret_cast<__half*>(ob + (half * 16 + j) * 64 + lane * 2) = __float2half_rn(o);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_3d(&p.mapVt, ob, sx, n0 + c * 32 - p.vt_col0, sb);
        bulk_commit_group();
      }
      ++st.nstore;
      continue;
    }
    const uint8_t* rs = nullptr;
    uint32_t slot = 0;
    if (p.resid) {
      // the chunk group c % EW (= cpar) owns ring slots {cpar, cpar + EW}, filled alternately: every fill of a slot is
      // consumed by the same four warps in order, so the one-bit phase parity cannot alias.  (A ring indexed by the
      // global chunk count lets a group that skips revolutions mistake fill f - 2 of a slot for fill f: it hung the
      // 16-warp epilogue with five chunks per tile.)
      slot = cpar + EW * (st.res_k & 1);
      mbar_wait(&res_full[slot], (st.res_k >> 1) & 1);
      ++st.res_k;
      rs = res_ring + slot * G2_RES_STAGE + (row0 + lane) * 64;
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      uint32_t v[16];
      tmem_ld_32x16(taddr + c * 32 + half * 16, v);
      tmem_ld_wait();
      const float* bs = bias_s + c * 32 + half * 16;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int j8 = half * 2 + q;
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 bv = *reinterpret_cast<const float2*>(bs + q * 8 + 2 * j);
          upk2(fma2(pk2(__uint_as_float(v[q * 8 + 2 * j]), __uint_as_float(v[q * 8 + 2 * j + 1])), alpha2, pk2(bv.x, bv.y)),
               o[2 * j], o[2 * j + 1]);
        }
        if (act) {  // one branch on the common act = 0 path
          if (act == 1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = silu_f(o[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = leaky02(o[j]);
          }
        }
        if (rs) {
          const uint4 r4 = *reinterpret_cast<const uint4*>(rs + ((j8 ^ sw) << 4));
          const __half2* h = reinterpret_cast<const __half2*>(&r4);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            o[2 * j] += f.x;
            o[2 * j + 1] += f.y;
          }
        }
        *reinterpret_cast<uint4*>(ob + lane * 64 + ((j8 ^ sw) << 4)) =
            make_uint4(pack_h2(o[0], o[1]), pack_h2(o[2], o[3]), pack_h2(o[4], o[5]), pack_h2(o[6], o[7]));
      }
    }
    fence_proxy_async_smem();
    __syncwarp();  // also orders every lane's ring reads before the release below
    if (lane == 0) {
      if (p.resid) mbar_arrive(&res_empty[slot]);
      tma_store_4d(&p.mapOut, ob, n0 + c * 32, sx, sy, sb);
      bulk_commit_group();
    }
    ++st.nstore;
  }
}

}  // namespace sdw
