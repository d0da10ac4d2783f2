// sdw_norm.cu — the HBM-bound layers between the tensor-core kernels (all fp32 math, fp16 NHWC I/O):
//   GroupNorm(+SiLU), LayerNorm, row softmax, the tiny-channel direct convolutions (conv_in: 4 -> C,
//   conv_out: C -> 4 / 3 with the VAE post-process fused), post_quant_conv, fp32 small linear layers
//   (time-embedding MLP and the per-ResBlock time projections) and the sinusoidal timestep embedding.
// Reference call sites: the layers inside `self.unet(...)` (stable_diffusion_pipeline.py:418) and
// `self.vae.decode(...)` (:433); post-process = :435-438 + numpy_to_pil (:450).
#include "sdw_internal.h"
#include "sdw_ptx.cuh"

namespace sdw {

// =============================================================================================
// GroupNorm: three small deterministic kernels.
//   gn_partial : grid (nchunks, B). Each block sums x and x^2 per group over its pixel chunk (all channels,
//                coalesced 16-byte loads, fixed reduction order) -> partial[b][chunk][g] = (sum, sumsq).
//   gn_finalize: one warp per (b, g) reduces the chunk partials in a fixed order -> (mean, rstd).
//   gn_apply   : grid (pixel tiles, B): y = (x - mean) * rstd * gamma + beta (optionally SiLU), fp16 out.
// =============================================================================================
static constexpr int GN_MAX_CHUNKS = 1024;
static constexpr int GN_MAX_GROUPS = 64;

// per-thread partials go to shared memory and are reduced in index order (bit-reproducible).
__global__ void __launch_bounds__(256) gn_partial_det_kernel(const __half* __restrict__ x, int64_t ld, int C, int G,
                                                             int64_t P, int pix_per_chunk,
                                                             float2* __restrict__ part) {
  extern __shared__ float sm[];  // [rows][C] sums then [rows][C] squares
  // blocks walk the tensor from its END: the producing GEMM wrote it front to back, so the tail is what the 126 MB L2
  // still holds (a front-to-back read of a 157 MB tensor evicts every line just before it is needed); this pass then
  // ends at the front, which is where gn_apply starts (profiles/r02_norm_reverse_order_ab.txt)
  const int b = static_cast<int>(gridDim.y) - 1 - static_cast<int>(blockIdx.y);
  const int chunk = static_cast<int>(gridDim.x) - 1 - static_cast<int>(blockIdx.x);
  const int cg = C / G;
  const int vecs = C / 8;
  const int rows = max(1, min(min(static_cast<int>(blockDim.x) / vecs, 16), 6144 / C));
  const int64_t p0 = static_cast<int64_t>(chunk) * pix_per_chunk;
  const int64_t p1 = min(P, p0 + pix_per_chunk);
  const __half* xb = x + static_cast<int64_t>(b) * P * ld;
  float* ssum = sm;
  float* ssq = sm + rows * C;
  for (int item = threadIdx.x; item < rows * vecs; item += blockDim.x) {
    const int v = item % vecs, prow = item / vecs;
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
    int64_t p = p0 + prow;
    // 4 independent 16-byte loads in flight per thread
    for (; p + 3 * rows < p1; p += 4 * rows) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) u[k] = *reinterpret_cast<const uint4*>(xb + (p + k * rows) * ld + v * 8);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const __half2* h = reinterpret_cast<const __half2*>(&u[k]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(h[j]);
          s[2 * j] += f.x;
          q[2 * j] = fmaf(f.x, f.x, q[2 * j]);
          s[2 * j + 1] += f.y;
          q[2 * j + 1] = fmaf(f.y, f.y, q[2 * j + 1]);
        }
      }
    }
    for (; p < p1; p += rows) {
      const uint4 u = *reinterpret_cast<const uint4*>(xb + p * ld + v * 8);
      const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h[j]);
        s[2 * j] += f.x;
        q[2 * j] = fmaf(f.x, f.x, q[2 * j]);
        s[2 * j + 1] += f.y;
        q[2 * j + 1] = fmaf(f.y, f.y, q[2 * j + 1]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      ssum[prow * C + v * 8 + j] = s[j];
      ssq[prow * C + v * 8 + j] = q[j];
    }
  }
  __syncthreads();
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    float a = 0.f, c = 0.f;
    for (int r = 0; r < rows; ++r)
      for (int j = 0; j < cg; ++j) {
        a += ssum[r * C + g * cg + j];
        c += ssq[r * C + g * cg + j];
      }
    part[(static_cast<int64_t>(b) * gridDim.x + chunk) * G + g] = make_float2(a, c);
  }
}

// one warp per (b, g): fixed-order reduction of the chunk partials -> (mean, rstd)
__global__ void __launch_bounds__(256) gn_finalize_kernel(const float2* __restrict__ part, int nchunks, int G, int BG,
                                                          float count, float eps, float2* __restrict__ stats) {
  const int idx = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (idx >= BG) return;
  const int lane = threadIdx.x & 31;
  const int b = idx / G, g = idx % G;
  float a = 0.f, c = 0.f;
  for (int k = lane; k < nchunks; k += 32) {
    const float2 pr = part[(static_cast<int64_t>(b) * nchunks + k) * G + g];
    a += pr.x;
    c += pr.y;
  }
  a = warp_sum(a);
  c = warp_sum(c);
  if (lane == 0) {
    const float mean = a / count;
    const float var = fmaxf(c / count - mean * mean, 0.f);
    stats[idx] = make_float2(mean, rsqrtf(var + eps));
  }
}

__global__ void __launch_bounds__(256, 3) gn_apply_kernel(const __half* __restrict__ x, int64_t ldx, int C, int G,
                                                          int64_t P, const float2* __restrict__ stats,
                                                          const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, int silu,
                                                          __half* __restrict__ y, int64_t ldy, int pix_per_block) {
  // per-channel affine of this sample, folded once per block: y = x * sa[c] + sb[c],
  //   sa = rstd_g * gamma_c, sb = beta_c - mean_g * rstd_g * gamma_c   (no group bookkeeping in the streaming loop)
  extern __shared__ float gn_aff[];  // [C] sa, [C] sb
  float* sa = gn_aff;
  float* sb = gn_aff + C;
  const int b = blockIdx.y;
  const int cg = C / G;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float2 st = stats[b * G + c / cg];
    const float a = st.y * gamma[c];
    sa[c] = a;
    sb[c] = fmaf(-st.x, a, beta[c]);
  }
  __syncthreads();
  const int vecs = C / 8;
  const int64_t p0 = static_cast<int64_t>(blockIdx.x) * pix_per_block;
  const int64_t p1 = min(P, p0 + pix_per_block);
  const __half* xb = x + static_cast<int64_t>(b) * P * ldx;
  __half* yb = y + static_cast<int64_t>(b) * P * ldy;
  auto apply8 = [&](const uint4& u, int v, int64_t p) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
    const float4 a0 = *reinterpret_cast<const float4*>(sa + v * 8), a1 = *reinterpret_cast<const float4*>(sa + v * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(sb + v * 8), b1 = *reinterpret_cast<const float4*>(sb + v * 8 + 4);
    const float aa[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(h[j]);
      o[2 * j] = fmaf(f.x, aa[2 * j], bb[2 * j]);
      o[2 * j + 1] = fmaf(f.y, aa[2 * j + 1], bb[2 * j + 1]);
    }
    if (silu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __fdividef(o[j], 1.f + __expf(-o[j]));
    }
    *reinterpret_cast<uint4*>(yb + p * ldy + v * 8) =
        make_uint4(pack_h2(o[0], o[1]), pack_h2(o[2], o[3]), pack_h2(o[4], o[5]), pack_h2(o[6], o[7]));
  };
  // 4 independent 16-byte loads in flight per thread.  (pixel, vector) of item `it` advance incrementally: the 64-bit
  // div / mod per item this loop used to do cost more issue slots than the normalisation itself
  const int dv = static_cast<int>(blockDim.x) % vecs, dp = static_cast<int>(blockDim.x) / vecs;
  int v = static_cast<int>(threadIdx.x) % vecs;
  int pl = static_cast<int>(threadIdx.x) / vecs;  // pixel relative to p0
  const int npix = static_cast<int>(p1 - p0);
  auto advance = [&](int& vv, int& pp) {
    vv += dv;
    pp += dp;
    if (vv >= vecs) {
      vv -= vecs;
      ++pp;
    }
  };
  // software pipeline: batch k+1 (4 x 16 B per thread) is in flight while batch k is normalised — with a single batch
  // the ~64 KB an SM had in flight during the load phases only could not cover the HBM latency-bandwidth product
  struct Batch {
    uint4 u[4];
    int vv[4];
    int pp[4];
    int n;
  };
  Batch A, Bt;
  auto load_batch = [&](Batch& t) {
    t.n = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      t.vv[k] = v;
      t.pp[k] = pl;
      if (pl < npix) {
        t.u[k] = *reinterpret_cast<const uint4*>(xb + (p0 + pl) * ldx + v * 8);
        t.n = k + 1;
      }
      advance(v, pl);
    }
  };
  auto run_batch = [&](const Batch& t) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k < t.n) apply8(t.u[k], t.vv[k], p0 + t.pp[k]);
  };
  load_batch(A);
#pragma unroll 1
  while (true) {
    if (A.n == 4) load_batch(Bt);
    else Bt.n = 0;
    run_batch(A);
    if (Bt.n == 0) break;
    if (Bt.n == 4) load_batch(A);
    else A.n = 0;
    run_batch(Bt);
    if (A.n == 0) break;
  }
}

// (A single-launch variant — one thread-block cluster per sample, statistics exchanged through distributed shared memory,
//  the slice normalised while still in L2 — was built, measured slower (64x64x320, batch 32: 130 us vs 82 us; VAE
//  512x512x128: 2.1 ms vs 0.82 ms: 18 clusters of 8 CTAs keep too few loads in flight) and removed.)

// chunks per sample: enough blocks to fill the machine (B * nchunks >= ~4 waves) while keeping >= 16 pixels each
int gn_chunks(int64_t P, int B) {
  int64_t want = (148 * 7 + B - 1) / B;  // 7 blocks of the stats kernel fit an SM (30 KB of shared memory each)
  int64_t n = std::min<int64_t>(want, P / 16);
  if (n < 1) n = 1;
  if (n > GN_MAX_CHUNKS) n = GN_MAX_CHUNKS;
  return static_cast<int>(n);
}

// workspace: partials [B][nchunks][G] float2 followed by stats [B][G] float2
size_t gn_workspace_bytes(int B) { return (static_cast<size_t>(B) * GN_MAX_CHUNKS * GN_MAX_GROUPS + B * GN_MAX_GROUPS) * sizeof(float2); }

int groupnorm_launches() { return 3; }

int groupnorm(const __half* x, int64_t ldx, int B, int64_t P, int C, int G, const float* gamma, const float* beta,
              float eps, int silu, __half* y, int64_t ldy, float2* partial_ws, cudaStream_t stream) {
  SDW_REQUIRE(C % 8 == 0 && C % G == 0 && G <= GN_MAX_GROUPS, "GroupNorm: C % 8, C % G, G <= 64");
  SDW_REQUIRE(ldx % 8 == 0 && ldy % 8 == 0, "GroupNorm: row pitch must be a multiple of 8");
  const int nchunks = gn_chunks(P, B);
  const int ppc = static_cast<int>((P + nchunks - 1) / nchunks);
  const int vecs = C / 8;
  const int rows = std::max(1, std::min(std::min(256 / vecs, 16), 6144 / C));
  const size_t smem = static_cast<size_t>(2) * rows * C * sizeof(float);
  SDW_REQUIRE(smem <= 48 * 1024, "GroupNorm: channel count too large for the stats kernel");
  float2* stats = partial_ws + static_cast<size_t>(B) * nchunks * G;
  gn_partial_det_kernel<<<dim3(nchunks, B), 256, smem, stream>>>(x, ldx, C, G, P, ppc, partial_ws);
  const int BG = B * G;
  gn_finalize_kernel<<<(BG + 7) / 8, 256, 0, stream>>>(partial_ws, nchunks, G, BG, static_cast<float>(P) * (C / G), eps,
                                                       stats);
  // one full wave: 148 SMs x 8 resident 256-thread blocks, split evenly over the samples (the former fixed ~100-pixel
  // tiles gave 1376 blocks = 1.16 waves at 64x64x320, batch 32: the second wave ran 16 % full)
  const int64_t per_sample = std::max<int64_t>(1, (148 * 3) / B);  // 3 resident blocks per SM (launch bounds)
  const int ppb = static_cast<int>(std::max<int64_t>(1, (P + per_sample - 1) / per_sample));
  const unsigned tiles = static_cast<unsigned>((P + ppb - 1) / ppb);
  gn_apply_kernel<<<dim3(tiles, B), 256, static_cast<size_t>(2) * C * sizeof(float), stream>>>(x, ldx, C, G, P, stats, gamma,
                                                                                            beta, silu, y, ldy, ppb);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// =============================================================================================
// LayerNorm over the channel dim: one warp per token row, fp32 two-pass in registers.
// =============================================================================================
template <int MAXV, int R>  // 16-byte vectors per lane per row, rows per warp (independent loads in flight)
__global__ void __launch_bounds__(256) layernorm_kernel(const __half* __restrict__ x, int64_t ldx, int64_t rows,
                                                        int C, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps,
                                                        __half* __restrict__ y, int64_t ldy) {
  // blocks walk the rows from the END — the tail of the tensor is what the L2 still holds of the producing GEMM's
  // output, and the consumer GEMM then finds the head of the normalised tensor (written last) in L2
  const int64_t blk = static_cast<int64_t>(gridDim.x) - 1 - blockIdx.x;
  const int64_t row0 = (blk * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R;
  if (row0 >= rows) return;
  const int lane = threadIdx.x & 31;
  const int vecs = C / 8;
  uint4 u[R][MAXV];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = lane + i * 32;
      if (vi < vecs && row0 + r < rows) u[r][i] = *reinterpret_cast<const uint4*>(x + (row0 + r) * ldx + vi * 8);
    }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t row = row0 + r;
    if (row >= rows) break;  // warp-uniform
    float v[MAXV][8];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = lane + i * 32;
      if (vi < vecs) {
        const __half2* h = reinterpret_cast<const __half2*>(&u[r][i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(h[j]);
          v[i][2 * j] = f.x;
          v[i][2 * j + 1] = f.y;
          sum += f.x + f.y;
        }
      }
    }
    sum = warp_sum(sum);
    const float mean = sum / C;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = lane + i * 32;
      if (vi < vecs) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float d = v[i][j] - mean;
          sq = fmaf(d, d, sq);
        }
      }
    }
    sq = warp_sum(sq);
    const float rstd = rsqrtf(sq / C + eps);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int vi = lane + i * 32;
      if (vi < vecs) {
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + vi * 8) + 1);
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + vi * 8));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(beta + vi * 8) + 1);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * gg[j] + bb[j];
        uint4 w;
        w.x = pack_h2(o[0], o[1]);
        w.y = pack_h2(o[2], o[3]);
        w.z = pack_h2(o[4], o[5]);
        w.w = pack_h2(o[6], o[7]);
        *reinterpret_cast<uint4*>(y + row * ldy + vi * 8) = w;
      }
    }
  }
}

// LayerNorm for C = 40 * LPR (320 / 640 / 1280: every width of the SD UNets): LPR lanes share a row, five 16-byte vectors
// per lane, so all 32 lanes carry data (the generic kernel runs its second vector slot 25 % full at C = 320), the
// reductions stay inside LPR-lane groups, the arithmetic is packed fp32x2 and gamma / beta come from shared memory.
// ncu on the generic kernel at C = 320: issue slots 65 % busy at 34 % occupancy and 37 % of the DRAM peak — it was bound
// by its instruction count (~200 per 16-byte vector), not by HBM (profiles/r02_ncu_norms.txt).
// (A persistent "streaming" form of the generic kernel — fixed grid, next row group's loads in flight — was measured
//  SLOWER, 112 vs 87 us at C = 320, and dropped: the loads were never the problem.)
template <int LPR, int ITER>
__global__ void __launch_bounds__(256) layernorm_c40_kernel(const __half* __restrict__ x, int64_t ldx, int64_t rows,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps,
                                                            __half* __restrict__ y, int64_t ldy) {
  constexpr int C = 40 * LPR, RW = 32 / LPR;  // channels; rows per warp and iteration
  extern __shared__ float ln_gb[];             // [C] gamma, [C] beta
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    ln_gb[c] = gamma[c];
    ln_gb[C + c] = beta[c];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane % LPR, rsel = lane / LPR;  // position inside the row's lane group; which of the warp's rows
  const int64_t blk = static_cast<int64_t>(gridDim.x) - 1 - blockIdx.x;  // back to front, as layernorm_kernel
  const int64_t row_base = (blk * (blockDim.x >> 5) + warp) * (RW * ITER);
  uint4 u[ITER][5];
#pragma unroll
  for (int it = 0; it < ITER; ++it) {
    const int64_t row = row_base + it * RW + rsel;
    if (row < rows) {
#pragma unroll
      for (int i = 0; i < 5; ++i) u[it][i] = *reinterpret_cast<const uint4*>(x + row * ldx + (sub + i * LPR) * 8);
    }
  }
  const float inv_c = 1.f / C;
#pragma unroll
  for (int it = 0; it < ITER; ++it) {
    const int64_t row = row_base + it * RW + rsel;
    const bool ok = row < rows;  // whole lane groups are in or out; the shuffles below stay inside a group
    uint64_t v[5][4];
    uint64_t s2 = pk2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const __half2* h = reinterpret_cast<const __half2*>(&u[it][i]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = ok ? __half22float2(h[j]) : make_float2(0.f, 0.f);
        v[i][j] = pk2(f.x, f.y);
        s2 = add2(s2, v[i][j]);
      }
    }
    float sa, sb;
    upk2(s2, sa, sb);
    float sum = sa + sb;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * inv_c;
    const uint64_t nm2 = pk2(-mean, -mean);
    uint64_t q2 = pk2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[i][j] = add2(v[i][j], nm2);
        q2 = fma2(v[i][j], v[i][j], q2);
      }
    upk2(q2, sa, sb);
    float sq = sa + sb;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq * inv_c + eps);
    const uint64_t r2 = pk2(rstd, rstd);
    if (ok) {
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int c0 = (sub + i * LPR) * 8;
        const float4 g0 = *reinterpret_cast<const float4*>(ln_gb + c0), g1 = *reinterpret_cast<const float4*>(ln_gb + c0 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(ln_gb + C + c0), b1 = *reinterpret_cast<const float4*>(ln_gb + C + c0 + 4);
        float o0, o1, o2, o3, o4, o5, o6, o7;
        upk2(fma2(mul2(v[i][0], r2), pk2(g0.x, g0.y), pk2(b0.x, b0.y)), o0, o1);
        upk2(fma2(mul2(v[i][1], r2), pk2(g0.z, g0.w), pk2(b0.z, b0.w)), o2, o3);
        upk2(fma2(mul2(v[i][2], r2), pk2(g1.x, g1.y), pk2(b1.x, b1.y)), o4, o5);
        upk2(fma2(mul2(v[i][3], r2), pk2(g1.z, g1.w), pk2(b1.z, b1.w)), o6, o7);
        *reinterpret_cast<uint4*>(y + row * ldy + c0) =
            make_uint4(pack_h2(o0, o1), pack_h2(o2, o3), pack_h2(o4, o5), pack_h2(o6, o7));
      }
    }
  }
}

template <int LPR>
static int launch_ln_c40(const __half* x, int64_t ldx, int64_t rows, const float* gamma, const float* beta, float eps,
                         __half* y, int64_t ldy, cudaStream_t stream) {
  constexpr int ITER = 2, C = 40 * LPR;
  const int64_t rows_per_block = 8 * (32 / LPR) * ITER;
  const unsigned blocks = static_cast<unsigned>((rows + rows_per_block - 1) / rows_per_block);
  layernorm_c40_kernel<LPR, ITER><<<blocks, 256, static_cast<size_t>(2) * C * sizeof(float), stream>>>(x, ldx, rows, gamma,
                                                                                                      beta, eps, y, ldy);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

int layernorm(const __half* x, int64_t ldx, int64_t rows, int C, const float* gamma, const float* beta, float eps,
              __half* y, int64_t ldy, cudaStream_t stream) {
  SDW_REQUIRE(C % 8 == 0 && C <= 8 * 32 * 8, "LayerNorm: C % 8 == 0 and C <= 2048");
  const int vecs = C / 8;
  // the UNet widths take the lane-group kernel
  const bool vec_ok = (ldx % 8 == 0) && (ldy % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0 &&
                      ((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0;
  if (vec_ok) {
    if (C == 320) return launch_ln_c40<8>(x, ldx, rows, gamma, beta, eps, y, ldy, stream);
    if (C == 640) return launch_ln_c40<16>(x, ldx, rows, gamma, beta, eps, y, ldy, stream);
    if (C == 1280) return launch_ln_c40<32>(x, ldx, rows, gamma, beta, eps, y, ldy, stream);
  }
  if (vecs <= 64) {
    const unsigned blocks = static_cast<unsigned>((rows + 31) / 32);
    layernorm_kernel<2, 4><<<blocks, 256, 0, stream>>>(x, ldx, rows, C, gamma, beta, eps, y, ldy);
  } else if (vecs <= 160) {
    const unsigned blocks = static_cast<unsigned>((rows + 15) / 16);
    layernorm_kernel<5, 2><<<blocks, 256, 0, stream>>>(x, ldx, rows, C, gamma, beta, eps, y, ldy);
  } else {
    const unsigned blocks = static_cast<unsigned>((rows + 7) / 8);
    layernorm_kernel<8, 1><<<blocks, 256, 0, stream>>>(x, ldx, rows, C, gamma, beta, eps, y, ldy);
  }
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// =============================================================================================
// row softmax in place (scores already scaled by the QK^T epilogue): one warp per row for n <= 1024,
// one 256-thread block per row otherwise.  fp32 math, fp16 storage.
// =============================================================================================
__global__ void __launch_bounds__(256) softmax_warp_kernel(__half* __restrict__ s, int64_t ld, int64_t rows, int n) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  __half* r = s + row * ld;
  float v[32];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + i * 32;
    v[i] = c < n ? __half2float(r[c]) : -INFINITY;
    m = fmaxf(m, v[i]);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + i * 32;
    v[i] = c < n ? __expf(v[i] - m) : 0.f;
    sum += v[i];
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + i * 32;
    if (c < n) r[c] = __float2half_rn(v[i] * inv);
  }
}

__global__ void __launch_bounds__(256) softmax_block_kernel(__half* __restrict__ s, int64_t ld, int n) {
  __shared__ float red[32];
  __half* r = s + static_cast<int64_t>(blockIdx.x) * ld;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float m = -INFINITY;
  for (int c = threadIdx.x; c < n; c += blockDim.x) m = fmaxf(m, __half2float(r[c]));
  m = warp_max(m);
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = lane < (blockDim.x >> 5) ? red[lane] : -INFINITY;
  m = warp_max(m);
  __syncthreads();
  float sum = 0.f;
  for (int c = threadIdx.x; c < n; c += blockDim.x) sum += __expf(__half2float(r[c]) - m);
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int c = threadIdx.x; c < n; c += blockDim.x) r[c] = __float2half_rn(__expf(__half2float(r[c]) - m) * inv);
}

int softmax_rows(__half* s, int64_t ld, int64_t rows, int n, cudaStream_t stream) {
  SDW_REQUIRE(n > 0 && rows > 0, "softmax: empty");
  if (n <= 1024)
    softmax_warp_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, stream>>>(s, ld, rows, n);
  else
    softmax_block_kernel<<<static_cast<unsigned>(rows), 256, 0, stream>>>(s, ld, n);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// =============================================================================================
// conv_in: 3x3 pad 1, tiny Cin (4) -> N channels.  Block = N threads (one output channel each, weights in
// registers), loops over a tile of pixels whose 3x3xCin patches sit in shared memory.
// w layout: [N][Cin][3][3] fp16 (the checkpoint's OIHW), bias fp32.
// =============================================================================================
__device__ __forceinline__ float in_val(__half v) { return __half2float(v); }
__device__ __forceinline__ float in_val(uint8_t v) { return static_cast<float>(v) / 255.f; }  // Real-ESRGAN: img / 255

template <int CIN, typename TIn = __half>
__global__ void __launch_bounds__(512) conv_in_kernel(const TIn* __restrict__ x, int64_t ldx, int B, int H, int W,
                                                       const __half* __restrict__ w, const float* __restrict__ bias,
                                                       int N, __half* __restrict__ y, int64_t ldy,
                                                       int pix_per_block) {
  // patch[pair][k] = (x of pixel 2*pair, x of pixel 2*pair + 1) for the 9*CIN taps: one 16-byte broadcast read feeds two
  // packed FMAs (two taps x two pixels); thread = output channel, its 9*CIN weights live in registers
  constexpr int K = 9 * CIN;
  constexpr int KP = (K + 1) & ~1;  // an even row length keeps the 16-byte reads aligned; the pad tap is zero
  extern __shared__ float2 patch2[];  // [pix_per_block / 2][KP]
  const int64_t P = static_cast<int64_t>(B) * H * W;
  const int64_t p0 = static_cast<int64_t>(blockIdx.x) * pix_per_block;
  const int np = static_cast<int>(min(static_cast<int64_t>(pix_per_block), P - p0));
  for (int i = threadIdx.x; i < pix_per_block * KP; i += blockDim.x) {
    const int k = i % KP;
    const int c = k % CIN;
    const int tap = k / CIN;
    const int lp = i / KP;
    const int64_t p = p0 + lp;
    float v = 0.f;
    if (lp < np && k < K) {
      const int xw = static_cast<int>(p % W), yh = static_cast<int>((p / W) % H);
      const int64_t b = p / (static_cast<int64_t>(W) * H);
      const int yy = yh + tap / 3 - 1, xx = xw + tap % 3 - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = in_val(x[((b * H + yy) * W + xx) * ldx + c]);
    }
    reinterpret_cast<float*>(patch2)[((lp >> 1) * KP + k) * 2 + (lp & 1)] = v;
  }
  __syncthreads();
  const int n = threadIdx.x;
  if (n >= N) return;
  uint64_t wr[KP];
  wr[KP - 1] = 0;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap)
#pragma unroll
    for (int c = 0; c < CIN; ++c) {
      const float wv = __half2float(w[(static_cast<int64_t>(n) * CIN + c) * 9 + tap]);
      wr[tap * CIN + c] = pk2(wv, wv);
    }
  const float bn = bias ? bias[n] : 0.f;
  for (int pr = 0; pr * 2 < np; ++pr) {
    uint64_t acc = pk2(bn, bn);
    const float4* row = reinterpret_cast<const float4*>(patch2 + pr * KP);
#pragma unroll
    for (int k = 0; k < KP / 2; ++k) {
      const float4 v = row[k];
      acc = fma2(pk2(v.x, v.y), wr[2 * k], acc);
      acc = fma2(pk2(v.z, v.w), wr[2 * k + 1], acc);
    }
    float a0, a1;
    upk2(acc, a0, a1);
    y[(p0 + 2 * pr) * ldy + n] = __float2half_rn(a0);
    if (2 * pr + 1 < np) y[(p0 + 2 * pr + 1) * ldy + n] = __float2half_rn(a1);
  }
}

int conv_in_small(const __half* x, int64_t ldx, int B, int H, int W, int Cin, const __half* w, const float* bias,
                  int N, __half* y, int64_t ldy, cudaStream_t stream) {
  SDW_REQUIRE(Cin == 4, "conv_in: latent channel count must be 4");
  SDW_REQUIRE(N <= 512, "conv_in: N <= 512");
  const int ppb = 64;
  const int64_t P = static_cast<int64_t>(B) * H * W;
  const int threads = (N + 31) / 32 * 32;
  conv_in_kernel<4><<<static_cast<unsigned>((P + ppb - 1) / ppb), threads, ppb * 36 * sizeof(float), stream>>>(
      x, ldx, B, H, W, w, bias, N, y, ldy, ppb);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

int conv_in_u8(const uint8_t* x, int B, int H, int W, const __half* w, const float* bias, int N, __half* y,
               int64_t ldy, cudaStream_t stream) {
  SDW_REQUIRE(N <= 512, "conv_in: N <= 512");
  const int ppb = 64;
  const int64_t P = static_cast<int64_t>(B) * H * W;
  const int threads = (N + 31) / 32 * 32;
  conv_in_kernel<3, uint8_t><<<static_cast<unsigned>((P + ppb - 1) / ppb), threads, ppb * 28 * sizeof(float), stream>>>(
      x, 3, B, H, W, w, bias, N, y, ldy, ppb);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// =============================================================================================
// conv_out: 3x3 pad 1, C -> NOUT (<= 4) channels, one warp per output pixel; lanes split the channels.
// Input is the already normalised + SiLU'd fp16 NHWC tensor.  w layout: OIHW fp16 [NOUT][C][3][3].
//   out_f32  : fp32 NHWC [P][NOUT] (UNet eps)          — optional
//   out_u8   : uint8 NHWC [P][NOUT] = round(clamp(v/2+0.5,0,1)*255) (VAE frame; P:435-438 + numpy_to_pil) — optional;
//              UNIT01: round(clamp(v,0,1)*255) (Real-ESRGAN's output post-process)
// =============================================================================================
// A block owns a TS x TS pixel tile: its (TS+2)^2 halo is staged once in shared memory (the row-per-warp version
// re-read every input pixel nine times from L2: 245 us for the UNet's 320->4 conv, ~6 ms for the VAE's 128->3), the
// weights sit next to it; a warp computes 8 pixels at a time, lanes split the channels, one tap's weights in registers.
template <int NOUT, int TS, bool UNIT01 = false>
__global__ void __launch_bounds__(256) conv_out_kernel(const __half* __restrict__ x, int64_t ldx, int B, int H, int W,
                                                       int C, const __half* __restrict__ w,
                                                       const float* __restrict__ bias, float* __restrict__ out_f32,
                                                       uint8_t* __restrict__ out_u8) {
  constexpr int HT = TS + 2;
  extern __shared__ __align__(16) uint8_t co_smem[];
  __half* halo = reinterpret_cast<__half*>(co_smem);  // [HT*HT][C]
  __half* ws = halo + HT * HT * C;                     // [NOUT][9][C]
  const int tiles_x = (W + TS - 1) / TS, tiles_y = (H + TS - 1) / TS;
  const int ntiles = B * tiles_x * tiles_y;
  // OIHW -> [n][tap][c], once per (persistent) block: 16-byte loads along the source, eight in flight per thread
  {
    const int nvec = NOUT * 9 * C / 8;  // C % 8 == 0
    for (int v0 = threadIdx.x; v0 < nvec; v0 += 4 * blockDim.x) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int v = v0 + k * blockDim.x;
        u[k] = v < nvec ? __ldg(reinterpret_cast<const uint4*>(w) + v) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int v = v0 + k * blockDim.x;
        if (v >= nvec) continue;
        const __half* h = reinterpret_cast<const __half*>(&u[k]);
        int i = v * 8;
        int n = i / (9 * C), rem = i - n * 9 * C;
        int c = rem / 9, tap = rem - c * 9;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          ws[(n * 9 + tap) * C + c] = h[e];
          if (++tap == 9) {
            tap = 0;
            if (++c == C) {
              c = 0;
              ++n;
            }
          }
        }
      }
    }
  }
  const int c8n = C / 8;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
  const int tx = tile % tiles_x, ty = (tile / tiles_x) % tiles_y;
  const int64_t b = tile / (tiles_x * tiles_y);
  const int x0 = tx * TS, y0 = ty * TS;
  __syncthreads();  // the previous tile's halo has been consumed (and the weights are staged)
  for (int i0 = threadIdx.x; i0 < HT * HT * c8n; i0 += 4 * blockDim.x) {
    uint4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * blockDim.x;
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      if (i < HT * HT * c8n) {
        const int c8 = i % c8n, hp = i / c8n;
        const int yy = y0 + hp / HT - 1, xx = x0 + hp % HT - 1;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W)
          v[k] = *reinterpret_cast<const uint4*>(x + ((b * H + yy) * W + xx) * ldx + c8 * 8);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * blockDim.x;
      if (i < HT * HT * c8n) *reinterpret_cast<uint4*>(halo + (i / c8n) * C + (i % c8n) * 8) = v[k];
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // group g of warp `warp`: pixels q = (g * 8 + warp) * 8 + j, j < 8 — eight consecutive pixels of one tile row
  for (int g = 0; g * 64 + warp * 8 < TS * TS; ++g) {
    const int q0 = (g * 8 + warp) * 8;
    const int py = q0 / TS, px0 = q0 % TS;
    float acc[8][NOUT];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int n = 0; n < NOUT; ++n) acc[j][n] = 0.f;
    for (int tap = 0; tap < 9; ++tap) {
      const __half* hrow = halo + ((py + tap / 3) * HT + px0 + tap % 3) * C;
      for (int c = lane * 2; c < C; c += 64) {
        float2 wv[NOUT];
#pragma unroll
        for (int n = 0; n < NOUT; ++n) wv[n] = __half22float2(*reinterpret_cast<const __half2*>(&ws[(n * 9 + tap) * C + c]));
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 xv = __half22float2(*reinterpret_cast<const __half2*>(hrow + j * C + c));
#pragma unroll
          for (int n = 0; n < NOUT; ++n) {
            acc[j][n] = fmaf(xv.x, wv[n].x, acc[j][n]);
            acc[j][n] = fmaf(xv.y, wv[n].y, acc[j][n]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int n = 0; n < NOUT; ++n) acc[j][n] = warp_sum(acc[j][n]);
    // lane j < 8 writes pixel j
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (lane == j) {
        const int yy = y0 + py, xx = x0 + px0 + j;
        if (yy < H && xx < W) {
          const int64_t p = (b * H + yy) * W + xx;
#pragma unroll
          for (int n = 0; n < NOUT; ++n) {
            const float v = acc[j][n] + (bias ? bias[n] : 0.f);
            if (out_f32) out_f32[p * NOUT + n] = v;
            if (out_u8) {
              const float q = fminf(fmaxf(UNIT01 ? v : v * 0.5f + 0.5f, 0.f), 1.f);
              out_u8[p * NOUT + n] = static_cast<uint8_t>(rintf(q * 255.f));
            }
          }
        }
      }
    }
  }
  }  // tile loop
}

template <int NOUT, int TS, bool UNIT01 = false>
static int launch_conv_out(const __half* x, int64_t ldx, int B, int H, int W, int C, const __half* w, const float* bias,
                           float* out_f32, uint8_t* out_u8, cudaStream_t stream) {
  const size_t smem = (static_cast<size_t>((TS + 2) * (TS + 2)) + NOUT * 9) * C * sizeof(__half);
  SDW_REQUIRE(smem <= 227 * 1024, "conv_out: channel count too large for the halo tile");
  static bool attr_done = false;
  if (!attr_done) {
    SDW_CUDA_OK(cudaFuncSetAttribute(conv_out_kernel<NOUT, TS, UNIT01>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_done = true;
  }
  const int64_t tiles = static_cast<int64_t>(B) * ((H + TS - 1) / TS) * ((W + TS - 1) / TS);
  const int64_t blocks = std::min<int64_t>(tiles, 148 * 2);  // persistent: the weights are staged once per block
  conv_out_kernel<NOUT, TS, UNIT01><<<static_cast<unsigned>(blocks), 256, smem, stream>>>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

int conv_out_small(const __half* x, int64_t ldx, int B, int H, int W, int C, const __half* w, const float* bias,
                   int nout, float* out_f32, uint8_t* out_u8, cudaStream_t stream, int unit01) {
  SDW_REQUIRE(nout == 3 || nout == 4, "conv_out: 3 or 4 output channels");
  SDW_REQUIRE(C % 8 == 0 && ldx % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "conv_out: 16-byte aligned channel rows");
  // 16 x 16 tiles when their halo fits comfortably (C <= 128), 8 x 8 otherwise
  const bool big = C <= 128 && H >= 16 && W >= 16;
  if (unit01) {
    SDW_REQUIRE(nout == 3, "conv_out: the [0, 1] post-process is for RGB output");
    return big ? launch_conv_out<3, 16, true>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream)
               : launch_conv_out<3, 8, true>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream);
  }
  if (nout == 4)
    return big ? launch_conv_out<4, 16>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream)
               : launch_conv_out<4, 8>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream);
  return big ? launch_conv_out<3, 16>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream)
             : launch_conv_out<3, 8>(x, ldx, B, H, W, C, w, bias, out_f32, out_u8, stream);
}

// =============================================================================================
// VAE input: z = post_quant_conv(latents / scaling) ; latents fp32 NCHW [F][C][H][W] -> fp16 NHWC [F][H][W][C]
// (stable_diffusion_pipeline.py:432 `1 / 0.18215 * latents`, then AutoencoderKL.decode's post_quant_conv 1x1)
// =============================================================================================
__global__ void vae_in_kernel(const float* __restrict__ x, float inv_scale, const __half* __restrict__ w,
                              const float* __restrict__ bias, int F, int C, int H, int W, __half* __restrict__ z) {
  const int64_t P = static_cast<int64_t>(F) * H * W;
  const int64_t p = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int64_t hw = static_cast<int64_t>(H) * W;
  const int64_t f = p / hw, r = p % hw;
  float in[8];
  for (int c = 0; c < C; ++c) in[c] = x[(f * C + c) * hw + r] * inv_scale;
  for (int n = 0; n < C; ++n) {
    float acc = bias ? bias[n] : 0.f;
    for (int c = 0; c < C; ++c) acc = fmaf(in[c], __half2float(w[n * C + c]), acc);
    z[p * C + n] = __float2half_rn(acc);
  }
}

int vae_in(const float* x, float inv_scale, const __half* w, const float* bias, int F, int C, int H, int W, __half* z,
           cudaStream_t stream) {
  SDW_REQUIRE(C <= 8, "latent channels <= 8");
  const int64_t P = static_cast<int64_t>(F) * H * W;
  vae_in_kernel<<<static_cast<unsigned>((P + 255) / 256), 256, 0, stream>>>(x, inv_scale, w, bias, F, C, H, W, z);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// =============================================================================================
// fp32 small linear: out[m][n] = act_out( bias[n] + sum_k act_in(in[m][k]) * W[n][k] ), W fp16 [N][K].
// One warp per output element.  Used for the time-embedding MLP and the 22 ResBlock time projections,
// evaluated once per schedule for ALL timesteps (they depend on t only — SURVEY.md K8).
// =============================================================================================
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ in, int64_t ldi,
                                                         const __half* __restrict__ w, const float* __restrict__ bias,
                                                         int M, int N, int K, int silu_in, int silu_out,
                                                         float* __restrict__ out, int64_t ldo) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (idx >= static_cast<int64_t>(M) * N) return;
  const int m = static_cast<int>(idx / N), n = static_cast<int>(idx % N);
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) {
    float a = in[m * ldi + k];
    if (silu_in) a = silu_f(a);
    acc = fmaf(a, __half2float(w[static_cast<int64_t>(n) * K + k]), acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    acc += bias ? bias[n] : 0.f;
    if (silu_out) acc = silu_f(acc);
    out[m * ldo + n] = acc;
  }
}

int linear_f32(const float* in, int64_t ldi, const __half* w, const float* bias, int M, int N, int K, int silu_in,
               int silu_out, float* out, int64_t ldo, cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(M) * N;
  linear_f32_kernel<<<static_cast<unsigned>((total + 7) / 8), 256, 0, stream>>>(in, ldi, w, bias, M, N, K, silu_in,
                                                                                 silu_out, out, ldo);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// sinusoidal timestep embedding, flip_sin_to_cos = True, freq_shift = 0: out[s] = cat[cos(t f), sin(t f)]
// rounded to fp16 like the reference's `.to(dtype=self.dtype)` cast before time_embedding.
__global__ void timestep_embed_kernel(const float* __restrict__ t, int n, int dim, int round_f16,
                                      float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * dim) return;
  const int s = i / dim, j = i % dim;
  const int half = dim / 2;
  const int k = j % half;
  const float freq = expf(-logf(10000.f) * static_cast<float>(k) / static_cast<float>(half));
  const float a = t[s] * freq;
  float v = j < half ? cosf(a) : sinf(a);
  if (round_f16) v = __half2float(__float2half_rn(v));
  out[i] = v;
}

int timestep_embed(const float* t, int n, int dim, int round_f16, float* out, cudaStream_t stream) {
  timestep_embed_kernel<<<(n * dim + 255) / 256, 256, 0, stream>>>(t, n, dim, round_f16, out);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

// fp16 -> fp32 vector conversion (biases, norm affine parameters)
__global__ void h2f_kernel(const __half* __restrict__ in, float* __restrict__ out, int64_t n, const int* perm_geglu,
                           int N) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t src = i;
  if (N > 0) {  // GEGLU bias interleave, same row permutation as pack_weight
    const int r = static_cast<int>(i);
    const int blk = r >> 6, within = r & 63;
    src = within < 32 ? blk * 32 + within : N / 2 + blk * 32 + (within - 32);
  }
  out[i] = __half2float(in[src]);
}

int half_to_float(const __half* in, float* out, int64_t n, int geglu_N, cudaStream_t stream) {
  h2f_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(in, out, n, nullptr, geglu_N);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace sdw
