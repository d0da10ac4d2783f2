// sdw_gemm.cu — the tcgen05 implicit-GEMM kernel behind every Conv2d 3x3 / 1x1,
// Linear and batched matmul of the UNet2DCondition / AutoencoderKL-decoder hot path
// (reference call sites: stable_diffusion_pipeline.py:418 `self.unet(...)`, :433 `self.vae.decode`).
//
// Shape of the kernel (one 128 x BN output tile per CTA, 2 CTAs co-resident per SM):
//   warp 0    : TMA producer — per K block (tap, 64-channel chunk) one 4-D box load of the
//               shifted NHWC activation tile (OOB halo = zero fill = conv padding) and one
//               box of the K-major weight tile, SWIZZLE_128B, into a STAGES-deep smem ring.
//   warp 1    : TMEM allocator + MMA issuer — one elected thread issues 4 x tcgen05.mma
//               (M=128, N=BN, K=16) per K block, accumulating fp32 in TMEM; tcgen05.commit
//               releases the smem stage / signals the epilogue.
//   warps 2-5 : epilogue — tcgen05.ld the accumulator (thread = output row), fuse
//               alpha / bias / time-embedding row vector / SiLU / residual / GEGLU /
//               per-head V^T scatter, write fp16.
#include "sdw_internal.h"
#include "sdw_gemm_epi.cuh"
#include "sdw_ptx.cuh"

#include <cudaTypedefs.h>

#include <algorithm>
#include <cstring>

namespace sdw {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KiB
static constexpr int GEMM_THREADS = 192;

template <int BN>
struct GemmCfg {
  static constexpr int B_STAGE_BYTES = BN * BK * 2;
  static constexpr int STAGES = BN <= 64 ? 4 : 3;
  static constexpr int TMEM_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
  static constexpr int SMEM_BYTES = STAGES * (A_STAGE_BYTES + B_STAGE_BYTES) + 1024 /*align*/ + 256 /*barriers*/;
};

template <int BN>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_tc_kernel(const __grid_constant__ GemmKParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * A_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_b + STAGES * Cfg::B_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- tile coordinates -------------------------------------------------
  const int m_tile = blockIdx.x;
  const int tw = m_tile % p.tiles_w;
  const int th = (m_tile / p.tiles_w) % p.tiles_h;
  const int tb = m_tile / (p.tiles_w * p.tiles_h);
  const int x0 = tw * p.bw, y0 = th * p.bh, b0 = tb * p.bb;
  const int n0 = blockIdx.y * BN;
  const int num_kb = p.ntaps * p.kchunks;

  // ---- one-time setup -----------------------------------------------------
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.mapA[0]);
    tma_prefetch_desc(&p.mapB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_ptr_smem;

  if (warp == 0) {
    // =========================== TMA producer ===============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        const int tap = kb / p.kchunks;
        const int kc = kb - tap * p.kchunks;
        mbar_expect_tx(&full_bar[stage], A_STAGE_BYTES + Cfg::B_STAGE_BYTES);
        tma_load_4d(&p.mapA[p.tap_map[tap]], &full_bar[stage], smem_a + stage * A_STAGE_BYTES, kc * BK,
                    x0 + p.tap_dx[tap], y0 + p.tap_dy[tap], b0);
        tma_load_4d(&p.mapB, &full_bar[stage], smem_b + stage * Cfg::B_STAGE_BYTES, kb * BK, n0,
                    p.b_batched ? y0 : 0, p.b_batched ? b0 : 0);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===================================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint64_t da = make_desc_k_sw128(smem_u32(smem_a + stage * A_STAGE_BYTES));
        const uint64_t db = make_desc_k_sw128(smem_u32(smem_b + stage * Cfg::B_STAGE_BYTES));
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // advance 16 fp16 = 32 B inside the 128-B swizzle row: +2 in the (>>4) address field
          umma_f16_ss(tmem_acc, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[stage]);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      umma_commit(tmem_full_bar);
    }
  } else {
    // =========================== epilogue ======================================
    gemm_epilogue<BN>(p, tmem_acc, warp, lane, x0, y0, b0, n0, tmem_full_bar);
  }

  // ---- teardown -------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_acc, Cfg::TMEM_COLS);
  }
}

// =============================================================================
// host side
// =============================================================================
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static bool g_plan_only = false;  // validate plans without a driver (CPU-side tests); nothing can be launched
void set_plan_only(bool on) { g_plan_only = on; }

template <int BN>
static int set_attr() {
  SDW_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   GemmCfg<BN>::SMEM_BYTES));
  return 0;
}

int gemm_init() {
  if (g_encode || g_plan_only) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  SDW_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (qres != cudaDriverEntryPointSuccess || !fn) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return 2;
  }
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  if (int e = set_attr<32>()) return e;
  if (int e = set_attr<64>()) return e;
  if (int e = set_attr<128>()) return e;
  if (int e = set_attr<160>()) return e;
  return 0;
}

// rank-`rank` fp16 tensor map, dim 0 contiguous, SWIZZLE_128B, zero OOB fill.
int encode_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
               const uint32_t* box, int swizzle_bytes) {
  if (int e = gemm_init()) return e;
  cuuint64_t gdim[5];
  cuuint64_t gstride[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) {
      gstride[i - 1] = strides_elems[i] * 2;
      if (gstride[i - 1] % 16 != 0) {
        set_error("TMA global stride must be a multiple of 16 bytes");
        return 1;
      }
    }
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0) {
    set_error("TMA global base must be 16-byte aligned");
    return 1;
  }
  for (int i = 0; i < rank; ++i) {
    if (bx[i] == 0 || bx[i] > 256 || gdim[i] == 0) {
      set_error("TMA box dims must be in 1..256 and tensor dims non-zero");
      return 1;
    }
  }
  if (g_plan_only) return 0;
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, const_cast<void*>(base), gdim, gstride, bx, es,
                        CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle_bytes == 0 ? CU_TENSOR_MAP_SWIZZLE_NONE
                                           : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B),
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return 2;
  }
  return 0;
}

static int pow2_floor(int v) {
  int p = 1;
  while (p * 2 <= v) p *= 2;
  return p;
}

int plan_gemm(const GemmDesc& d, GemmLaunch* L) {
  SDW_REQUIRE(d.A && d.Wt && d.out, "null operand");
  SDW_REQUIRE(d.C > 0 && d.W > 0 && d.H > 0 && d.B > 0 && d.N > 0, "empty problem");
  SDW_REQUIRE(d.act >= 0 && d.act <= 2, "act: 0 none, 1 SiLU, 2 LeakyReLU(0.2)");
  SDW_REQUIRE(!d.resid2 || (d.resid && d.mode == GEMM_PLAIN), "a second residual needs a first one and plain mode");
  GemmKParams& p = L->p;
  std::memset(&p, 0, sizeof(p));
  const int kchunks = (d.C + BK - 1) / BK;
  const int Cp = kchunks * BK;
  p.kchunks = kchunks;
  p.ntaps = d.conv == 0 ? 1 : (d.conv == 3 ? 4 : 9);
  // domain (lattice the M tiles walk over) and the tap table
  int Wd = d.W, Hd = d.H;
  int nmaps = 1;
  p.os = 1;
  p.ox = p.oy = 0;
  if (d.conv == 0) {
    p.tap_map[0] = 0;
    p.tap_dx[0] = p.tap_dy[0] = 0;
  } else if (d.conv == 1) {
    for (int t = 0; t < 9; ++t) {
      p.tap_map[t] = 0;
      p.tap_dy[t] = static_cast<int8_t>(t / 3 - 1);
      p.tap_dx[t] = static_cast<int8_t>(t % 3 - 1);
    }
  } else if (d.conv == 2) {
    SDW_REQUIRE(d.W % 2 == 0 && d.H % 2 == 0, "stride-2 conv needs even extents");
    Wd = d.W / 2;
    Hd = d.H / 2;
    nmaps = 4;
    // in = 2*o + k - 1 : k=0 -> parity 1 shift -1 ; k=1 -> parity 0 shift 0 ; k=2 -> parity 1 shift 0
    const int par[3] = {1, 0, 1};
    const int sh[3] = {-1, 0, 0};
    for (int t = 0; t < 9; ++t) {
      const int ky = t / 3, kx = t % 3;
      p.tap_map[t] = static_cast<int8_t>(par[ky] * 2 + par[kx]);
      p.tap_dy[t] = static_cast<int8_t>(sh[ky]);
      p.tap_dx[t] = static_cast<int8_t>(sh[kx]);
    }
  } else if (d.conv == 3) {
    // nearest-up x2 then 3x3, folded into a 2x2 conv per output parity (weights from pack_weight_up4):
    // parity 0 reads low-res rows {yo-1, yo}, parity 1 reads {yo, yo+1}; same for columns
    for (int t = 0; t < 4; ++t) {
      const int a = t >> 1, b = t & 1;
      p.tap_map[t] = 0;
      p.tap_dy[t] = static_cast<int8_t>(d.up_py ? a : a - 1);
      p.tap_dx[t] = static_cast<int8_t>(d.up_px ? b : b - 1);
    }
    p.os = 2;
    p.ox = d.up_px;
    p.oy = d.up_py;
  } else {
    SDW_REQUIRE(false, "unknown conv kind");
  }
  p.W = Wd;
  p.H = Hd;
  p.B = d.B;
  const int64_t OW = static_cast<int64_t>(Wd) * p.os, OH = static_cast<int64_t>(Hd) * p.os;
  // tile geometry: bw*bh*bb = 128
  int bw = std::min(pow2_floor(Wd), BM);
  if (Wd > BM) bw = BM;
  int bh = std::min(pow2_floor(Hd), BM / bw);
  int bb = BM / (bw * bh);
  if (d.b_batched) {
    SDW_REQUIRE(d.conv == 0, "batched matmul is 1x1");
    bw = BM;
    bh = 1;
    bb = 1;
  }
  p.bw = bw;
  p.bh = bh;
  p.bb = bb;
  p.tiles_w = (Wd + bw - 1) / bw;
  p.tiles_h = (Hd + bh - 1) / bh;
  const int tiles_b = (d.B + bb - 1) / bb;
  p.N = d.N;
  p.b_batched = d.b_batched;
  // kernel version: CTA pairs need >= 2 M tiles and a wide-enough N; batched matmuls must pair within one (h, b)
  const int m_tiles = p.tiles_w * p.tiles_h * tiles_b;
  int ver = d.ver;
  if (ver == 0) ver = (m_tiles >= 2 && d.N >= 128 && (!d.b_batched || p.tiles_w % 2 == 0)) ? 2 : 1;
  if (ver == 2) SDW_REQUIRE(!d.b_batched || p.tiles_w % 2 == 0, "2-CTA batched matmul needs an even tile count per row");
  // tap reuse (3x3 stride 1, CTA pairs): 16 x 8-pixel tiles, one 10-row activation box per (channel chunk, kx).  Only
  // two operand stages of the two-accumulator tile would fit next to the 3-tap boxes, so two accumulators mean per-tap loads.
  bool reuse = false;
  {
    const bool can = ver == 2 && d.conv == 1 && Wd % 16 == 0 && Hd % 8 == 0;
    if (d.tr == 2) SDW_REQUIRE(can, "tap reuse needs a 3x3 stride-1 conv on the CTA-pair kernel with W % 16 == 0, H % 8 == 0");
    if (d.tr == 2) SDW_REQUIRE(d.nsub != 2, "two accumulators per activation tile need the per-tap mainloop, not tap reuse");
    reuse = can && d.tr != 1 && d.nsub != 2;
    if (reuse) {
      p.bw = bw = 16;
      p.bh = bh = 8;
      p.bb = bb = 1;
      p.tiles_w = Wd / 16;
      p.tiles_h = Hd / 8;
    }
  }
  p.tap_reuse = reuse ? 1 : 0;
  L->tr = p.tap_reuse;
  const int m_tiles_f = p.tiles_w * p.tiles_h * ((d.B + bb - 1) / bb);
  // BLOCK_N choice
  int bn = d.bn;
  int nsub = 1;
  if (ver == 2 && (bn == 0 || d.nsub == 2)) {
    // The 2-CTA kernel is L2->SM bandwidth bound (profiles/r01_mma_eff_vs_blockN.txt): a tile costs about
    // (16 KB of A + 64 B x columns of W) per K block, so the choice minimises waves x bytes over
    // BLOCK_N in {256, 192, 160, 128} and, for long-K problems, the two-accumulator 2 x 160 tile (single-buffered TMEM).
    struct Cand { int bn, nsub; };
    const Cand cand[5] = {{160, 2}, {256, 1}, {192, 1}, {160, 1}, {128, 1}};
    const int mp = (m_tiles_f + 1) / 2;
    const int kblocks = p.ntaps * kchunks;
    // activation bytes per CTA per K block: a 128 x 64 tile, or a third of the 10-row box; the MMA floor is 2 clk per
    // column at ~41 B/clk/SM of operand ingest -> 82 "bytes" per column
    const double a_bytes = reuse ? 20480.0 / 3.0 : 16384.0;
    double best_cost = 1e30;
    int best_bn = 128;
    for (const Cand& c : cand) {
      if (d.bn && d.bn != c.bn) continue;
      if (d.nsub && d.nsub != c.nsub) continue;
      if (d.mode == GEMM_GEGLU && c.bn % 64 != 0) continue;
      if (c.nsub == 2 && (kblocks < 18 || d.mode != GEMM_PLAIN || reuse) && d.nsub != 2) continue;
      const int width = c.bn * c.nsub;
      const int tiles = mp * ((d.N + width - 1) / width);
      const int waves = (tiles + 73) / 74;
      double cost = static_cast<double>(waves) * std::max(a_bytes + 64.0 * width, 82.0 * width);
      // measured (profiles/r01_gemm_shapes_tap_reuse.txt): with 3-tap stages only 3 stages of BLOCK_N = 256 fit and the
      // variant gains nothing over per-tap loads
      if (reuse && c.bn == 256) cost = static_cast<double>(waves) * 31000.0;
      if (c.nsub == 2) cost *= 1.0 + 24.0 / kblocks;  // un-overlapped epilogue ~ 24 K-block times (fit: profiles/r01_gemm_shapes_nsub2.txt)
      if (cost < best_cost) {
        best_cost = cost;
        best_bn = c.bn;
        nsub = c.nsub;
      }
    }
    bn = best_bn;
  }
  if (bn == 0) {
    if (d.mode == GEMM_GEGLU) bn = 128;
    else if (d.N % 160 == 0 && d.N % 128 != 0) bn = 160;
    else if (d.N <= 32) bn = 32;
    else if (d.N <= 64) bn = 64;
    else bn = 128;
  }
  SDW_REQUIRE(bn == 32 || bn == 64 || bn == 128 || bn == 160 || ((bn == 192 || bn == 256) && ver == 2),
              "unsupported BLOCK_N (192 and 256 need the CTA-pair kernel)");
  if (ver == 2) SDW_REQUIRE(bn >= 128, "the 2-CTA kernel needs BLOCK_N >= 128");
  L->ver = ver;
  L->nsub = nsub;
  if (d.mode == GEMM_GEGLU) SDW_REQUIRE(bn % 64 == 0 && d.N % 64 == 0, "GEGLU needs 64-column pairs");
  if (d.mode == GEMM_QKV_VT) SDW_REQUIRE(d.vt && d.vt_col0 % 32 == 0 && d.vt_d > 0, "bad V^T split");
  L->bn = bn;
  L->grid = dim3(m_tiles_f, (d.N + bn - 1) / bn, 1);
  {
    // store staging pays off when the epilogue, not the mainloop, bounds the tile (short K, wide N)
    const int kblocks = p.ntaps * kchunks;
    p.stage_stores = kblocks <= 10 && d.N >= 640 ? 1 : 0;
    // the coalescing stage keeps 32-bit row offsets
    const int64_t max_off = static_cast<int64_t>(d.B) * OH * OW * std::max<int64_t>(d.ldc, d.ldr ? d.ldr : d.ldc);
    SDW_REQUIRE(max_off < (int64_t(1) << 31) || ver == 1, "output too large for the 2-CTA epilogue (>= 2^31 elements)");
  }
  L->ew = 2;
  if (ver == 2) {
    p.m_pairs = (m_tiles_f + 1) / 2;
    p.n_tiles = (d.N + bn * nsub - 1) / (bn * nsub);
    L->grid = dim3(2 * std::min(p.m_pairs * p.n_tiles, 74), 1, 1);  // one CTA pair per SM pair
    // division-free tile coordinates (sdw_gemm2.cu: tile_coords)
    {
      const int n_groups = p.n_tiles;
      const int64_t max_t = static_cast<int64_t>(p.m_pairs) * n_groups, max_m = 2 * static_cast<int64_t>(p.m_pairs) + 1;
      auto magic = [](int64_t dv) { return dv <= 1 ? 0u : static_cast<uint32_t>(((int64_t(1) << 32) + dv - 1) / dv); };
      const int64_t twh = static_cast<int64_t>(p.tiles_w) * p.tiles_h;
      SDW_REQUIRE(max_t * n_groups < (int64_t(1) << 32) && max_m * twh < (int64_t(1) << 32), "tile grid too large for the 32-bit fast division");
      p.mg_ng = magic(n_groups);
      p.mg_tw = magic(p.tiles_w);
      p.mg_twh = magic(twh);
    }
  }
  {
    auto lg2 = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
    p.lg_bw = lg2(p.bw);
    p.lg_bh = lg2(p.bh);
    SDW_REQUIRE((1 << p.lg_bw) == p.bw && (1 << p.lg_bh) == p.bh, "tile extents must be powers of two");
  }
  // tensor maps: A
  for (int m = 0; m < nmaps; ++m) {
    const __half* base = d.A;
    uint64_t dims[4] = {static_cast<uint64_t>(d.C), static_cast<uint64_t>(d.W), static_cast<uint64_t>(d.H),
                        static_cast<uint64_t>(d.B)};
    uint64_t strides[4] = {1, static_cast<uint64_t>(d.sW), static_cast<uint64_t>(d.sH), static_cast<uint64_t>(d.sB)};
    if (d.conv == 2) {
      const int py = m / 2, px = m % 2;
      base = d.A + py * d.sH + px * d.sW;
      dims[1] = Wd;
      dims[2] = Hd;
      strides[1] = 2 * d.sW;
      strides[2] = 2 * d.sH;
    }
    // degenerate extents still need a non-zero, 16B-multiple stride
    for (int i = 1; i < 4; ++i)
      if (strides[i] == 0) strides[i] = static_cast<uint64_t>(Cp);
    uint32_t box[4] = {BK, static_cast<uint32_t>(bw), static_cast<uint32_t>(reuse ? bh + 2 : bh), static_cast<uint32_t>(bb)};
    if (int e = encode_map(&p.mapA[m], base, 4, dims, strides, box)) return e;
  }
  {
    const int64_t ldb = d.ldb ? d.ldb : static_cast<int64_t>(p.ntaps) * Cp;
    uint64_t dims[4] = {static_cast<uint64_t>(d.Kb ? d.Kb : static_cast<int64_t>(p.ntaps) * Cp),
                        static_cast<uint64_t>(d.N), static_cast<uint64_t>(d.b_batched ? Hd : 1),
                        static_cast<uint64_t>(d.b_batched ? d.B : 1)};
    uint64_t strides[4] = {1, static_cast<uint64_t>(ldb), static_cast<uint64_t>(d.b_batched ? d.sBh : 0),
                           static_cast<uint64_t>(d.b_batched ? d.sBb : 0)};
    for (int i = 2; i < 4; ++i)
      if (strides[i] == 0) strides[i] = static_cast<uint64_t>(ldb);
    uint32_t box[4] = {BK, static_cast<uint32_t>(ver == 2 ? bn / 2 : bn), 1, 1};
    if (int e = encode_map(&p.mapB, d.Wt, 4, dims, strides, box)) return e;
  }
  // ---- epilogue flavour and pipeline depth of the 2-CTA kernel ----------------------------------------------------
  p.epi_tma = 0;
  p.nstages = 0;
  if (ver == 2) {
    const int64_t osW = d.o_sW || d.o_sH || d.o_sB ? d.o_sW : d.ldc;
    const int64_t osH = d.o_sW || d.o_sH || d.o_sB ? d.o_sH : OW * d.ldc;
    const int64_t osB = d.o_sW || d.o_sH || d.o_sB ? d.o_sB : OH * OW * d.ldc;
    const int64_t ldr = d.ldr ? d.ldr : d.ldc;
    const int64_t rsW = d.r_sW || d.r_sH || d.r_sB ? d.r_sW : ldr;
    const int64_t rsH = d.r_sW || d.r_sH || d.r_sB ? d.r_sH : OW * ldr;
    const int64_t rsB = d.r_sW || d.r_sH || d.r_sB ? d.r_sB : OH * OW * ldr;
    auto ok16 = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0; };
    auto ok_strides = [&](int64_t sw, int64_t sh, int64_t sb) {
      return sw > 0 && sw % 8 == 0 && (Hd == 1 || sh % 8 == 0) && (d.B == 1 || sb % 8 == 0);
    };
    const int ncols = d.mode == GEMM_GEGLU ? d.N / 2 : (d.mode == GEMM_QKV_VT ? d.vt_col0 : d.N);
    // V^T scatter through TMA: token lattice (H == 1, 128-token tiles), 32-column chunks never straddle vt_col0
    const bool vt_ok = d.mode != GEMM_QKV_VT ||
                       (Hd == 1 && bw == BM && d.conv == 0 && d.vt_col0 % 32 == 0 && d.vt_ld % 8 == 0 && ok16(d.vt) &&
                        d.vt_ntok == Wd && !d.resid);
    bool can = nsub == 1 && !d.b_batched && vt_ok && !d.resid2 && (!d.rowvec || d.rowvec_ld == 0) &&
               d.N % 8 == 0 && bn <= 256 && ok16(d.out) && ok_strides(osW, osH, osB) && (!d.bias || ok16(d.bias)) &&
               (!d.resid || (ok16(d.resid) && ok_strides(rsW, rsH, rsB) && d.mode == GEMM_PLAIN));
    if (d.et == 2) SDW_REQUIRE(can, "the TMA epilogue needs the CTA-pair kernel, plain/GEGLU mode, no row vector and 16-byte aligned views");
    const int kblocks = p.ntaps * kchunks;
    // short-K GEMMs are bound by their epilogue (profiles/r01_ncu_epilogue_shortk.md) and gain up to 2x; long-K ones
    // lose one operand stage to the epilogue buffers but still come out ahead end to end (bench: 8.49 -> 8.56 frames/s),
    // so the TMA epilogue is used wherever it is eligible
    p.epi_tma = can && (d.et == 0 || d.et == 2) ? 1 : 0;
    const int a_stage = reuse ? 20480 : 16384;
    const int b_stage = (reuse ? 3 : 1) * nsub * (bn / 2) * 128;
    const int epi_bytes = p.epi_tma ? G2_EPI_OUT + G2_EPI_BIAS + (d.resid ? G2_RES_STAGES * G2_RES_STAGE : 0) : G2_EPI_OLD;
    p.nstages = std::min(8, (G2_SMEM_USABLE - G2_BAR_BYTES - epi_bytes) / (a_stage + b_stage));
    SDW_REQUIRE(p.nstages >= 2, "no room for a two-stage operand pipeline");
    // epilogue width: four warps per TMEM lane quarter where the epilogue, not the MMA, sets the tile time — K <= 448
    // (the 64x64-level transformer linears, K = 320: GEGLU 434 -> 383 us, QKV-like 218 -> 161 us, out-projection 99 ->
    // 88 us at batch 60, same box; from K = 640 on the MMA is the longer leg and the wider epilogue loses 2-10 %:
    // profiles/r02_epilogue_width_ab_same_box.txt)
    {
      const bool can4 = p.epi_tma && nsub == 1 && !reuse;
      if (d.ew == 4) SDW_REQUIRE(can4, "the 16-warp epilogue needs the TMA epilogue, one accumulator and the per-tap mainloop");
      const int want4 = d.ew ? d.ew == 4 : kblocks <= 7;
      L->ew = can4 && want4 ? 4 : 2;
      if (L->ew == 4) {  // 16 per-warp bias copies instead of 8, eight residual ring slots instead of four
        const int extra = G2_EPI_BIAS + (d.resid ? G2_RES_STAGES * G2_RES_STAGE : 0);
        p.nstages = std::min(8, (G2_SMEM_USABLE - G2_BAR_BYTES - epi_bytes - extra) / (a_stage + b_stage));
        SDW_REQUIRE(p.nstages >= 2, "no room for a two-stage operand pipeline");
      }
    }
    if (p.epi_tma) {
      // output lattice: column, then the tile lattice (w, h, b) with the parity scatter folded into base + strides
      const int sw_ = std::min(bw, 32), sh_ = std::min(bh, 32 / sw_), sb_ = 32 / (sw_ * sh_);
      uint64_t dims[4] = {static_cast<uint64_t>(ncols), static_cast<uint64_t>(Wd), static_cast<uint64_t>(Hd),
                          static_cast<uint64_t>(d.B)};
      auto fix = [&](uint64_t* st) {  // extents of one still need a legal stride
        for (int i = 2; i < 4; ++i)
          if (st[i] == 0 || st[i] % 8 != 0) st[i] = st[1] * static_cast<uint64_t>(Wd);
      };
      uint64_t so[4] = {1, static_cast<uint64_t>(osW * p.os), static_cast<uint64_t>(osH * p.os), static_cast<uint64_t>(osB)};
      fix(so);
      uint32_t box_o[4] = {32, static_cast<uint32_t>(sw_), static_cast<uint32_t>(sh_), static_cast<uint32_t>(sb_)};
      if (int e = encode_map(&p.mapOut, d.out + p.oy * osH + p.ox * osW, 4, dims, so, box_o, 64)) return e;
      if (d.mode == GEMM_QKV_VT) {
        const int vrows = d.N - d.vt_col0;  // heads * d rows of V^T per sample
        uint64_t dv[3] = {static_cast<uint64_t>(Wd), static_cast<uint64_t>(vrows), static_cast<uint64_t>(d.B)};
        uint64_t sv[3] = {1, static_cast<uint64_t>(d.vt_ld), static_cast<uint64_t>(d.vt_ld) * static_cast<uint64_t>(d.vt_heads) * d.vt_d};
        uint32_t bv[3] = {32, 32, 1};
        SDW_REQUIRE(vrows == d.vt_heads * d.vt_d, "V^T rows must be heads x d");
        if (int e = encode_map(&p.mapVt, d.vt, 3, dv, sv, bv, 0)) return e;
      }
      if (d.resid) {
        uint64_t sr[4] = {1, static_cast<uint64_t>(rsW * p.os), static_cast<uint64_t>(rsH * p.os), static_cast<uint64_t>(rsB)};
        fix(sr);
        uint32_t box_r[4] = {32, static_cast<uint32_t>(bw), static_cast<uint32_t>(bh), static_cast<uint32_t>(bb)};
        if (int e = encode_map(&p.mapRes, d.resid + p.oy * rsH + p.ox * rsW, 4, dims, sr, box_r, 64)) return e;
      }
    }
  }
  p.bias = d.bias;
  p.rowvec = d.rowvec;
  p.rowvec_ld = d.rowvec_ld;
  p.resid = d.resid;
  p.resid2 = d.resid2;
  p.res2_scale = d.res2_scale;
  p.out = d.out;
  if (d.o_sW || d.o_sH || d.o_sB) {
    p.o_sW = d.o_sW; p.o_sH = d.o_sH; p.o_sB = d.o_sB;
  } else {
    p.o_sW = d.ldc; p.o_sH = OW * d.ldc; p.o_sB = OH * OW * d.ldc;
  }
  if (d.r_sW || d.r_sH || d.r_sB) {
    p.r_sW = d.r_sW; p.r_sH = d.r_sH; p.r_sB = d.r_sB;
  } else {
    const int64_t ldr = d.ldr ? d.ldr : d.ldc;
    p.r_sW = ldr; p.r_sH = OW * ldr; p.r_sB = OH * OW * ldr;
  }
  p.mode = d.mode;
  p.act = d.act;
  p.alpha = d.alpha;
  p.vt_col0 = d.vt_col0;
  p.vt_d = d.vt_d;
  p.vt_heads = d.vt_heads;
  p.vt_ntok = d.vt_ntok > 0 ? d.vt_ntok : 1;
  p.vt = d.vt;
  p.vt_ld = d.vt_ld;
  return 0;
}

int launch_gemm(const GemmLaunch& l, cudaStream_t stream) {
  if (l.ver == 2) return launch_gemm2(l, stream);
  switch (l.bn) {
    case 32:
      gemm_tc_kernel<32><<<l.grid, GEMM_THREADS, GemmCfg<32>::SMEM_BYTES, stream>>>(l.p);
      break;
    case 64:
      gemm_tc_kernel<64><<<l.grid, GEMM_THREADS, GemmCfg<64>::SMEM_BYTES, stream>>>(l.p);
      break;
    case 128:
      gemm_tc_kernel<128><<<l.grid, GEMM_THREADS, GemmCfg<128>::SMEM_BYTES, stream>>>(l.p);
      break;
    case 160:
      gemm_tc_kernel<160><<<l.grid, GEMM_THREADS, GemmCfg<160>::SMEM_BYTES, stream>>>(l.p);
      break;
    default:
      set_error("bad BLOCK_N");
      return 1;
  }
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace sdw
