// sdw_internal.h — host-side internal API shared by the kernels' launchers, the
// engine (sdw_engine.cu) and the C-ABI (sdw_capi.cu).  Not part of the public ABI.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

namespace sdw {

// ---------------------------------------------------------------------------
// error plumbing: every launcher returns 0 on success; message in thread-local
// ---------------------------------------------------------------------------
void set_error(const std::string& msg);
const char* last_error();
#define SDW_CUDA_OK(expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      (void)cudaGetLastError(); /* do not leave the error latched for the caller's next CUDA call */ \
      ::sdw::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
      return 2;                                                                                \
    }                                                                                          \
  } while (0)
#define SDW_REQUIRE(cond, msg)                                                                 \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      ::sdw::set_error(std::string("invalid argument: ") + (msg) + " [" #cond "]");            \
      return 1;                                                                                \
    }                                                                                          \
  } while (0)

// ---------------------------------------------------------------------------
// kernel launch with the programmatic-dependent-launch attribute (SDW_PDL=0 disables it)
// ---------------------------------------------------------------------------
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------
// tcgen05 implicit-GEMM (conv3x3 / conv1x1 / linear / batched matmul)
// ---------------------------------------------------------------------------
// out[pix, n] = epi( sum_{tap, c} A[lattice(tap)][pix shifted by (dx,dy)][c] * Wt[n][tap*Cp + c] )
// A is an NHWC fp16 lattice (C, W, H, B) read through up to four TMA maps (one
// per input sub-lattice; >1 only for stride-2 convs), Wt is K-major [N][ntaps*Cp].
enum GemmMode : int {
  GEMM_PLAIN = 0,   // out[pix*ldc + n]
  GEMM_GEGLU = 1,   // packed (value|gate) 32-column pairs -> out[pix*ldc + n/2]
  GEMM_QKV_VT = 2,  // cols < vt_col0 plain; cols >= vt_col0 written transposed per head (V^T)
};

struct alignas(64) GemmKParams {
  CUtensorMap mapA[4];
  CUtensorMap mapB;
  int8_t tap_map[12], tap_dx[12], tap_dy[12];
  int ntaps, kchunks;       // K blocks = ntaps * kchunks, each 64 wide
  int W, H, B;              // tile-grid domain (the A lattice extents)
  int bw, bh, bb;           // M tile = bw*bh*bb = 128 lattice points
  int tiles_w, tiles_h;     // tiles per (w,h); tiles along b = gridDim.x / (tiles_w*tiles_h)
  // 2-CTA kernel: tile coordinates without integer divisions (7 per tile per warp used to be a quarter of the epilogue's
  // instruction stream on short-K GEMMs: profiles/r02_ncu_epilogue_shortk.md).  bw, bh, bb are powers of two (shifts);
  // n_groups, tiles_w, tiles_w * tiles_h go through q = umulhi(n, ceil(2^32 / d)), exact for n * d < 2^32 (planner-checked)
  int lg_bw, lg_bh;
  uint32_t mg_ng, mg_tw, mg_twh;  // 0 = divisor 1
  int N;                    // GEMM N (packed columns)
  int b_batched;            // 1: weight map coords (.., y0, b0) = lattice (h, b) (batched matmul)
  int stage_stores;         // 1: bounce output chunks through shared memory for coalesced stores (wide-N GEMMs)
  int m_pairs, n_tiles;     // 2-CTA persistent kernel: tile grid (pairs of 128-row M tiles x BN-wide N tiles)
  int tap_reuse;            // 1: 3x3 conv with one (bh+2)-row activation box per (channel chunk, kx) shared by the 3 ky taps
  // TMA epilogue (2-CTA kernel, short-K GEMMs): output chunks leave through TMA stores, the residual tile arrives
  // through a TMA-fed shared-memory ring, the bias is staged per warp (sdw_gemm_epi.cuh: gemm_epilogue_tma)
  CUtensorMap mapOut;       // (columns, w, h, b) lattice of the output, box (32, slab_w, slab_h, slab_b), 64B swizzle
  CUtensorMap mapRes;       // ... of the residual, box (32, bw, bh, bb)
  CUtensorMap mapVt;        // GEMM_QKV_VT: V^T as (token, head * d + dd, sample), box (32 tokens, 32 rows), no swizzle
  int epi_tma;
  int nstages;              // mainloop pipeline depth (what the epilogue buffers leave of the 227 KB)
  // epilogue
  const float* bias;        // [N] or null
  const float* rowvec;      // [B][rowvec_ld] per-sample vector added per column (time-embedding proj) or null
  int rowvec_ld;
  const __half* resid;      // residual or null; element offset = b*r_sB + oy'*r_sH + ox'*r_sW + n
  int64_t r_sW, r_sH, r_sB;
  __half* out;              // element offset = b*o_sB + (y*os+oy)*o_sH + (x*os+ox)*o_sW + n
  int64_t o_sW, o_sH, o_sB;
  int os, ox, oy;
  int mode;
  int act;                  // 0 none, 1 SiLU, 2 LeakyReLU(0.2)
  float alpha;              // scale on the accumulator (before bias)
  // GEMM_QKV_VT
  int vt_col0, vt_d, vt_heads, vt_ntok;
  __half* vt;               // [b][head][d][vt_ld]
  int64_t vt_ld;
  // second residual (generic epilogue only): out = res2_scale * (epilogue result incl. resid) + resid2, same strides as resid
  const __half* resid2;
  float res2_scale;
};

struct GemmLaunch {
  GemmKParams p;
  dim3 grid;
  int bn;   // BLOCK_N variant
  int ver;  // 1: one 128xBN tile per CTA (sdw_gemm.cu); 2: persistent CTA pairs, 256xBN tiles (sdw_gemm2.cu)
  int nsub = 1;  // ver 2: accumulators per activation tile (2 -> 256 x 2*BN tiles, single-buffered TMEM)
  int ew = 2;    // ver 2: epilogue warps per TMEM lane quarter (4 -> the 640-thread kernel for epilogue-bound short-K GEMMs)
  int tr = 0;    // ver 2: 1 -> tap-reuse mainloop (3x3 stride-1 convs; GemmKParams::tap_reuse)
};

// Describes one implicit GEMM in host terms; plan_gemm() turns it into a launch.
struct GemmDesc {
  const __half* A = nullptr;       // lattice base
  int C = 0, W = 0, H = 1, B = 1;  // input lattice extents (elements)
  int64_t sW = 0, sH = 0, sB = 0;  // element strides of the input lattice (channel stride is 1)
  int conv = 0;                    // 0: 1x1 / linear; 1: 3x3 stride 1 pad 1; 2: 3x3 stride 2 pad 1; 3: nearest-up2 + 3x3 as a
                                   //    2x2 conv per output parity (up_px/up_py) on pack_weight_up4 weights
  int up_px = 0, up_py = 0;
  const __half* Wt = nullptr;      // [N][ntaps*Cp] (Cp = C rounded up to 64) K-major
  int N = 0;
  int64_t ldb = 0;                 // weight row pitch in elements (0 -> ntaps*Cp)
  int64_t Kb = 0;                  // valid K extent of the weight rows (0 -> ntaps*Cp); beyond it reads as zero
  int b_batched = 0;               // weights indexed by lattice (h, b): batched matmul
  int64_t sBh = 0, sBb = 0;        // weight strides (elements) along lattice h and b when b_batched
  const float* bias = nullptr;
  const float* rowvec = nullptr;
  int rowvec_ld = 0;
  const __half* resid = nullptr;
  int64_t ldr = 0;                 // residual pixel pitch (0 -> ldc); or explicit strides below
  int64_t r_sW = 0, r_sH = 0, r_sB = 0;
  __half* out = nullptr;
  int64_t ldc = 0;                 // output pixel pitch; NHWC-contiguous output unless o_s* are given
  int64_t o_sW = 0, o_sH = 0, o_sB = 0;
  int mode = GEMM_PLAIN;
  int act = 0;                     // 0 none, 1 SiLU, 2 LeakyReLU(0.2)
  float alpha = 1.f;
  const __half* resid2 = nullptr;  // second residual on the residual's strides: out = res2_scale * out + resid2
  float res2_scale = 1.f;
  int vt_col0 = 0, vt_d = 0, vt_heads = 0, vt_ntok = 0;
  __half* vt = nullptr;
  int64_t vt_ld = 0;
  int bn = 0;   // 0 = auto
  int ver = 0;  // 0 = auto, 1 / 2 force a kernel version
  int nsub = 0; // 0 = auto, 1 / 2: accumulators per activation tile in the 2-CTA kernel
  int ew = 0;   // 0 = auto, 2 / 4: epilogue warps per TMEM lane quarter in the 2-CTA kernel (4 needs the TMA epilogue)
  int tr = 0;   // 0 = auto, 1 = never, 2 = require the tap-reuse mainloop (3x3 stride-1 conv, W % 16 == 0, H % 8 == 0)
  int et = 0;   // 0 = auto, 1 = never, 2 = require the TMA epilogue
};

int plan_gemm(const GemmDesc& d, GemmLaunch* out);
int launch_gemm(const GemmLaunch& l, cudaStream_t stream);
int launch_gemm2(const GemmLaunch& l, cudaStream_t stream);
int gemm2_init();
void set_plan_only(bool on);
int gemm_init();  // resolves the driver entry point, sets smem attributes
// shared-memory budget of the 2-CTA kernel (sdw_gemm2.cu): barriers, then the operand ring, then the epilogue buffers
constexpr int G2_SMEM_DYN = 227 * 1024;                    // requested dynamic shared memory
constexpr int G2_SMEM_USABLE = G2_SMEM_DYN - 1024;         // after the 1 KB alignment slack
constexpr int G2_BAR_BYTES = 1024;
constexpr int G2_EPI_OLD = 8 * 2048;                       // 2 KB store-coalescing buffer per epilogue warp
constexpr int G2_EPI_OUT = 8 * 2 * 2048;                   // TMA epilogue: 32-row x 64-byte output slabs, two per warp (8 warps) or one (16)
constexpr int G2_EPI_BIAS = 8 * 1024;                      //   per-warp bias copy (<= 256 fp32 columns); twice that for 16 warps
constexpr int G2_RES_STAGES = 4, G2_RES_STAGE = 128 * 64;  //   residual ring: [128 rows x 32 columns] fp16 chunks, 4 slots (8 with 16 epilogue warps)
int encode_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
               const uint32_t* box, int swizzle_bytes = 128);

// ---------------------------------------------------------------------------
// fused attention (sdw_attn.cu)
// ---------------------------------------------------------------------------
struct AttnDesc {
  const __half* q = nullptr;   // [B][Nq][q_ld], head h at columns h*d
  int64_t q_ld = 0;
  const __half* k = nullptr;   // [B][Nk][k_ld], head h at columns h*d
  int64_t k_ld = 0;
  const __half* vt = nullptr;  // [B][heads][d][vt_ld]  (V transposed, written by the QKV GEMM epilogue)
  int64_t vt_ld = 0;
  int B = 0, Nq = 0, Nk = 0, heads = 0, d = 0;
  __half* out = nullptr;       // [B][Nq][out_ld], head h at columns h*d
  int64_t out_ld = 0;
};
struct AttnLaunch {
  alignas(64) unsigned char storage[704];
};
bool attn_supported(int d);
int plan_attention(const AttnDesc& a, AttnLaunch* L);
int launch_attention(const AttnLaunch& L, cudaStream_t stream);
void attention_plan_info(const AttnLaunch& L, int out[5]);
void attention_set_trace(long long* buf);  // device buffer [2][4096][8] of clock64 stamps written by CTA 0 of attn_pp_kernel (nullptr = off)

// ---------------------------------------------------------------------------
// fp32 helper kernels (sdw_elem.cu)
// ---------------------------------------------------------------------------
int slerp_lerp_batch(const void* lat_a, const void* lat_b, const void* emb_a, const void* emb_b, const float* t,
                     int n_frames, int64_t n_lat, int64_t n_emb, int is_f16, float thr, void* out_lat, void* out_emb,
                     cudaStream_t stream);
int cfg_sched_step(const float* eps, int has_uncond, float* x, float* x_base, float* hist, const void* coef, int F,
                   int C, int H, int W, void* next_in, int cpad, cudaStream_t stream);
int latents_init(const void* latents, int is_f16, float sigma, float in_scale, float* x, void* model_in, int cpad,
                 int dup, int F, int C, int H, int W, cudaStream_t stream);
int pack_weight(const void* w, int N, int C, int kh, int kw, int geglu, void* out, cudaStream_t stream);
// tiled = True (circular convolution padding): wrap-padded copy of an NHWC image / interior of a padded result
int wrap_pad(const void* x, int64_t ld_bytes, int B, int H, int W, int pix_bytes, int pad, void* y, cudaStream_t stream);
int crop_interior(const void* yp, int B, int H, int W, int pix_bytes, int crop, const void* resid_f16, int64_t ldr, void* out,
                  int64_t ldo_bytes, cudaStream_t stream);
// upsampler weights: 4 parity blocks of [N][4][Cp] (taps pre-summed); block p = py*2+px at out + p*N*4*Cp
int pack_weight_up4(const void* w, int N, int C, void* out, cudaStream_t stream);

// ---------------------------------------------------------------------------
// norm / softmax / small-channel layers (sdw_norm.cu)
// ---------------------------------------------------------------------------
int gn_chunks(int64_t P, int B);
size_t gn_workspace_bytes(int B);
int groupnorm_launches();  // kernels per GroupNorm (partial statistics, finalize, apply)
int groupnorm(const __half* x, int64_t ldx, int B, int64_t P, int C, int G, const float* gamma, const float* beta,
              float eps, int silu, __half* y, int64_t ldy, float2* partial_ws, cudaStream_t stream);
int layernorm(const __half* x, int64_t ldx, int64_t rows, int C, const float* gamma, const float* beta, float eps,
              __half* y, int64_t ldy, cudaStream_t stream);
int softmax_rows(__half* s, int64_t ld, int64_t rows, int n, cudaStream_t stream);
int conv_in_small(const __half* x, int64_t ldx, int B, int H, int W, int Cin, const __half* w, const float* bias,
                  int N, __half* y, int64_t ldy, cudaStream_t stream);
// 3x3 conv of a uint8 RGB NHWC image read as x / 255 (Real-ESRGAN conv_first), OIHW fp16 weights [N][3][3][3]
int conv_in_u8(const uint8_t* x, int B, int H, int W, const __half* w, const float* bias, int N, __half* y,
               int64_t ldy, cudaStream_t stream);
// unit01 = 0: uint8 = round(clamp(v/2+0.5, 0, 1)*255) (VAE); 1: round(clamp(v, 0, 1)*255) (Real-ESRGAN)
int conv_out_small(const __half* x, int64_t ldx, int B, int H, int W, int C, const __half* w, const float* bias,
                   int nout, float* out_f32, uint8_t* out_u8, cudaStream_t stream, int unit01 = 0);
int vae_in(const float* x, float inv_scale, const __half* w, const float* bias, int F, int C, int H, int W, __half* z,
           cudaStream_t stream);
int linear_f32(const float* in, int64_t ldi, const __half* w, const float* bias, int M, int N, int K, int silu_in,
               int silu_out, float* out, int64_t ldo, cudaStream_t stream);
int timestep_embed(const float* t, int n, int dim, int round_f16, float* out, cudaStream_t stream);
int half_to_float(const __half* in, float* out, int64_t n, int geglu_N, cudaStream_t stream);

}  // namespace sdw
