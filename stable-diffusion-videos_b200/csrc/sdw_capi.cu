// sdw_capi.cu — the extern "C" surface of libsdwalk.so (declared in include/sdwalk.h).
#include "../../include/sdwalk.h"
#include "sdw_internal.h"

#include <cstring>

namespace sdw {
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }
}  // namespace sdw

using namespace sdw;

extern "C" {

const char* sdw_last_error(void) { return sdw::last_error(); }
int sdw_abi_version(void) { return SDW_ABI_VERSION; }
void sdw_debug_plan_only(int on) { sdw::set_plan_only(on != 0); }

int sdw_slerp_lerp_batch(const void* lat_a, const void* lat_b, const void* emb_a, const void* emb_b, const float* t,
                         int n_frames, int64_t n_lat, int64_t n_emb, int dtype_is_f16, float dot_threshold,
                         void* out_lat, void* out_emb, void* stream) {
  return slerp_lerp_batch(lat_a, lat_b, emb_a, emb_b, t, n_frames, n_lat, n_emb, dtype_is_f16, dot_threshold,
                          out_lat, out_emb, static_cast<cudaStream_t>(stream));
}

int sdw_cfg_sched_step(const void* eps_nhwc, int has_uncond, float* x, float* x_base, float* hist,
                       const sdw_step_coef* coef, int F, int C, int H, int W, void* next_in, int next_in_cpad,
                       void* stream) {
  return cfg_sched_step(static_cast<const float*>(eps_nhwc), has_uncond, x, x_base, hist, coef, F, C, H, W, next_in,
                        next_in_cpad, static_cast<cudaStream_t>(stream));
}

int sdw_latents_init(const void* latents, int dtype_is_f16, float init_noise_sigma, float in_scale, float* x,
                     void* model_in, int model_in_cpad, int dup, int F, int C, int H, int W, void* stream) {
  return latents_init(latents, dtype_is_f16, init_noise_sigma, in_scale, x, model_in, model_in_cpad, dup, F, C, H, W,
                      static_cast<cudaStream_t>(stream));
}

static int to_desc(const sdw_gemm_desc* c, GemmDesc& d);

// planner introspection (host only; works in plan-only mode without a GPU): what plan_gemm chose for this descriptor
int sdw_debug_plan(const sdw_gemm_desc* c, int32_t out[12]) {
  SDW_REQUIRE(c != nullptr && out != nullptr, "null");
  GemmDesc d;
  if (int e = to_desc(c, d)) return e;
  GemmLaunch L;
  if (int e = plan_gemm(d, &L)) return e;
  out[0] = L.ver; out[1] = L.bn; out[2] = L.nsub; out[3] = L.ew; out[4] = L.tr;
  out[5] = L.p.epi_tma; out[6] = L.p.nstages; out[7] = 0;
  out[8] = static_cast<int32_t>(L.grid.x); out[9] = L.p.bw; out[10] = L.p.bh; out[11] = L.p.bb;
  return 0;
}

int sdw_gemm(const sdw_gemm_desc* c, void* stream) {
  SDW_REQUIRE(c != nullptr, "null desc");
  GemmDesc d;
  if (int e = to_desc(c, d)) return e;
  GemmLaunch L;
  if (int e = plan_gemm(d, &L)) return e;
  return launch_gemm(L, static_cast<cudaStream_t>(stream));
}

int sdw_gemm_res2(const sdw_gemm_desc* c, const void* resid2, float res2_scale, void* stream) {
  SDW_REQUIRE(c != nullptr && resid2 != nullptr, "null");
  GemmDesc d;
  if (int e = to_desc(c, d)) return e;
  d.resid2 = static_cast<const __half*>(resid2);
  d.res2_scale = res2_scale;
  GemmLaunch L;
  if (int e = plan_gemm(d, &L)) return e;
  return launch_gemm(L, static_cast<cudaStream_t>(stream));
}

static int to_desc(const sdw_gemm_desc* c, GemmDesc& d) {
  d.A = static_cast<const __half*>(c->A);
  d.C = c->C; d.W = c->W; d.H = c->H; d.B = c->B;
  d.sW = c->sW; d.sH = c->sH; d.sB = c->sB;
  d.conv = c->conv; d.up_px = c->up_px; d.up_py = c->up_py;
  d.Wt = static_cast<const __half*>(c->Wt);
  d.N = c->N; d.ldb = c->ldb; d.Kb = c->Kb;
  d.b_batched = c->b_batched; d.sBh = c->sBh; d.sBb = c->sBb;
  d.bias = c->bias; d.rowvec = c->rowvec; d.rowvec_ld = c->rowvec_ld;
  d.resid = static_cast<const __half*>(c->resid); d.ldr = c->ldr;
  d.out = static_cast<__half*>(c->out); d.ldc = c->ldc;
  d.o_sW = c->o_sW; d.o_sH = c->o_sH; d.o_sB = c->o_sB;
  d.mode = c->mode; d.act = c->act; d.alpha = c->alpha;
  d.vt_col0 = c->vt_col0; d.vt_d = c->vt_d; d.vt_heads = c->vt_heads; d.vt_ntok = c->vt_ntok;
  d.vt = static_cast<__half*>(c->vt); d.vt_ld = c->vt_ld;
  d.bn = c->bn;
  d.ver = c->ver;
  d.nsub = c->nsub;
  d.ew = c->ew;
  d.tr = c->tr;
  d.et = c->et;
  return 0;
}

int sdw_attention(const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* vt, int64_t vt_ld, int B,
                  int Nq, int Nk, int heads, int d, void* out, int64_t out_ld, void* stream) {
  AttnDesc a;
  a.q = static_cast<const __half*>(q); a.q_ld = q_ld;
  a.k = static_cast<const __half*>(k); a.k_ld = k_ld;
  a.vt = static_cast<const __half*>(vt); a.vt_ld = vt_ld;
  a.B = B; a.Nq = Nq; a.Nk = Nk; a.heads = heads; a.d = d;
  a.out = static_cast<__half*>(out); a.out_ld = out_ld;
  AttnLaunch L;
  if (int e = plan_attention(a, &L)) return e;
  return launch_attention(L, static_cast<cudaStream_t>(stream));
}

int sdw_groupnorm(const void* x, int64_t ldx, int B, int64_t P, int C, int G, const float* gamma, const float* beta,
                  float eps, int silu, void* y, int64_t ldy, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float2* ws = nullptr;  // workspace of the three-kernel path (the engine keeps one in its arena)
  SDW_CUDA_OK(cudaMallocAsync(&ws, gn_workspace_bytes(B), st));
  const int rc = groupnorm(static_cast<const __half*>(x), ldx, B, P, C, G, gamma, beta, eps, silu, static_cast<__half*>(y),
                           ldy, ws, st);
  cudaFreeAsync(ws, st);
  return rc;
}

int sdw_layernorm(const void* x, int64_t ldx, int64_t rows, int C, const float* gamma, const float* beta, float eps,
                  void* y, int64_t ldy, void* stream) {
  return layernorm(static_cast<const __half*>(x), ldx, rows, C, gamma, beta, eps, static_cast<__half*>(y), ldy,
                   static_cast<cudaStream_t>(stream));
}

void sdw_debug_attention_trace(void* buf) { sdw::attention_set_trace(static_cast<long long*>(buf)); }

int sdw_debug_attention_plan(int B, int Nq, int Nk, int heads, int d, int32_t out[5]) {
  SDW_REQUIRE(out != nullptr, "null");
  AttnDesc a;
  // fake 16-byte aligned addresses: nothing is dereferenced by the planner (tensor maps are validated in plan-only mode)
  a.q = reinterpret_cast<const __half*>(uintptr_t(1) << 30); a.q_ld = static_cast<int64_t>(heads) * d;
  a.k = reinterpret_cast<const __half*>(uintptr_t(2) << 30); a.k_ld = a.q_ld;
  a.vt = reinterpret_cast<const __half*>(uintptr_t(3) << 30); a.vt_ld = (Nk + 7) / 8 * 8;
  a.B = B; a.Nq = Nq; a.Nk = Nk; a.heads = heads; a.d = d;
  a.out = reinterpret_cast<__half*>(uintptr_t(4) << 30); a.out_ld = a.q_ld;
  AttnLaunch L;
  if (int e = plan_attention(a, &L)) return e;
  int v[5];
  attention_plan_info(L, v);
  for (int i = 0; i < 5; ++i) out[i] = v[i];
  return 0;
}

int sdw_pack_weight_up4(const void* w_oihw, int N, int C, void* out, void* stream) {
  return pack_weight_up4(w_oihw, N, C, out, static_cast<cudaStream_t>(stream));
}

int sdw_pack_weight(const void* w_oihw, int N, int C, int kh, int kw, int geglu_interleave, void* out, void* stream) {
  return pack_weight(w_oihw, N, C, kh, kw, geglu_interleave, out, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
