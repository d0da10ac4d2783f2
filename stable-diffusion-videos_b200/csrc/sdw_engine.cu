// sdw_engine.cu — the native runtime of the latent-walk hot path.
//
// One engine = one (UNet2DCondition, AutoencoderKL decoder) pair at a fixed latent resolution and a fixed
// number of frames per call F.  It owns nothing but offsets: weights, activations and workspaces all live in
// ONE caller-supplied arena (a torch tensor), laid out by a bump allocator at bind time.  The model graph is
// turned once into a static launch plan (tensor maps encoded up-front); a sample call replays
//     prologue (ctx assembly, cross-attention K/V — step-invariant per frame, hoisted)
//     n_steps x { UNet plan ; CFG + scheduler step }           stable_diffusion_pipeline.py:412-430
//     VAE-decoder plan -> uint8 NHWC frames                      stable_diffusion_pipeline.py:432-438, 450
// optionally captured into a CUDA graph.
//
// Layout: activations NHWC fp16 (tokens [B, HW, C] are the same memory), latent state fp32 NCHW,
// weights K-major [N][tap][ceil64(C)] fp16 (packed once at load), biases / norm affines fp32.
#include "../../include/sdwalk.h"
#include "sdw_internal.h"

#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <vector>

namespace sdw {

int unet_ctx_assemble(const __half* cond, const __half* uncond, int F, int dup, int64_t per, __half* out,
                      cudaStream_t stream);

namespace {

struct T {  // NHWC fp16 view
  __half* p = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  int64_t ld = 0;
  int64_t pixels() const { return static_cast<int64_t>(B) * H * W; }
};

enum ParamKind { P_PACKED, P_RAW, P_VEC, P_PACKED_UP4 };
struct ParamSlot {
  ParamKind kind;
  void* dst;
  int N, C, kh, kw;
  int geglu;
  int64_t numel;
  bool loaded = false;
};

using OpFn = std::function<int(cudaStream_t, int /*step*/)>;

struct Engine {
  sdw_engine_config cfg{};
  bool dry = true;
  uint8_t* base = nullptr;
  size_t off = 0;
  size_t arena_bytes = 0;
  std::map<std::string, ParamSlot> params;
  std::vector<OpFn> prologue, unet_ops, vae_ops;
  int n_launch_prologue = 0, n_launch_unet = 0, n_launch_vae = 0;
  int* launch_counter = nullptr;
  // fixed buffers
  int Bn = 0;  // UNet batch = F * (guidance ? 2 : 1)
  __half* model_in = nullptr;   // [Bn][H][W][4]
  float* eps = nullptr;         // [Bn][H][W][4]
  float* x = nullptr;           // [F][4][H][W]
  float* x_base = nullptr;
  float* hist = nullptr;        // [4][F][4][H][W]
  __half* ctx = nullptr;        // [Bn][tokens][D]
  __half* cond_stage = nullptr; // [F][tokens][D]
  __half* uncond_stage = nullptr;
  int uncond_batch = 1;  // 1: one unconditional embedding shared by all frames; frames: one per frame (per-sample negative prompts)
  void* lat_stage = nullptr;    // [F][4][H][W] fp32-sized
  uint8_t* out_u8 = nullptr;    // [F][8H][8W][3]
  float* out_img_f32 = nullptr; // pre-clamp decoder output (debug / parity)
  float2* gn_ws = nullptr;
  __half* S = nullptr;          // attention score scratch
  size_t S_elems = 0;
  // time-embedding tables
  float* t_dev = nullptr;       // [max_steps]
  float* t_sin = nullptr;       // [max_steps][ch0]
  float* t_h1 = nullptr;        // [max_steps][4 ch0]
  float* temb = nullptr;        // [max_steps][4 ch0]
  struct TProj { const __half* w; const float* b; float* table; int cout; };
  std::vector<TProj> tprojs;
  const __half *te_w1 = nullptr, *te_w2 = nullptr;
  const float *te_b1 = nullptr, *te_b2 = nullptr;
  // schedule
  int n_steps = 0;
  std::vector<sdw_step_coef> coefs;
  float init_sigma = 1.f, first_in_scale = 1.f;
  // graph
  cudaGraphExec_t graph_exec = nullptr;
  int graph_steps = -1;
  std::string err;

  // ---- arena ---------------------------------------------------------------
  void* alloc(size_t bytes, size_t align = 1024) {
    off = (off + align - 1) / align * align;
    void* p = dry ? nullptr : base + off;
    off += bytes;
    return p;
  }
  T act(int B, int H, int W, int C) {
    T t;
    t.B = B; t.H = H; t.W = W; t.C = C; t.ld = C;
    t.p = static_cast<__half*>(alloc(static_cast<size_t>(B) * H * W * C * 2));
    return t;
  }
  // ---- activation liveness.  The launch plan is a fixed sequence on one stream, so lifetimes are known at build time:
  //   * block temporaries (everything a ResBlock / transformer block allocates besides its output) live in a SCRATCH
  //     stack that is rewound when the block has been emitted (Scope);
  //   * the VAE decoder is a pure chain, its block outputs alternate between two PING-PONG slots;
  //   * weights, tables, skip-concat buffers, UNet block outputs and I/O stay in the persistent bump region.
  // Layout: [persistent | ping | pong | scratch]; the dry run measures the four sizes, the bound run places the bases.
  size_t soff = 0, speak = 0, pers_bytes = 0, pp_peak[2] = {0, 0};
  int pp_count = 0;
  uint8_t* sbase = nullptr;
  uint8_t* pp_base[2] = {nullptr, nullptr};
  void* salloc(size_t bytes, size_t align = 1024) {
    soff = (soff + align - 1) / align * align;
    void* p = dry ? nullptr : sbase + soff;
    soff += bytes;
    speak = std::max(speak, soff);
    return p;
  }
  T tmp(int B, int H, int W, int C) {
    T t;
    t.B = B; t.H = H; t.W = W; t.C = C; t.ld = C;
    t.p = static_cast<__half*>(salloc(static_cast<size_t>(B) * H * W * C * 2));
    return t;
  }
  T pingpong(int B, int H, int W, int C) {  // the tensor allocated two calls ago is dead by construction (pure chain)
    const int slot = pp_count++ & 1;
    const size_t bytes = static_cast<size_t>(B) * H * W * C * 2;
    pp_peak[slot] = std::max(pp_peak[slot], bytes);
    T t;
    t.B = B; t.H = H; t.W = W; t.C = C; t.ld = C;
    t.p = dry ? nullptr : reinterpret_cast<__half*>(pp_base[slot]);
    return t;
  }
  struct Scope {
    Engine* e;
    size_t mark;
    explicit Scope(Engine* eng) : e(eng), mark(eng->soff) {}
    ~Scope() { e->soff = mark; }
  };
  static T slice(const T& big, int c0, int C) {
    T t = big;
    t.p = big.p ? big.p + c0 : nullptr;
    t.C = C;
    return t;
  }

  // ---- parameters ----------------------------------------------------------
  const __half* w_packed(const std::string& name, int N, int C, int k, int geglu = 0, __half* into = nullptr,
                         bool placed = false) {
    const int cp = (C + 63) / 64 * 64;
    const size_t bytes = static_cast<size_t>(N) * k * k * cp * 2;
    __half* dst = placed ? into : static_cast<__half*>(alloc(bytes));
    ParamSlot s{P_PACKED, dst, N, C, k, k, geglu, static_cast<int64_t>(N) * C * k * k};
    params[name] = s;
    return dst;
  }
  // upsampler conv: four parity blocks of pre-summed 2x2 taps (pack_weight_up4)
  const __half* w_packed_up4(const std::string& name, int N, int C) {
    const int cp = (C + 63) / 64 * 64;
    __half* dst = static_cast<__half*>(alloc(static_cast<size_t>(N) * 16 * cp * 2));
    params[name] = ParamSlot{P_PACKED_UP4, dst, N, C, 3, 3, 0, static_cast<int64_t>(N) * C * 9};
    return dst;
  }
  const __half* w_raw(const std::string& name, int64_t numel) {
    __half* dst = static_cast<__half*>(alloc(static_cast<size_t>(numel) * 2));
    params[name] = ParamSlot{P_RAW, dst, 0, 0, 0, 0, 0, numel};
    return dst;
  }
  const float* vec(const std::string& name, int n, int geglu_N = 0) {
    float* dst = static_cast<float*>(alloc(static_cast<size_t>(n) * 4));
    params[name] = ParamSlot{P_VEC, dst, geglu_N, 0, 0, 0, 0, n};
    return dst;
  }

  // ---- op emission ---------------------------------------------------------
  std::vector<OpFn>* cur = nullptr;
  int* cur_count = nullptr;
  // tags parallel to the op lists (tooling: sdw_engine_debug_profile); `tag_next` names the op about to be emitted
  std::vector<std::string> prologue_tags, unet_tags, vae_tags;
  std::string tag_next;
  void emit(OpFn f, int launches = 1) {
    if (!dry) {
      cur->push_back(std::move(f));
      std::vector<std::string>& tags = cur == &prologue ? prologue_tags : (cur == &unet_ops ? unet_tags : vae_tags);
      tags.push_back(tag_next.empty() ? std::string("op") : tag_next);
    }
    tag_next.clear();
    *cur_count += launches;
  }
  int emit_gemm(const GemmDesc& d, const float* rowvec_table = nullptr, int rowvec_stride = 0) {
    if (dry) {
      *cur_count += 1;
      return 0;
    }
    auto L = std::make_shared<GemmLaunch>();
    if (int e = plan_gemm(d, L.get())) return e;
    {
      char buf[160];
      std::snprintf(buf, sizeof buf, "gemm conv%d C%d %dx%dx%d N%d mode%d bn%d nsub%d tr%d%s", d.conv, d.C, d.B, d.H, d.W, d.N,
                    d.mode, L->bn, L->nsub, L->tr, d.b_batched ? " batched" : "");
      tag_next = buf;
    }
    emit([L, rowvec_table, rowvec_stride](cudaStream_t st, int step) {
      if (rowvec_table) {
        GemmLaunch l = *L;
        l.p.rowvec = rowvec_table + static_cast<int64_t>(step) * rowvec_stride;
        l.p.rowvec_ld = 0;  // same vector for every sample of the batch
        return launch_gemm(l, st);
      }
      return launch_gemm(*L, st);
    }, 0);
    *cur_count += 1;
    return 0;
  }
  // tiled = True: circular padding (reference P:841-858 patches every Conv2d to padding_mode="circular").  A 3x3 conv on the
  // torus = the zero-padded conv of the wrap-padded image, cropped: pad (1 pixel; 2 for the stride-2 conv so that the
  // output centres stay on even coordinates), run the unchanged tcgen05 kernel on the padded lattice, crop (+ residual).
  bool tiled = false;
  int conv(const T& x, const __half* w, const float* bias, int N, int kind, const T& out, const T* resid = nullptr,
           const float* rowvec_table = nullptr, int mode = GEMM_PLAIN) {
    if (!tiled || kind == 0) return conv_zero_pad(x, w, bias, N, kind, out, resid, rowvec_table, mode);
    Scope scope(this);
    const int pad = kind == 2 ? 2 : 1;
    T xp = tmp(x.B, x.H + 2 * pad, x.W + 2 * pad, x.C);
    tag_next = "wrap pad (tiled)";
    emit([=](cudaStream_t st, int) { return wrap_pad(x.p, x.ld * 2, x.B, x.H, x.W, x.C * 2, pad, xp.p, st); });
    const int oh = kind == 2 ? xp.H / 2 : (kind == 3 ? xp.H * 2 : xp.H), ow = kind == 2 ? xp.W / 2 : (kind == 3 ? xp.W * 2 : xp.W);
    const int crop = kind == 3 ? 2 : 1;
    T yp = tmp(x.B, oh, ow, N);
    if (int e = conv_zero_pad(xp, w, bias, N, kind, yp, nullptr, rowvec_table, mode)) return e;
    const T r = resid ? *resid : T{};
    const bool has_r = resid != nullptr;
    tag_next = "crop (tiled)";
    emit([=](cudaStream_t st, int) {
      return crop_interior(yp.p, out.B, out.H, out.W, N * 2, crop, has_r ? r.p : nullptr, r.ld, out.p, out.ld * 2, st);
    });
    return 0;
  }
  // the 4-channel edge convs of both nets (CUDA-core kernels) in tiled mode: same pad / run / crop scheme
  int conv_in_edge(const T& xin, const __half* w, const float* b, int n, const T& o) {
    if (!tiled) {
      emit([=](cudaStream_t st, int) { return conv_in_small(xin.p, xin.ld, xin.B, xin.H, xin.W, xin.C, w, b, n, o.p, o.ld, st); });
      return 0;
    }
    Scope scope(this);
    T xp = tmp(xin.B, xin.H + 2, xin.W + 2, xin.C);
    T yp = tmp(xin.B, xin.H + 2, xin.W + 2, n);
    emit([=](cudaStream_t st, int) {
      if (int e = wrap_pad(xin.p, xin.ld * 2, xin.B, xin.H, xin.W, xin.C * 2, 1, xp.p, st)) return e;
      if (int e = conv_in_small(xp.p, xp.ld, xp.B, xp.H, xp.W, xp.C, w, b, n, yp.p, yp.ld, st)) return e;
      return crop_interior(yp.p, o.B, o.H, o.W, n * 2, 1, nullptr, 0, o.p, o.ld * 2, st);
    }, 3);
    return 0;
  }
  int conv_out_edge(const T& n, const __half* w, const float* b, int oc, float* out_f32, uint8_t* out_u8) {
    if (!tiled) {
      emit([=](cudaStream_t st, int) { return conv_out_small(n.p, n.ld, n.B, n.H, n.W, n.C, w, b, oc, out_f32, out_u8, st); });
      return 0;
    }
    Scope scope(this);
    T xp = tmp(n.B, n.H + 2, n.W + 2, n.C);
    const size_t pp = static_cast<size_t>(n.B) * (n.H + 2) * (n.W + 2);
    float* f32p = static_cast<float*>(salloc(pp * oc * 4));
    uint8_t* u8p = out_u8 ? static_cast<uint8_t*>(salloc(pp * oc)) : nullptr;
    emit([=](cudaStream_t st, int) {
      if (int e = wrap_pad(n.p, n.ld * 2, n.B, n.H, n.W, n.C * 2, 1, xp.p, st)) return e;
      if (int e = conv_out_small(xp.p, xp.ld, xp.B, xp.H, xp.W, xp.C, w, b, oc, f32p, u8p, st)) return e;
      if (out_f32)
        if (int e = crop_interior(f32p, n.B, n.H, n.W, oc * 4, 1, nullptr, 0, out_f32, oc * 4, st)) return e;
      if (out_u8) return crop_interior(u8p, n.B, n.H, n.W, oc, 1, nullptr, 0, out_u8, oc, st);
      return 0;
    }, 4);
    return 0;
  }
  int conv_zero_pad(const T& x, const __half* w, const float* bias, int N, int kind, const T& out, const T* resid = nullptr,
                    const float* rowvec_table = nullptr, int mode = GEMM_PLAIN) {
    const int npar = kind == 3 ? 4 : 1;
    for (int par = 0; par < npar; ++par) {
      GemmDesc d;
      d.A = x.p; d.C = x.C; d.W = x.W; d.H = x.H; d.B = x.B;
      d.sW = x.ld; d.sH = static_cast<int64_t>(x.W) * x.ld; d.sB = static_cast<int64_t>(x.H) * x.W * x.ld;
      d.conv = kind; d.up_py = par / 2; d.up_px = par % 2;
      d.Wt = w; d.N = N; d.bias = bias;
      if (kind == 3 && w) d.Wt = w + static_cast<size_t>(par) * N * 4 * ((x.C + 63) / 64 * 64);
      d.out = out.p; d.ldc = out.ld;
      if (resid) { d.resid = resid->p; d.ldr = resid->ld; }
      d.mode = mode;
      if (int e = emit_gemm(d, rowvec_table, N)) return e;
    }
    return 0;
  }
  // tokens view: treat [B,H,W,C] as one row lattice (W = B*H*W) — used for Linear layers
  int linear(const T& x, const __half* w, const float* bias, int N, const T& out, const T* resid = nullptr,
             int mode = GEMM_PLAIN) {
    GemmDesc d;
    d.A = x.p; d.C = x.C; d.W = static_cast<int>(x.pixels()); d.H = 1; d.B = 1;
    d.sW = x.ld; d.sH = 0; d.sB = 0;
    d.Wt = w; d.N = N; d.bias = bias;
    d.out = out.p; d.ldc = out.ld;
    if (resid) { d.resid = resid->p; d.ldr = resid->ld; }
    d.mode = mode;
    return emit_gemm(d);
  }
  void gn(const T& x, const std::string& name, float eps, int silu, const T& out) {
    const float* g = vec(name + ".weight", x.C);
    const float* b = vec(name + ".bias", x.C);
    const int G = cfg_groups;
    float2* ws = gn_ws;
    tag_next = "groupnorm C" + std::to_string(x.C) + " " + std::to_string(x.B) + "x" + std::to_string(x.H) + "x" + std::to_string(x.W);
    emit([=](cudaStream_t st, int) {
      return groupnorm(x.p, x.ld, x.B, static_cast<int64_t>(x.H) * x.W, x.C, G, g, b, eps, silu, out.p, out.ld, ws, st);
    }, groupnorm_launches());
  }
  void ln(const T& x, const std::string& name, const T& out) {
    const float* g = vec(name + ".weight", x.C);
    const float* b = vec(name + ".bias", x.C);
    tag_next = "layernorm C" + std::to_string(x.C) + " rows" + std::to_string(x.pixels());
    emit([=](cudaStream_t st, int) { return layernorm(x.p, x.ld, x.pixels(), x.C, g, b, 1e-5f, out.p, out.ld, st); });
  }
  int cfg_groups = 32;

  // unfused attention: S = alpha Q K^T (head-batched tcgen05 GEMM) ; softmax rows ; O = P V
  int attention(const __half* q, int64_t q_ld, const __half* k, int64_t k_ld, const __half* vt, int64_t vt_ld, int Bq,
                int Nq, int Nk, int heads, int d, const T& out) {
    if (attn_supported(d)) {
      if (dry) {
        *cur_count += 1;
        return 0;
      }
      AttnDesc a;
      a.q = q; a.q_ld = q_ld; a.k = k; a.k_ld = k_ld; a.vt = vt; a.vt_ld = vt_ld;
      a.B = Bq; a.Nq = Nq; a.Nk = Nk; a.heads = heads; a.d = d;
      a.out = out.p; a.out_ld = out.ld;
      auto L = std::make_shared<AttnLaunch>();
      if (int e = plan_attention(a, L.get())) return e;
      tag_next = "attention d" + std::to_string(d) + " B" + std::to_string(Bq) + " h" + std::to_string(heads) + " Nq" +
                 std::to_string(Nq) + " Nk" + std::to_string(Nk);
      emit([L](cudaStream_t st, int) { return launch_attention(*L, st); });
      return 0;
    }
    // S is materialised for a CHUNK of samples at a time (<= unfused_chunk(...) samples: about 64 MB of scores, which the
    // 126 MB L2 keeps resident between the QK^T GEMM, the row softmax and the PV GEMM) — not for the whole batch, which at
    // 30 frames of the VAE's 4096-token mid-block attention was 1 GB written once and read twice
    const int64_t Nkp = (Nk + 7) / 8 * 8;
    const int chunk = unfused_chunk(Bq, heads, Nq, Nkp);
    for (int b0 = 0; b0 < Bq; b0 += chunk) {
      const int nb = std::min(chunk, Bq - b0);
      GemmDesc g;
      g.A = q ? q + static_cast<int64_t>(b0) * Nq * q_ld : nullptr; g.C = d; g.W = Nq; g.H = heads; g.B = nb;
      g.sW = q_ld; g.sH = d; g.sB = static_cast<int64_t>(Nq) * q_ld;
      g.Wt = k ? k + static_cast<int64_t>(b0) * Nk * k_ld : nullptr; g.N = Nk; g.ldb = k_ld; g.Kb = d;
      g.b_batched = 1; g.sBh = d; g.sBb = static_cast<int64_t>(Nk) * k_ld;
      g.out = S; g.ldc = Nkp;
      g.o_sW = Nkp; g.o_sH = static_cast<int64_t>(Nq) * Nkp; g.o_sB = static_cast<int64_t>(heads) * Nq * Nkp;
      g.alpha = 1.f / std::sqrt(static_cast<float>(d));
      if (int e = emit_gemm(g)) return e;
      __half* Sp = S;
      const int64_t rows = static_cast<int64_t>(nb) * heads * Nq;
      emit([=](cudaStream_t st, int) { return softmax_rows(Sp, Nkp, rows, Nk, st); });
      GemmDesc h;
      h.A = S; h.C = Nk; h.W = Nq; h.H = heads; h.B = nb;
      h.sW = Nkp; h.sH = static_cast<int64_t>(Nq) * Nkp; h.sB = static_cast<int64_t>(heads) * Nq * Nkp;
      h.Wt = vt ? vt + static_cast<int64_t>(b0) * heads * d * vt_ld : nullptr; h.N = d; h.ldb = vt_ld; h.Kb = Nk;
      h.b_batched = 1; h.sBh = static_cast<int64_t>(d) * vt_ld; h.sBb = static_cast<int64_t>(heads) * d * vt_ld;
      h.out = out.p ? out.p + static_cast<int64_t>(b0) * Nq * out.ld : nullptr; h.ldc = out.ld;
      h.o_sW = out.ld; h.o_sH = d; h.o_sB = static_cast<int64_t>(Nq) * out.ld;
      if (int e = emit_gemm(h)) return e;
    }
    return 0;
  }
  // samples per chunk of the unfused attention: as many as fit ~64 MB of fp16 scores, at least one
  static int unfused_chunk(int Bq, int heads, int64_t Nq, int64_t Nkp) {
    const int64_t per_sample = static_cast<int64_t>(heads) * Nq * Nkp * 2;
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(Bq, (int64_t(64) << 20) / std::max<int64_t>(1, per_sample))));
  }

  // ---- model pieces ----------------------------------------------------------
  int resnet(const std::string& pre, const T& x, int cout, bool has_temb, float eps, const T& out) {
    Scope scope(this);
    T n1 = tmp(x.B, x.H, x.W, x.C);
    gn(x, pre + ".norm1", eps, 1, n1);
    T h1 = tmp(x.B, x.H, x.W, cout);
    const __half* w1 = w_packed(pre + ".conv1.weight", cout, x.C, 3);
    const float* b1 = vec(pre + ".conv1.bias", cout);
    const float* table = nullptr;
    if (has_temb) {
      TProj tp;
      tp.w = w_raw(pre + ".time_emb_proj.weight", static_cast<int64_t>(cout) * temb_ch());
      tp.b = vec(pre + ".time_emb_proj.bias", cout);
      tp.table = static_cast<float*>(alloc(static_cast<size_t>(cfg.max_steps) * cout * 4));
      tp.cout = cout;
      tprojs.push_back(tp);
      table = tp.table;
    }
    if (int e = conv(n1, w1, b1, cout, 1, h1, nullptr, table)) return e;
    T n2 = tmp(x.B, x.H, x.W, cout);
    gn(h1, pre + ".norm2", eps, 1, n2);
    const __half* w2 = w_packed(pre + ".conv2.weight", cout, cout, 3);
    const float* b2 = vec(pre + ".conv2.bias", cout);
    T res = x;
    if (x.C != cout) {
      const __half* ws = w_packed(pre + ".conv_shortcut.weight", cout, x.C, 1);
      const float* bs = vec(pre + ".conv_shortcut.bias", cout);
      T sc = tmp(x.B, x.H, x.W, cout);
      if (int e = conv(x, ws, bs, cout, 0, sc)) return e;
      res = sc;
    }
    return conv(n2, w2, b2, cout, 1, out, &res);
  }

  struct CrossKV { const __half* k; const __half* vt; int64_t k_ld, vt_ld; };

  int transformer(const std::string& pre, const T& x, int heads, const T& out) {
    const int C = x.C, d = C / heads, Bq = x.B, Nq = x.H * x.W;
    const int tokens = cfg.ctx_tokens, D = cfg.cross_attention_dim;
    Scope scope(this);
    T g0 = tmp(x.B, x.H, x.W, C);
    gn(x, pre + ".norm", 1e-6f, 0, g0);
    T hA = tmp(x.B, x.H, x.W, C);
    if (int e = conv(g0, w_packed(pre + ".proj_in.weight", C, C, 1), vec(pre + ".proj_in.bias", C), C, 0, hA)) return e;
    const std::string tb = pre + ".transformer_blocks.0";
    T t1 = tmp(x.B, x.H, x.W, C);
    // --- self attention
    ln(hA, tb + ".norm1", t1);
    __half* wqkv = static_cast<__half*>(alloc(static_cast<size_t>(3) * C * ((C + 63) / 64 * 64) * 2));
    const int cp = (C + 63) / 64 * 64;
    w_packed(tb + ".attn1.to_q.weight", C, C, 1, 0, wqkv, true);
    w_packed(tb + ".attn1.to_k.weight", C, C, 1, 0, wqkv ? wqkv + static_cast<size_t>(C) * cp : nullptr, true);
    w_packed(tb + ".attn1.to_v.weight", C, C, 1, 0, wqkv ? wqkv + static_cast<size_t>(2) * C * cp : nullptr, true);
    T qk = tmp(x.B, x.H, x.W, 2 * C);
    const int64_t vt_ld = (Nq + 7) / 8 * 8;
    __half* vt = static_cast<__half*>(salloc(static_cast<size_t>(Bq) * heads * d * vt_ld * 2));
    {
      GemmDesc g;
      g.A = t1.p; g.C = C; g.W = Nq; g.H = 1; g.B = Bq;
      g.sW = t1.ld; g.sH = 0; g.sB = static_cast<int64_t>(Nq) * t1.ld;
      g.Wt = wqkv; g.N = 3 * C;
      g.out = qk.p; g.ldc = qk.ld;
      g.mode = GEMM_QKV_VT;
      g.vt_col0 = 2 * C; g.vt_d = d; g.vt_heads = heads; g.vt_ntok = Nq; g.vt = vt; g.vt_ld = vt_ld;
      if (int e = emit_gemm(g)) return e;
    }
    T ao = tmp(x.B, x.H, x.W, C);
    if (int e = attention(qk.p, qk.ld, qk.p ? qk.p + C : nullptr, qk.ld, vt, vt_ld, Bq, Nq, Nq, heads, d, ao)) return e;
    T hB = tmp(x.B, x.H, x.W, C);
    if (int e = linear(ao, w_packed(tb + ".attn1.to_out.0.weight", C, C, 1), vec(tb + ".attn1.to_out.0.bias", C), C,
                       hB, &hA))
      return e;
    // --- cross attention (K/V of the text context are step-invariant: computed in the prologue)
    ln(hB, tb + ".norm2", t1);
    T q2 = tmp(x.B, x.H, x.W, C);
    if (int e = linear(t1, w_packed(tb + ".attn2.to_q.weight", C, C, 1), nullptr, C, q2)) return e;
    const int dcp = (D + 63) / 64 * 64;
    __half* wkv = static_cast<__half*>(alloc(static_cast<size_t>(2) * C * dcp * 2));
    w_packed(tb + ".attn2.to_k.weight", C, D, 1, 0, wkv, true);
    w_packed(tb + ".attn2.to_v.weight", C, D, 1, 0, wkv ? wkv + static_cast<size_t>(C) * dcp : nullptr, true);
    __half* kx = static_cast<__half*>(alloc(static_cast<size_t>(Bq) * tokens * C * 2));
    const int64_t vx_ld = (tokens + 7) / 8 * 8;
    __half* vx = static_cast<__half*>(alloc(static_cast<size_t>(Bq) * heads * d * vx_ld * 2));
    {
      std::vector<OpFn>* save = cur;
      int* save_c = cur_count;
      cur = &prologue;
      cur_count = &n_launch_prologue;
      GemmDesc g;
      g.A = ctx; g.C = D; g.W = Bq * tokens; g.H = 1; g.B = 1;
      g.sW = D;
      g.Wt = wkv; g.N = 2 * C;
      g.out = kx; g.ldc = C;
      g.mode = GEMM_QKV_VT;
      g.vt_col0 = C; g.vt_d = d; g.vt_heads = heads; g.vt_ntok = tokens; g.vt = vx; g.vt_ld = vx_ld;
      int e = emit_gemm(g);
      cur = save;
      cur_count = save_c;
      if (e) return e;
    }
    if (int e = attention(q2.p, q2.ld, kx, C, vx, vx_ld, Bq, Nq, tokens, heads, d, ao)) return e;
    T hC = tmp(x.B, x.H, x.W, C);
    if (int e = linear(ao, w_packed(tb + ".attn2.to_out.0.weight", C, C, 1), vec(tb + ".attn2.to_out.0.bias", C), C,
                       hC, &hB))
      return e;
    // --- feed-forward (GEGLU)
    ln(hC, tb + ".norm3", t1);
    T ff = tmp(x.B, x.H, x.W, 4 * C);
    if (int e = linear(t1, w_packed(tb + ".ff.net.0.proj.weight", 8 * C, C, 1, 1),
                       vec(tb + ".ff.net.0.proj.bias", 8 * C, 8 * C), 8 * C, ff, nullptr, GEMM_GEGLU))
      return e;
    T hD = tmp(x.B, x.H, x.W, C);
    if (int e = linear(ff, w_packed(tb + ".ff.net.2.weight", C, 4 * C, 1), vec(tb + ".ff.net.2.bias", C), C, hD, &hC))
      return e;
    return conv(hD, w_packed(pre + ".proj_out.weight", C, C, 1), vec(pre + ".proj_out.bias", C), C, 0, out, &x);
  }

  int temb_ch() const { return cfg.block_out_channels[0] * 4; }
  int heads_at(int level) const { return cfg.attention_heads[level]; }

  int build_unet() {
    cur = &unet_ops;
    cur_count = &n_launch_unet;
    cfg_groups = cfg.norm_num_groups;
    const int nlev = cfg.num_levels, L = cfg.layers_per_block;
    const int* ch = cfg.block_out_channels;
    const int H0 = cfg.latent_h, W0 = cfg.latent_w;
    SDW_REQUIRE((H0 % (1 << (nlev - 1))) == 0 && (W0 % (1 << (nlev - 1))) == 0,
                "latent size must be divisible by 2^(levels-1)");
    // time embedding parameters
    te_w1 = w_raw("time_embedding.linear_1.weight", static_cast<int64_t>(temb_ch()) * ch[0]);
    te_b1 = vec("time_embedding.linear_1.bias", temb_ch());
    te_w2 = w_raw("time_embedding.linear_2.weight", static_cast<int64_t>(temb_ch()) * temb_ch());
    te_b2 = vec("time_embedding.linear_2.bias", temb_ch());
    // concat buffers of the up path: cat[i][j] = [h (rin) | skip]
    std::vector<int> rev(ch, ch + nlev);
    std::reverse(rev.begin(), rev.end());
    struct CatInfo { T buf; int rin, skip; };
    std::vector<std::vector<CatInfo>> cat(nlev);
    {
      int cout = rev[0];
      for (int i = 0; i < nlev; ++i) {
        const int prev = cout;
        cout = rev[i];
        const int cin = rev[std::min(i + 1, nlev - 1)];
        const int lev = nlev - 1 - i;
        for (int j = 0; j <= L; ++j) {
          CatInfo ci;
          ci.skip = (j == L) ? cin : cout;
          ci.rin = (j == 0) ? prev : cout;
          ci.buf = act(Bn, H0 >> lev, W0 >> lev, ci.rin + ci.skip);
          cat[i].push_back(ci);
        }
      }
    }
    const int n_skips = nlev * (L + 1);
    auto skip_dest = [&](int k) {  // k-th pushed skip is popped by consumer index n_skips-1-k
      const int c = n_skips - 1 - k;
      CatInfo& ci = cat[c / (L + 1)][c % (L + 1)];
      return slice(ci.buf, ci.rin, ci.skip);
    };
    int k = 0;
    // conv_in
    T xin;
    xin.p = model_in; xin.B = Bn; xin.H = H0; xin.W = W0; xin.C = cfg.in_channels; xin.ld = cfg.in_channels;
    T h = skip_dest(k++);
    {
      const __half* w = w_raw("conv_in.weight", static_cast<int64_t>(ch[0]) * cfg.in_channels * 9);
      const float* b = vec("conv_in.bias", ch[0]);
      const T o = h;
      const int cin = cfg.in_channels, n = ch[0];
      tag_next = "conv_in 4->C (CUDA cores)";
      (void)cin;
      if (int e = conv_in_edge(xin, w, b, n, o)) return e;
    }
    // down path
    for (int i = 0; i < nlev; ++i) {
      const bool last = i == nlev - 1;
      const std::string bp = "down_blocks." + std::to_string(i);
      for (int j = 0; j < L; ++j) {
        T dest = skip_dest(k++);
        if (!last) {
          T r = act(h.B, h.H, h.W, ch[i]);
          if (int e = resnet(bp + ".resnets." + std::to_string(j), h, ch[i], true, cfg.norm_eps, r)) return e;
          if (int e = transformer(bp + ".attentions." + std::to_string(j), r, heads_at(i), dest)) return e;
        } else {
          if (int e = resnet(bp + ".resnets." + std::to_string(j), h, ch[i], true, cfg.norm_eps, dest)) return e;
        }
        h = dest;
      }
      if (!last) {
        T dest = skip_dest(k++);
        if (int e = conv(h, w_packed(bp + ".downsamplers.0.conv.weight", ch[i], ch[i], 3),
                         vec(bp + ".downsamplers.0.conv.bias", ch[i]), ch[i], 2, dest))
          return e;
        h = dest;
      }
    }
    // mid
    {
      const int c = ch[nlev - 1];
      T a = act(h.B, h.H, h.W, c), b = act(h.B, h.H, h.W, c);
      if (int e = resnet("mid_block.resnets.0", h, c, true, cfg.norm_eps, a)) return e;
      if (int e = transformer("mid_block.attentions.0", a, heads_at(nlev - 1), b)) return e;
      T dest = slice(cat[0][0].buf, 0, cat[0][0].rin);
      if (int e = resnet("mid_block.resnets.1", b, c, true, cfg.norm_eps, dest)) return e;
    }
    // up path
    T final_h;
    for (int i = 0; i < nlev; ++i) {
      const bool last = i == nlev - 1;
      const int cout = rev[i];
      const int lev = nlev - 1 - i;
      const std::string bp = "up_blocks." + std::to_string(i);
      T up_in;
      for (int j = 0; j <= L; ++j) {
        const T xcat = cat[i][j].buf;
        T dest;
        if (j < L) dest = slice(cat[i][j + 1].buf, 0, cout);
        else dest = act(Bn, H0 >> lev, W0 >> lev, cout);
        if (i > 0) {
          T r = act(xcat.B, xcat.H, xcat.W, cout);
          if (int e = resnet(bp + ".resnets." + std::to_string(j), xcat, cout, true, cfg.norm_eps, r)) return e;
          if (int e = transformer(bp + ".attentions." + std::to_string(j), r, heads_at(lev), dest)) return e;
        } else {
          if (int e = resnet(bp + ".resnets." + std::to_string(j), xcat, cout, true, cfg.norm_eps, dest)) return e;
        }
        up_in = dest;
      }
      if (!last) {
        T dest = slice(cat[i + 1][0].buf, 0, cat[i + 1][0].rin);
        if (int e = conv(up_in, w_packed_up4(bp + ".upsamplers.0.conv.weight", cout, cout),
                         vec(bp + ".upsamplers.0.conv.bias", cout), cout, 3, dest))
          return e;
      } else {
        final_h = up_in;
      }
    }
    // out
    T n = act(final_h.B, final_h.H, final_h.W, final_h.C);
    gn(final_h, "conv_norm_out", cfg.norm_eps, 1, n);
    {
      const __half* w = w_raw("conv_out.weight", static_cast<int64_t>(cfg.out_channels) * ch[0] * 9);
      const float* b = vec("conv_out.bias", cfg.out_channels);
      float* e_out = eps;
      const int oc = cfg.out_channels;
      tag_next = "conv_out C->4 (CUDA cores)";
      if (int e = conv_out_edge(n, w, b, oc, e_out, nullptr)) return e;
    }
    return 0;
  }

  int build_vae() {
    cur = &vae_ops;
    cur_count = &n_launch_vae;
    cfg_groups = cfg.vae_norm_num_groups;
    const int F = cfg.frames, H0 = cfg.latent_h, W0 = cfg.latent_w, lc = cfg.in_channels;
    const int nlev = cfg.vae_num_levels;
    const int* ch = cfg.vae_block_out_channels;
    const int ctop = ch[nlev - 1];
    // post_quant_conv (1x1, lc -> lc) on latents / scaling_factor
    T z = pingpong(F, H0, W0, lc);
    {
      const __half* w = w_raw("vae.post_quant_conv.weight", static_cast<int64_t>(lc) * lc);
      const float* b = vec("vae.post_quant_conv.bias", lc);
      const float* xs = x;
      const float inv = 1.f / cfg.vae_scaling_factor;
      tag_next = "vae_in (scale + post_quant 1x1)";
      emit([=](cudaStream_t st, int) { return vae_in(xs, inv, w, b, F, lc, H0, W0, z.p, st); });
    }
    T h = pingpong(F, H0, W0, ctop);
    {
      const __half* w = w_raw("vae.decoder.conv_in.weight", static_cast<int64_t>(ctop) * lc * 9);
      const float* b = vec("vae.decoder.conv_in.bias", ctop);
      const T o = h;
      tag_next = "vae conv_in 4->C (CUDA cores)";
      if (int e = conv_in_edge(z, w, b, ctop, o)) return e;
    }
    // mid block
    {
      T a = pingpong(F, H0, W0, ctop);
      if (int e = resnet("vae.decoder.mid_block.resnets.0", h, ctop, false, 1e-6f, a)) return e;
      // single-head attention, d = C
      const std::string ap = "vae.decoder.mid_block.attentions.0";
      Scope scope(this);
      T g0 = tmp(F, H0, W0, ctop);
      gn(a, ap + ".group_norm", 1e-6f, 0, g0);
      const int C = ctop, Nq = H0 * W0, cp = (C + 63) / 64 * 64;
      __half* wqkv = static_cast<__half*>(alloc(static_cast<size_t>(3) * C * cp * 2));
      w_packed(ap + ".to_q.weight", C, C, 1, 0, wqkv, true);
      w_packed(ap + ".to_k.weight", C, C, 1, 0, wqkv ? wqkv + static_cast<size_t>(C) * cp : nullptr, true);
      w_packed(ap + ".to_v.weight", C, C, 1, 0, wqkv ? wqkv + static_cast<size_t>(2) * C * cp : nullptr, true);
      float* bqkv = static_cast<float*>(alloc(static_cast<size_t>(3) * C * 4));
      params[ap + ".to_q.bias"] = ParamSlot{P_VEC, bqkv, 0, 0, 0, 0, 0, C};
      params[ap + ".to_k.bias"] = ParamSlot{P_VEC, bqkv ? bqkv + C : nullptr, 0, 0, 0, 0, 0, C};
      params[ap + ".to_v.bias"] = ParamSlot{P_VEC, bqkv ? bqkv + 2 * C : nullptr, 0, 0, 0, 0, 0, C};
      T qk = tmp(F, H0, W0, 2 * C);
      const int64_t vt_ld = (Nq + 7) / 8 * 8;
      __half* vt = static_cast<__half*>(salloc(static_cast<size_t>(F) * C * vt_ld * 2));
      {
        GemmDesc g;
        g.A = g0.p; g.C = C; g.W = Nq; g.H = 1; g.B = F;
        g.sW = g0.ld; g.sH = 0; g.sB = static_cast<int64_t>(Nq) * g0.ld;
        g.Wt = wqkv; g.N = 3 * C; g.bias = bqkv;
        g.out = qk.p; g.ldc = qk.ld;
        g.mode = GEMM_QKV_VT;
        g.vt_col0 = 2 * C; g.vt_d = C; g.vt_heads = 1; g.vt_ntok = Nq; g.vt = vt; g.vt_ld = vt_ld;
        if (int e = emit_gemm(g)) return e;
      }
      T ao = tmp(F, H0, W0, C);
      if (int e = attention(qk.p, qk.ld, qk.p ? qk.p + C : nullptr, qk.ld, vt, vt_ld, F, Nq, Nq, 1, C, ao)) return e;
      T b = pingpong(F, H0, W0, C);
      if (int e = linear(ao, w_packed(ap + ".to_out.0.weight", C, C, 1), vec(ap + ".to_out.0.bias", C), C, b, &a))
        return e;
      T c = pingpong(F, H0, W0, C);
      if (int e = resnet("vae.decoder.mid_block.resnets.1", b, ctop, false, 1e-6f, c)) return e;
      h = c;
    }
    // up blocks
    int cout = ctop;
    for (int i = 0; i < nlev; ++i) {
      cout = ch[nlev - 1 - i];
      const std::string bp = "vae.decoder.up_blocks." + std::to_string(i);
      for (int j = 0; j <= cfg.vae_layers_per_block; ++j) {
        T o = pingpong(h.B, h.H, h.W, cout);
        if (int e = resnet(bp + ".resnets." + std::to_string(j), h, cout, false, 1e-6f, o)) return e;
        h = o;
      }
      if (i < nlev - 1) {
        T o = pingpong(h.B, h.H * 2, h.W * 2, cout);
        if (int e = conv(h, w_packed_up4(bp + ".upsamplers.0.conv.weight", cout, cout),
                         vec(bp + ".upsamplers.0.conv.bias", cout), cout, 3, o))
          return e;
        h = o;
      }
    }
    T n = pingpong(h.B, h.H, h.W, h.C);
    gn(h, "vae.decoder.conv_norm_out", 1e-6f, 1, n);
    {
      const __half* w = w_raw("vae.decoder.conv_out.weight", static_cast<int64_t>(cfg.vae_out_channels) * h.C * 9);
      const float* b = vec("vae.decoder.conv_out.bias", cfg.vae_out_channels);
      uint8_t* o8 = out_u8;
      float* of = out_img_f32;
      const int oc = cfg.vae_out_channels;
      tag_next = "vae conv_out C->3 + uint8 (CUDA cores)";
      if (int e = conv_out_edge(n, w, b, oc, of, o8)) return e;
    }
    return 0;
  }

  int build(bool dry_run, void* arena) {
    dry = dry_run;
    base = static_cast<uint8_t*>(arena);
    off = 0;
    soff = 0;
    pp_count = 0;
    if (dry) {
      speak = pp_peak[0] = pp_peak[1] = 0;
    } else {  // sizes measured by the dry run
      pp_base[0] = base + pers_bytes;
      pp_base[1] = pp_base[0] + (pp_peak[0] + 1023) / 1024 * 1024;
      sbase = pp_base[1] + (pp_peak[1] + 1023) / 1024 * 1024;
    }
    params.clear();
    prologue.clear(); unet_ops.clear(); vae_ops.clear(); tprojs.clear();
    n_launch_prologue = n_launch_unet = n_launch_vae = 0;
    const int F = cfg.frames, H = cfg.latent_h, W = cfg.latent_w, lc = cfg.in_channels;
    Bn = F * (cfg.guidance ? 2 : 1);
    const int64_t nlat = static_cast<int64_t>(F) * lc * H * W;
    model_in = static_cast<__half*>(alloc(static_cast<size_t>(Bn) * H * W * lc * 2));
    eps = static_cast<float*>(alloc(static_cast<size_t>(Bn) * H * W * cfg.out_channels * 4));
    x = static_cast<float*>(alloc(nlat * 4));
    x_base = static_cast<float*>(alloc(nlat * 4));
    hist = static_cast<float*>(alloc(nlat * 4 * 4));
    lat_stage = alloc(nlat * 4);
    const int64_t per = static_cast<int64_t>(cfg.ctx_tokens) * cfg.cross_attention_dim;
    ctx = static_cast<__half*>(alloc(static_cast<size_t>(Bn) * per * 2));
    cond_stage = static_cast<__half*>(alloc(static_cast<size_t>(Bn) * per * 2));  // room for a full [Bn] context
    uncond_stage = static_cast<__half*>(alloc(static_cast<size_t>(cfg.frames) * per * 2));
    const int OH = H * cfg.vae_scale, OW = W * cfg.vae_scale;
    out_u8 = static_cast<uint8_t*>(alloc(static_cast<size_t>(F) * OH * OW * cfg.vae_out_channels));
    out_img_f32 = static_cast<float*>(alloc(static_cast<size_t>(F) * OH * OW * cfg.vae_out_channels * 4));
    gn_ws = static_cast<float2*>(alloc(gn_workspace_bytes(std::max(Bn, F))));
    // attention score scratch of the UNFUSED path: the VAE mid attention (d = 512), and UNet level-0 self attention only
    // when its head dim has no fused kernel
    {
      const int64_t n0 = static_cast<int64_t>(H) * W;
      int64_t unet_s = 0;
      for (int l = 0; l < cfg.num_levels; ++l) {
        const int hl = std::max(1, cfg.attention_heads[l]);
        if (attn_supported(cfg.block_out_channels[l] / hl)) continue;
        const int64_t nl = static_cast<int64_t>(H >> l) * (W >> l);
        const int64_t nlp = (nl + 7) / 8 * 8;
        unet_s = std::max(unet_s, static_cast<int64_t>(unfused_chunk(Bn, hl, nl, nlp)) * hl * nl * nlp);
      }
      const int64_t n0p = (n0 + 7) / 8 * 8;
      int64_t vae_s = static_cast<int64_t>(unfused_chunk(F, 1, n0, n0p)) * n0 * n0p;  // a chunk of samples, not the batch
      S_elems = static_cast<size_t>(std::max(unet_s, vae_s));
      S = static_cast<__half*>(alloc(S_elems * 2));
    }
    t_dev = static_cast<float*>(alloc(static_cast<size_t>(cfg.max_steps) * 4));
    t_sin = static_cast<float*>(alloc(static_cast<size_t>(cfg.max_steps) * cfg.block_out_channels[0] * 4));
    t_h1 = static_cast<float*>(alloc(static_cast<size_t>(cfg.max_steps) * temb_ch() * 4));
    temb = static_cast<float*>(alloc(static_cast<size_t>(cfg.max_steps) * temb_ch() * 4));
    if (int e = build_unet()) return e;
    if (int e = build_vae()) return e;
    if (dry) {
      pers_bytes = (off + 4095) / 4096 * 4096;
      arena_bytes = pers_bytes + (pp_peak[0] + 1023) / 1024 * 1024 + (pp_peak[1] + 1023) / 1024 * 1024 + speak + 4096;
    }
    return 0;
  }
};

}  // namespace
}  // namespace sdw

// ================================================================================================
// C ABI
// ================================================================================================
using namespace sdw;

namespace sdw {
__global__ void ctx_assemble_kernel(const __half* __restrict__ cond, const __half* __restrict__ uncond, int F, int dup,
                                    int64_t per, __half* __restrict__ out, int uncond_per_frame) {
  const int64_t total = static_cast<int64_t>(F) * (dup ? 2 : 1) * per;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t b = i / per, r = i % per;
    if (dup) out[i] = b < F ? uncond[(uncond_per_frame ? b * per : 0) + r] : cond[(b - F) * per + r];  // cat([uncond(.repeat(F)), cond]) — P:352-358
    else out[i] = cond[i];
  }
}
int unet_ctx_assemble(const __half* cond, const __half* uncond, int F, int dup, int64_t per, __half* out,
                      cudaStream_t stream, int uncond_per_frame = 0) {
  ctx_assemble_kernel<<<148 * 2, 256, 0, stream>>>(cond, uncond, F, dup, per, out, uncond_per_frame);
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}
}  // namespace sdw

static int validate(const sdw_engine_config* c) {
  SDW_REQUIRE(c != nullptr, "null config");
  SDW_REQUIRE(c->num_levels >= 1 && c->num_levels <= 4 && c->vae_num_levels >= 1 && c->vae_num_levels <= 4,
              "1..4 levels");
  SDW_REQUIRE(c->in_channels == 4 && (c->out_channels == 4), "latent channels must be 4");
  SDW_REQUIRE(c->vae_out_channels == 3, "VAE decoder must output 3 channels");
  SDW_REQUIRE(c->frames >= 1 && c->latent_h >= 1 && c->latent_w >= 1, "bad sizes");
  SDW_REQUIRE(c->max_steps >= 1 && c->max_steps <= 1024, "max_steps in 1..1024");
  SDW_REQUIRE(c->cross_attention_dim % 8 == 0 && c->ctx_tokens >= 1, "bad context shape");
  for (int i = 0; i < c->num_levels; ++i) {
    const int ch = c->block_out_channels[i];
    SDW_REQUIRE(ch % 8 == 0 && ch % c->norm_num_groups == 0, "UNet channels must divide by 8 and by the groups");
    SDW_REQUIRE(c->attention_heads[i] >= 1 && ch % c->attention_heads[i] == 0 &&
                    (ch / c->attention_heads[i]) % 8 == 0,
                "head dim must be a multiple of 8");
    SDW_REQUIRE(ch % 32 == 0, "UNet channels must be multiples of 32 (QKV split)");
  }
  for (int i = 0; i < c->vae_num_levels; ++i)
    SDW_REQUIRE(c->vae_block_out_channels[i] % 8 == 0 && c->vae_block_out_channels[i] % c->vae_norm_num_groups == 0,
                "VAE channels must divide by 8 and by the groups");
  SDW_REQUIRE(c->vae_block_out_channels[c->vae_num_levels - 1] % 32 == 0, "VAE top channels multiple of 32");
  SDW_REQUIRE(c->vae_scale == (1 << (c->vae_num_levels - 1)), "vae_scale must be 2^(vae levels - 1)");
  return 0;
}

extern "C" {

int sdw_engine_create(const sdw_engine_config* cfg, sdw_engine** out) {
  SDW_REQUIRE(out != nullptr, "null out");
  if (int e = validate(cfg)) return e;
  Engine* E = new Engine();
  E->cfg = *cfg;
  E->tiled = cfg->tiled != 0;
  if (int e = E->build(true, nullptr)) {
    delete E;
    return e;
  }
  *out = reinterpret_cast<sdw_engine*>(E);
  return 0;
}

void sdw_engine_destroy(sdw_engine* e) {
  Engine* E = reinterpret_cast<Engine*>(e);
  if (!E) return;
  if (E->graph_exec) cudaGraphExecDestroy(E->graph_exec);
  delete E;
}

int sdw_engine_arena_bytes(const sdw_engine* e, uint64_t* bytes) {
  SDW_REQUIRE(e && bytes, "null");
  *bytes = reinterpret_cast<const Engine*>(e)->arena_bytes;
  return 0;
}

int sdw_engine_bind(sdw_engine* e, void* arena, uint64_t bytes) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && arena, "null");
  SDW_REQUIRE(bytes >= E->arena_bytes, "arena too small");
  SDW_REQUIRE(reinterpret_cast<uintptr_t>(arena) % 1024 == 0, "arena must be 1024-byte aligned");
  if (int err = gemm_init()) return err;
  if (E->graph_exec) {
    cudaGraphExecDestroy(E->graph_exec);
    E->graph_exec = nullptr;
  }
  return E->build(false, arena);
}

int sdw_engine_num_params(const sdw_engine* e) { return e ? static_cast<int>(reinterpret_cast<const Engine*>(e)->params.size()) : -1; }

int sdw_engine_param_info(const sdw_engine* e, int index, const char** name, int64_t* numel) {
  const Engine* E = reinterpret_cast<const Engine*>(e);
  SDW_REQUIRE(E && index >= 0 && index < static_cast<int>(E->params.size()), "bad index");
  auto it = E->params.begin();
  std::advance(it, index);
  if (name) *name = it->first.c_str();
  if (numel) *numel = it->second.numel;
  return 0;
}

int sdw_engine_load_param(sdw_engine* e, const char* name, const void* src_f16, int64_t numel, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && name && src_f16, "null");
  SDW_REQUIRE(!E->dry, "engine not bound to an arena");
  auto it = E->params.find(name);
  if (it == E->params.end()) {
    set_error(std::string("unknown parameter: ") + name);
    return 1;
  }
  ParamSlot& s = it->second;
  if (s.numel != numel) {
    set_error(std::string("parameter size mismatch for ") + name + ": expected " + std::to_string(s.numel) + ", got " +
              std::to_string(numel));
    return 1;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = 0;
  if (s.kind == P_PACKED) rc = pack_weight(src_f16, s.N, s.C, s.kh, s.kw, s.geglu, s.dst, st);
  else if (s.kind == P_PACKED_UP4) rc = pack_weight_up4(src_f16, s.N, s.C, s.dst, st);
  else if (s.kind == P_RAW) {
    SDW_CUDA_OK(cudaMemcpyAsync(s.dst, src_f16, static_cast<size_t>(numel) * 2, cudaMemcpyDeviceToDevice, st));
  } else rc = half_to_float(static_cast<const __half*>(src_f16), static_cast<float*>(s.dst), numel, s.N, st);
  if (rc == 0) s.loaded = true;
  return rc;
}

int sdw_engine_missing_params(const sdw_engine* e, const char** first_missing) {
  const Engine* E = reinterpret_cast<const Engine*>(e);
  SDW_REQUIRE(E, "null");
  int n = 0;
  for (auto& kv : E->params)
    if (!kv.second.loaded) {
      if (n == 0 && first_missing) *first_missing = kv.first.c_str();
      ++n;
    }
  return n;
}

int sdw_engine_set_schedule(sdw_engine* e, int n_steps, const float* timesteps, const sdw_step_coef* coefs,
                            float init_noise_sigma, float first_in_scale, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && timesteps && coefs, "null");
  SDW_REQUIRE(!E->dry, "engine not bound");
  SDW_REQUIRE(n_steps >= 1 && n_steps <= E->cfg.max_steps, "n_steps exceeds max_steps");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  E->n_steps = n_steps;
  E->coefs.assign(coefs, coefs + n_steps);
  E->init_sigma = init_noise_sigma;
  E->first_in_scale = first_in_scale;
  if (E->graph_exec) {
    cudaGraphExecDestroy(E->graph_exec);
    E->graph_exec = nullptr;
  }
  SDW_CUDA_OK(cudaMemcpyAsync(E->t_dev, timesteps, static_cast<size_t>(n_steps) * 4, cudaMemcpyHostToDevice, st));
  SDW_CUDA_OK(cudaStreamSynchronize(st));  // the host array may be a temporary
  const int c0 = E->cfg.block_out_channels[0], tc = E->temb_ch();
  if (int rc = timestep_embed(E->t_dev, n_steps, c0, 0, E->t_sin, st)) return rc;
  if (int rc = linear_f32(E->t_sin, c0, E->te_w1, E->te_b1, n_steps, tc, c0, 0, 1, E->t_h1, tc, st)) return rc;
  if (int rc = linear_f32(E->t_h1, tc, E->te_w2, E->te_b2, n_steps, tc, tc, 0, 0, E->temb, tc, st)) return rc;
  for (auto& tp : E->tprojs)
    if (int rc = linear_f32(E->temb, tc, tp.w, tp.b, n_steps, tp.cout, tc, 1, 0, tp.table, tp.cout, st)) return rc;
  return 0;
}

static int run_ops(std::vector<OpFn>& ops, cudaStream_t st, int step) {
  for (auto& f : ops)
    if (int rc = f(st, step)) return rc;
  return 0;
}

static int run_all(Engine* E, cudaStream_t st) {
  const sdw_engine_config& c = E->cfg;
  const int F = c.frames, H = c.latent_h, W = c.latent_w, lc = c.in_channels;
  const int64_t per = static_cast<int64_t>(c.ctx_tokens) * c.cross_attention_dim;
  if (int rc = unet_ctx_assemble(E->cond_stage, E->uncond_stage, F, c.guidance, per, E->ctx, st, E->uncond_batch > 1)) return rc;
  if (int rc = run_ops(E->prologue, st, 0)) return rc;
  if (int rc = latents_init(E->lat_stage, 0, E->init_sigma, E->first_in_scale, E->x, E->model_in, lc, c.guidance, F, lc,
                            H, W, st))
    return rc;
  for (int s = 0; s < E->n_steps; ++s) {
    if (int rc = run_ops(E->unet_ops, st, s)) return rc;
    if (int rc = cfg_sched_step(E->eps, c.guidance, E->x, E->x_base, E->hist, &E->coefs[s], F, lc, H, W,
                                s + 1 < E->n_steps ? E->model_in : nullptr, lc, st))
      return rc;
  }
  return run_ops(E->vae_ops, st, 0);
}

static int stage_inputs(Engine* E, const float* latents_f32, const void* cond_f16, const void* uncond_f16,
                        cudaStream_t st) {
  const sdw_engine_config& c = E->cfg;
  const int64_t nlat = static_cast<int64_t>(c.frames) * c.in_channels * c.latent_h * c.latent_w;
  const int64_t per = static_cast<int64_t>(c.ctx_tokens) * c.cross_attention_dim;
  SDW_CUDA_OK(cudaMemcpyAsync(E->lat_stage, latents_f32, nlat * 4, cudaMemcpyDeviceToDevice, st));
  SDW_CUDA_OK(cudaMemcpyAsync(E->cond_stage, cond_f16, static_cast<size_t>(c.frames) * per * 2, cudaMemcpyDeviceToDevice, st));
  if (c.guidance)
    SDW_CUDA_OK(cudaMemcpyAsync(E->uncond_stage, uncond_f16, static_cast<size_t>(E->uncond_batch) * per * 2, cudaMemcpyDeviceToDevice, st));
  return 0;
}

static int copy_outputs(Engine* E, uint8_t* out_u8, float* out_latents, float* out_raw_f32, cudaStream_t st) {
  const sdw_engine_config& c = E->cfg;
  const int64_t nlat = static_cast<int64_t>(c.frames) * c.in_channels * c.latent_h * c.latent_w;
  const size_t out_bytes = static_cast<size_t>(c.frames) * c.latent_h * c.vae_scale * c.latent_w * c.vae_scale * c.vae_out_channels;
  if (out_u8) SDW_CUDA_OK(cudaMemcpyAsync(out_u8, E->out_u8, out_bytes, cudaMemcpyDeviceToDevice, st));
  if (out_latents) SDW_CUDA_OK(cudaMemcpyAsync(out_latents, E->x, nlat * 4, cudaMemcpyDeviceToDevice, st));
  if (out_raw_f32)
    SDW_CUDA_OK(cudaMemcpyAsync(out_raw_f32, E->out_img_f32, out_bytes * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int sdw_engine_sample(sdw_engine* e, const float* latents_f32, const void* cond_f16, const void* uncond_f16,
                      uint8_t* out_u8, float* out_latents, float* out_raw_f32, int use_graph, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && latents_f32 && cond_f16 && out_u8, "null");
  SDW_REQUIRE(!E->dry && E->n_steps > 0, "engine not bound or schedule not set");
  SDW_REQUIRE(!E->cfg.guidance || uncond_f16, "guidance needs the unconditional embedding");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = stage_inputs(E, latents_f32, cond_f16, uncond_f16, st)) return rc;
  if (use_graph) {
    if (!E->graph_exec || E->graph_steps != E->n_steps) {
      if (E->graph_exec) {
        cudaGraphExecDestroy(E->graph_exec);
        E->graph_exec = nullptr;
      }
      cudaGraph_t graph = nullptr;
      SDW_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      int rc = run_all(E, st);
      cudaError_t ce = cudaStreamEndCapture(st, &graph);
      if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
      }
      SDW_CUDA_OK(ce);
      SDW_CUDA_OK(cudaGraphInstantiate(&E->graph_exec, graph, 0));
      cudaGraphDestroy(graph);
      E->graph_steps = E->n_steps;
    }
    SDW_CUDA_OK(cudaGraphLaunch(E->graph_exec, st));
  } else {
    if (int rc = run_all(E, st)) return rc;
  }
  return copy_outputs(E, out_u8, out_latents, out_raw_f32, st);
}

// ---- the same sampler in three segments, for per-step callbacks (stable_diffusion_pipeline.py:429-430): begin stages
// the inputs and runs the prologue, steps runs denoise steps [s0, s1) eagerly and hands the current latents out, end
// decodes.  sdw_engine_sample is begin + steps(0, n) + end under one CUDA graph.
int sdw_engine_sample_begin(sdw_engine* e, const float* latents_f32, const void* cond_f16, const void* uncond_f16,
                            void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && latents_f32 && cond_f16, "null");
  SDW_REQUIRE(!E->dry && E->n_steps > 0, "engine not bound or schedule not set");
  SDW_REQUIRE(!E->cfg.guidance || uncond_f16, "guidance needs the unconditional embedding");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const sdw_engine_config& c = E->cfg;
  if (int rc = stage_inputs(E, latents_f32, cond_f16, uncond_f16, st)) return rc;
  const int64_t per = static_cast<int64_t>(c.ctx_tokens) * c.cross_attention_dim;
  if (int rc = unet_ctx_assemble(E->cond_stage, E->uncond_stage, c.frames, c.guidance, per, E->ctx, st, E->uncond_batch > 1)) return rc;
  if (int rc = run_ops(E->prologue, st, 0)) return rc;
  return latents_init(E->lat_stage, 0, E->init_sigma, E->first_in_scale, E->x, E->model_in, c.in_channels, c.guidance,
                      c.frames, c.in_channels, c.latent_h, c.latent_w, st);
}

int sdw_engine_sample_steps(sdw_engine* e, int s0, int s1, float* out_latents, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && !E->dry && E->n_steps > 0, "engine not bound or schedule not set");
  SDW_REQUIRE(0 <= s0 && s0 <= s1 && s1 <= E->n_steps, "step range out of the schedule");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const sdw_engine_config& c = E->cfg;
  for (int s = s0; s < s1; ++s) {
    if (int rc = run_ops(E->unet_ops, st, s)) return rc;
    if (int rc = cfg_sched_step(E->eps, c.guidance, E->x, E->x_base, E->hist, &E->coefs[s], c.frames, c.in_channels,
                                c.latent_h, c.latent_w, s + 1 < E->n_steps ? E->model_in : nullptr, c.in_channels, st))
      return rc;
  }
  return copy_outputs(E, nullptr, out_latents, nullptr, st);
}

int sdw_engine_sample_end(sdw_engine* e, uint8_t* out_u8, float* out_latents, float* out_raw_f32, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && out_u8 && !E->dry, "null / engine not bound");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = run_ops(E->vae_ops, st, 0)) return rc;
  return copy_outputs(E, out_u8, out_latents, out_raw_f32, st);
}

int sdw_engine_set_uncond_batch(sdw_engine* e, int n) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && !E->dry, "engine not bound");
  SDW_REQUIRE(n == 1 || n == E->cfg.frames, "the unconditional batch is 1 (shared) or `frames` (one per frame)");
  if (n != E->uncond_batch && E->graph_exec) {  // the captured graph has the other addressing baked in
    cudaGraphExecDestroy(E->graph_exec);
    E->graph_exec = nullptr;
  }
  E->uncond_batch = n;
  return 0;
}

int sdw_engine_launches(const sdw_engine* e, int* prologue, int* unet, int* vae) {
  const Engine* E = reinterpret_cast<const Engine*>(e);
  SDW_REQUIRE(E, "null");
  if (prologue) *prologue = E->n_launch_prologue + 1;
  if (unet) *unet = E->n_launch_unet;
  if (vae) *vae = E->n_launch_vae;
  return 0;
}

// ---- debug / parity entry points -------------------------------------------------------------------
// tooling: time every op of one UNet forward (step 0) and of the VAE decode with CUDA events, after one untimed pass;
// writes "section<TAB>index<TAB>microseconds<TAB>tag" lines.  The engine must be bound and have sampled once.
int sdw_engine_debug_profile(sdw_engine* e, const char* path, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && path && !E->dry && E->n_steps > 0, "engine not bound / no schedule");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  FILE* f = std::fopen(path, "w");
  SDW_REQUIRE(f, "cannot open the profile file");
  struct Sec { const char* name; std::vector<OpFn>* ops; std::vector<std::string>* tags; };
  Sec secs[2] = {{"unet", &E->unet_ops, &E->unet_tags}, {"vae", &E->vae_ops, &E->vae_tags}};
  int rc = 0;
  for (const Sec& sc : secs) {
    if ((rc = run_ops(*sc.ops, st, 0))) break;
    const size_t n = sc.ops->size();
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& x : ev) cudaEventCreate(&x);
    cudaEventRecord(ev[0], st);
    for (size_t i = 0; i < n && !rc; ++i) {
      rc = (*sc.ops)[i](st, 0);
      cudaEventRecord(ev[i + 1], st);
    }
    cudaStreamSynchronize(st);
    for (size_t i = 0; i < n && !rc; ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      std::fprintf(f, "%s\t%zu\t%.2f\t%s\n", sc.name, i, ms * 1e3f, (*sc.tags)[i].c_str());
    }
    for (auto& x : ev) cudaEventDestroy(x);
    if (rc) break;
  }
  std::fclose(f);
  if (rc) return rc;
  SDW_CUDA_OK(cudaGetLastError());
  return 0;
}

int sdw_engine_debug_unet(sdw_engine* e, const float* x_nchw, int step, const void* ctx_f16, float* eps_nhwc_out,
                          void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && x_nchw && ctx_f16 && eps_nhwc_out, "null");
  SDW_REQUIRE(!E->dry && step >= 0 && step < E->n_steps, "engine not bound / bad step");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const sdw_engine_config& c = E->cfg;
  const int64_t per = static_cast<int64_t>(c.ctx_tokens) * c.cross_attention_dim;
  // x: [Bn][C][H][W] fp32 -> NHWC fp16 model input (no duplication, scale 1)
  SDW_CUDA_OK(cudaMemcpyAsync(E->ctx, ctx_f16, static_cast<size_t>(E->Bn) * per * 2, cudaMemcpyDeviceToDevice, st));
  // reuse hist[0..] as scratch for the fp32 state of Bn samples (hist holds 4*F*C*H*W >= Bn*C*H*W floats)
  if (int rc = latents_init(x_nchw, 0, 1.f, 1.f, E->hist, E->model_in, c.in_channels, 0, E->Bn, c.in_channels,
                            c.latent_h, c.latent_w, st))
    return rc;
  if (int rc = run_ops(E->prologue, st, 0)) return rc;
  if (int rc = run_ops(E->unet_ops, st, step)) return rc;
  SDW_CUDA_OK(cudaMemcpyAsync(eps_nhwc_out, E->eps,
                              static_cast<size_t>(E->Bn) * c.latent_h * c.latent_w * c.out_channels * 4,
                              cudaMemcpyDeviceToDevice, st));
  return 0;
}

// the two model calls of the hot loop as stand-alone entry points (SURVEY.md §8b export list): one UNet forward
// (stable_diffusion_pipeline.py:418) and one VAE decode + post-process (P:432-438)
int sdw_unet_forward(sdw_engine* e, const float* x_nchw, int step, const void* ctx_f16, float* eps_nhwc_out,
                     void* stream) {
  return sdw_engine_debug_unet(e, x_nchw, step, ctx_f16, eps_nhwc_out, stream);
}
int sdw_engine_debug_vae(sdw_engine* e, const float* latents_nchw, uint8_t* out_u8, float* out_f32_nhwc, void* stream);
int sdw_vae_decode_u8(sdw_engine* e, const float* latents_nchw, uint8_t* out_u8, float* out_f32_nhwc, void* stream) {
  return sdw_engine_debug_vae(e, latents_nchw, out_u8, out_f32_nhwc, stream);
}

int sdw_engine_debug_vae(sdw_engine* e, const float* latents_nchw, uint8_t* out_u8, float* out_f32_nhwc, void* stream) {
  Engine* E = reinterpret_cast<Engine*>(e);
  SDW_REQUIRE(E && latents_nchw && out_u8, "null");
  SDW_REQUIRE(!E->dry, "engine not bound");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const sdw_engine_config& c = E->cfg;
  const int64_t nlat = static_cast<int64_t>(c.frames) * c.in_channels * c.latent_h * c.latent_w;
  SDW_CUDA_OK(cudaMemcpyAsync(E->x, latents_nchw, nlat * 4, cudaMemcpyDeviceToDevice, st));
  if (int rc = run_ops(E->vae_ops, st, 0)) return rc;
  const size_t n = static_cast<size_t>(c.frames) * c.latent_h * c.vae_scale * c.latent_w * c.vae_scale * c.vae_out_channels;
  SDW_CUDA_OK(cudaMemcpyAsync(out_u8, E->out_u8, n, cudaMemcpyDeviceToDevice, st));
  if (out_f32_nhwc) SDW_CUDA_OK(cudaMemcpyAsync(out_f32_nhwc, E->out_img_f32, n * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // extern "C"
