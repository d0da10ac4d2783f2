// sdw_esrgan.cu — the 4x Real-ESRGAN upsampler (basicsr RRDBNet x4plus, the model behind the reference's
// RealESRGANModel, upsampling.py) as one native forward: uint8 RGB frames [n][H][W][3] -> uint8 [n][4H][4W][3].
//
//   conv_first   uint8 / 255 -> 3x3 3->64 on CUDA cores (sdw_norm.cu: conv_in_u8)
//   23 x RRDB    3 residual dense blocks each; conv1..4 (N = 32) + LeakyReLU write their channel slice of the dense
//                concat buffer [n][H][W][192] and read its channel prefix through TMA (row pitch 192); conv5 (N = 64)
//                fuses the block exit 0.2 (acc + b) + x, and on the third block the RRDB exit 0.2 (...) + x0
//   conv_body    + feat
//   2 x up       nearest x2 + 3x3 + LeakyReLU, folded to four 2x2 parity convs (pack_weight_up4)
//   conv_hr      3x3 + LeakyReLU at 4H x 4W
//   conv_last    3x3 64->3 at 4H x 4W, clamp(0, 1) * 255, round -> uint8 (sdw_norm.cu: conv_out_small, unit01)
// Every 3x3 conv in between runs on the tcgen05 implicit GEMM (sdw_gemm.cu, BLOCK_N 32 / 64).
//
// Arena (caller-owned, laid out at bind): packed weights, then feat [n][H][W][64], then one region the trunk and the
// tail share by liveness: three dense buffers D0..D2 during the trunk; U2 (4H x 4W x 64) and U3 (same, U1 = 2H x 2W x 64
// aliased on it) during the tail.  The input / output staging buffers live in the tail region too (the input is consumed
// by conv_first before the trunk starts; the outputs are written when only U3 is still live, over the dead U2).
#include "sdw_internal.h"

#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/sdwalk.h"

namespace sdw {
namespace {

__global__ void scale_f16_to_f32_kernel(const __half* __restrict__ in, float s, float* __restrict__ out, int64_t n) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __half2float(in[i]) * s;
}

struct EsrParam {
  void* dst = nullptr;
  int64_t numel = 0;
  int kind = 0;  // 0: fp32 vector (x scale), 1: 3x3 conv weight -> pack_weight, 2: raw OIHW fp16, 3: up conv -> pack_weight_up4
  int N = 0, C = 0;
  float scale = 1.f;
  bool loaded = false;
};

struct Conv {
  __half* w = nullptr;
  float* b = nullptr;
};

struct Esrgan {
  sdw_esrgan_config cfg;
  bool dry = true;
  uint8_t* base = nullptr;
  size_t used = 0, cap = 0;
  std::map<std::string, EsrParam> params;
  std::vector<std::string> order;
  Conv first, body, up1, up2, hr, last;
  std::vector<Conv> rdb;  // [block][3][5]
  __half *feat = nullptr, *D[3] = {nullptr, nullptr, nullptr}, *U1 = nullptr, *U2 = nullptr, *U3 = nullptr;
  uint8_t *in_stage = nullptr, *out_stage = nullptr;
  float* f32_stage = nullptr;
  // launch list for n frames, and its CUDA graph (key: n, pre-clamp output wanted)
  std::vector<std::function<int(cudaStream_t)>> ops;
  int ops_n = 0, ops_f32 = -1;
  cudaGraphExec_t graph = nullptr;
  int graph_n = 0, graph_f32 = -1;

  template <typename T>
  T* take(size_t n) {
    used = (used + 255) & ~size_t(255);
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + used);
    used += n * sizeof(T);
    return p;
  }
  // placement inside the shared region, relative to `r0`
  template <typename T>
  T* at(size_t r0, size_t off) {
    return dry ? nullptr : reinterpret_cast<T*>(base + r0 + off);
  }
  void reg(const std::string& name, void* dst, int64_t numel, int kind, int N = 0, int C = 0, float scale = 1.f) {
    EsrParam p;
    p.dst = dst; p.numel = numel; p.kind = kind; p.N = N; p.C = C; p.scale = scale;
    if (!params.count(name)) order.push_back(name);
    params[name] = p;
  }
  static int cp(int c) { return (c + 63) / 64 * 64; }
  // kind: 1 packed 3x3, 2 raw OIHW, 3 folded up-conv
  Conv conv(const std::string& name, int N, int C, int kind, float bias_scale = 1.f) {
    Conv cv;
    const size_t wn = kind == 1 ? static_cast<size_t>(N) * 9 * cp(C)
                                : (kind == 3 ? static_cast<size_t>(4) * N * 4 * cp(C) : static_cast<size_t>(N) * C * 9);
    cv.w = take<__half>(wn);
    cv.b = take<float>(N);
    reg(name + ".weight", cv.w, static_cast<int64_t>(N) * C * 9, kind, N, C);
    reg(name + ".bias", cv.b, N, 0, N, 0, bias_scale);
    return cv;
  }
  void layout() {
    const sdw_esrgan_config& c = cfg;
    const int nf = c.num_feat, g = c.num_grow_ch;
    used = 0;
    params.clear();
    order.clear();
    rdb.clear();
    first = conv("conv_first", nf, c.num_in_ch, 2);
    for (int i = 0; i < c.num_block; ++i)
      for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 5; ++k) {
          const std::string n = "body." + std::to_string(i) + ".rdb" + std::to_string(r + 1) + ".conv" + std::to_string(k + 1);
          // conv5's bias carries the 0.2 of the block exit 0.2 * (conv5(x) + b) + x: the epilogue computes alpha * acc + b
          rdb.push_back(k < 4 ? conv(n, g, nf + k * g, 1) : conv(n, nf, nf + 4 * g, 1, 0.2f));
        }
    body = conv("conv_body", nf, nf, 1);
    up1 = conv("conv_up1", nf, nf, 3);
    up2 = conv("conv_up2", nf, nf, 3);
    hr = conv("conv_hr", nf, nf, 1);
    last = conv("conv_last", c.num_out_ch, nf, 2);
    const size_t F = c.frames, P = static_cast<size_t>(c.height) * c.width;
    const int dc = nf + 4 * g;
    feat = take<__half>(F * P * nf);
    used = (used + 4095) & ~size_t(4095);
    const size_t r0 = used;
    auto al = [](size_t v) { return (v + 4095) & ~size_t(4095); };
    const size_t dbytes = al(F * P * dc * 2), ubytes = al(F * P * 16 * nf * 2);
    for (int i = 0; i < 3; ++i) D[i] = at<__half>(r0, i * dbytes);
    U2 = at<__half>(r0, 0);
    U3 = at<__half>(r0, ubytes);
    U1 = U3;
    // staging: input at the end of U3's range (dead until up2 writes U1 / U3); outputs inside U2 (dead once conv_hr ran)
    const size_t in_bytes = al(F * P * c.num_in_ch), out_bytes = al(F * P * 16 * c.num_out_ch);
    in_stage = at<uint8_t>(r0, 2 * ubytes - in_bytes);
    out_stage = at<uint8_t>(r0, 0);
    f32_stage = at<float>(r0, out_bytes);
    used = r0 + std::max(3 * dbytes, 2 * ubytes);
  }

  // ---- launch list ---------------------------------------------------------------------------
  int gemm(GemmDesc d) {
    GemmLaunch L;
    if (int e = plan_gemm(d, &L)) return e;
    ops.push_back([L](cudaStream_t st) { return launch_gemm(L, st); });
    return 0;
  }
  static GemmDesc conv3(const __half* A, int C, int64_t lda, int W, int H, int B, const Conv& cv, int N, __half* out,
                        int64_t ldc) {
    GemmDesc d;
    d.A = A; d.C = C; d.W = W; d.H = H; d.B = B;
    d.sW = lda; d.sH = lda * W; d.sB = lda * W * H;
    d.conv = 1; d.Wt = cv.w; d.N = N; d.bias = cv.b; d.out = out; d.ldc = ldc;
    return d;
  }
  int build_ops(int n, bool want_f32) {
    ops.clear();
    const sdw_esrgan_config& c = cfg;
    const int H = c.height, W = c.width, nf = c.num_feat, g = c.num_grow_ch, dc = nf + 4 * g;
    const int64_t P = static_cast<int64_t>(n) * H * W;
    {
      const uint8_t* in = in_stage;
      const Conv cv = first;
      __half* f = feat;
      ops.push_back([=](cudaStream_t st) { return conv_in_u8(in, n, H, W, cv.w, cv.b, nf, f, nf, st); });
      __half* d0 = D[0];
      ops.push_back([=](cudaStream_t st) {
        SDW_CUDA_OK(cudaMemcpy2DAsync(d0, dc * 2, f, nf * 2, nf * 2, P, cudaMemcpyDeviceToDevice, st));
        return 0;
      });
    }
    for (int i = 0; i < c.num_block; ++i)
      for (int r = 0; r < 3; ++r) {
        __half* src = D[r];
        __half* dst = D[(r + 1) % 3];
        for (int k = 0; k < 4; ++k) {
          GemmDesc d = conv3(src, nf + k * g, dc, W, H, n, rdb[(i * 3 + r) * 5 + k], g, src + nf + k * g, dc);
          d.act = 2;
          if (int e = gemm(d)) return e;
        }
        GemmDesc d = conv3(src, dc, dc, W, H, n, rdb[(i * 3 + r) * 5 + 4], nf, dst, dc);
        d.alpha = 0.2f;
        d.resid = src;
        d.ldr = dc;
        if (r == 2) {  // RRDB exit: 0.2 * (dense-block exit) + x0, x0 = the RRDB input still in D0 (= dst, same element)
          d.resid2 = D[0];
          d.res2_scale = 0.2f;
        }
        if (int e = gemm(d)) return e;
      }
    {  // trunk: conv_body(body) + feat -> D1[:, :64]
      GemmDesc d = conv3(D[0], nf, dc, W, H, n, body, nf, D[1], dc);
      d.resid = feat;
      d.ldr = nf;
      if (int e = gemm(d)) return e;
    }
    auto up = [&](const __half* A, int64_t lda, int w, int h, const Conv& cv, __half* out) -> int {
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
          GemmDesc d = conv3(A, nf, lda, w, h, n, cv, nf, out, nf);
          d.conv = 3; d.up_px = px; d.up_py = py;
          d.Wt = cv.w + static_cast<size_t>(py * 2 + px) * nf * 4 * cp(nf);
          d.act = 2;
          if (int e = gemm(d)) return e;
        }
      return 0;
    };
    if (int e = up(D[1], dc, W, H, up1, U1)) return e;
    if (int e = up(U1, nf, 2 * W, 2 * H, up2, U2)) return e;
    {
      GemmDesc d = conv3(U2, nf, nf, 4 * W, 4 * H, n, hr, nf, U3, nf);
      d.act = 2;
      if (int e = gemm(d)) return e;
    }
    {
      const __half* x = U3;
      const Conv cv = last;
      const int oc = c.num_out_ch;
      uint8_t* o8 = out_stage;
      float* of = want_f32 ? f32_stage : nullptr;
      ops.push_back([=](cudaStream_t st) { return conv_out_small(x, nf, n, 4 * H, 4 * W, nf, cv.w, cv.b, oc, of, o8, st, 1); });
    }
    ops_n = n;
    ops_f32 = want_f32 ? 1 : 0;
    return 0;
  }
  int run(cudaStream_t st) {
    for (auto& op : ops)
      if (int e = op(st)) return e;
    return 0;
  }
  void drop_graph() {
    if (graph) cudaGraphExecDestroy(graph);
    graph = nullptr;
    graph_n = 0;
    graph_f32 = -1;
  }
};

}  // namespace
}  // namespace sdw

using namespace sdw;

extern "C" {

int sdw_esrgan_create(const sdw_esrgan_config* cfg, sdw_esrgan** out) {
  SDW_REQUIRE(cfg && out, "null");
  SDW_REQUIRE(cfg->num_in_ch == 3 && cfg->num_out_ch == 3, "RGB in and out only (3 channels)");
  SDW_REQUIRE(cfg->scale == 4, "x4 models only (x2 / x1 RRDBNet need pixel_unshuffle)");
  SDW_REQUIRE(cfg->num_feat >= 8 && cfg->num_feat % 8 == 0 && cfg->num_grow_ch >= 8 && cfg->num_grow_ch % 8 == 0,
              "num_feat and num_grow_ch must be multiples of 8");
  SDW_REQUIRE(cfg->num_feat <= 256 && cfg->num_block >= 1, "bad RRDBNet configuration");
  // the trunk's three dense buffers must fit below the input staging at the end of the tail region (sdw_esrgan.cu: layout)
  SDW_REQUIRE(cfg->num_grow_ch <= 2 * cfg->num_feat, "num_grow_ch <= 2 * num_feat");
  SDW_REQUIRE(cfg->frames >= 1 && cfg->height >= 1 && cfg->width >= 1, "bad sizes");
  Esrgan* E = new Esrgan();
  E->cfg = *cfg;
  E->dry = true;
  E->layout();
  E->cap = E->used;
  *out = reinterpret_cast<sdw_esrgan*>(E);
  return 0;
}

void sdw_esrgan_destroy(sdw_esrgan* e) {
  Esrgan* E = reinterpret_cast<Esrgan*>(e);
  if (!E) return;
  E->drop_graph();
  delete E;
}

int sdw_esrgan_arena_bytes(const sdw_esrgan* e, uint64_t* bytes) {
  const Esrgan* E = reinterpret_cast<const Esrgan*>(e);
  SDW_REQUIRE(E && bytes, "null");
  *bytes = E->cap;
  return 0;
}

int sdw_esrgan_bind(sdw_esrgan* e, void* arena, uint64_t bytes) {
  Esrgan* E = reinterpret_cast<Esrgan*>(e);
  SDW_REQUIRE(E && arena, "null");
  SDW_REQUIRE(bytes >= E->cap, "arena too small");
  SDW_REQUIRE((reinterpret_cast<uintptr_t>(arena) & 4095) == 0, "arena must be 4096-byte aligned");
  E->drop_graph();
  E->base = static_cast<uint8_t*>(arena);
  E->dry = false;
  E->layout();
  // plan every launch now: shape / alignment errors surface at bind (also in plan-only mode, without a GPU)
  return E->build_ops(E->cfg.frames, false);
}

int sdw_esrgan_num_params(const sdw_esrgan* e) {
  const Esrgan* E = reinterpret_cast<const Esrgan*>(e);
  return E ? static_cast<int>(E->order.size()) : 0;
}

int sdw_esrgan_param_info(const sdw_esrgan* e, int index, const char** name, int64_t* numel) {
  const Esrgan* E = reinterpret_cast<const Esrgan*>(e);
  SDW_REQUIRE(E && index >= 0 && index < static_cast<int>(E->order.size()), "bad index");
  if (name) *name = E->order[index].c_str();
  if (numel) *numel = E->params.at(E->order[index]).numel;
  return 0;
}

int sdw_esrgan_load_param(sdw_esrgan* e, const char* name, const void* src_f16, int64_t numel, void* stream) {
  Esrgan* E = reinterpret_cast<Esrgan*>(e);
  SDW_REQUIRE(E && name && src_f16 && !E->dry, "null / engine not bound");
  auto it = E->params.find(name);
  SDW_REQUIRE(it != E->params.end(), "unknown Real-ESRGAN parameter");
  EsrParam& p = it->second;
  SDW_REQUIRE(numel == p.numel, "Real-ESRGAN parameter size mismatch");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __half* src = static_cast<const __half*>(src_f16);
  if (p.kind == 0) {
    scale_f16_to_f32_kernel<<<static_cast<unsigned>((numel + 255) / 256), 256, 0, st>>>(src, p.scale,
                                                                                          static_cast<float*>(p.dst), numel);
    SDW_CUDA_OK(cudaGetLastError());
  } else if (p.kind == 1) {
    if (int rc = pack_weight(src, p.N, p.C, 3, 3, 0, p.dst, st)) return rc;
  } else if (p.kind == 2) {
    SDW_CUDA_OK(cudaMemcpyAsync(p.dst, src, static_cast<size_t>(numel) * 2, cudaMemcpyDeviceToDevice, st));
  } else {
    if (int rc = pack_weight_up4(src, p.N, p.C, p.dst, st)) return rc;
  }
  p.loaded = true;
  return 0;
}

int sdw_esrgan_missing_params(const sdw_esrgan* e, const char** first_missing) {
  const Esrgan* E = reinterpret_cast<const Esrgan*>(e);
  if (!E) return -1;
  int n = 0;
  for (auto& name : E->order)
    if (!E->params.at(name).loaded) {
      if (n == 0 && first_missing) *first_missing = name.c_str();
      ++n;
    }
  return n;
}

int sdw_esrgan_forward(sdw_esrgan* e, const uint8_t* in_u8, int n, uint8_t* out_u8, float* out_f32, int use_graph,
                       void* stream) {
  Esrgan* E = reinterpret_cast<Esrgan*>(e);
  SDW_REQUIRE(E && in_u8 && out_u8 && !E->dry, "null / engine not bound");
  SDW_REQUIRE(n >= 1 && n <= E->cfg.frames, "n must be in 1..frames");
  SDW_REQUIRE(sdw_esrgan_missing_params(e, nullptr) == 0, "Real-ESRGAN parameters not loaded");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const sdw_esrgan_config& c = E->cfg;
  const size_t in_bytes = static_cast<size_t>(n) * c.height * c.width * c.num_in_ch;
  const size_t out_elems = static_cast<size_t>(n) * 16 * c.height * c.width * c.num_out_ch;
  const bool want_f32 = out_f32 != nullptr;
  if (E->ops_n != n || E->ops_f32 != (want_f32 ? 1 : 0))
    if (int rc = E->build_ops(n, want_f32)) return rc;
  SDW_CUDA_OK(cudaMemcpyAsync(E->in_stage, in_u8, in_bytes, cudaMemcpyDeviceToDevice, st));
  if (use_graph) {
    if (!E->graph || E->graph_n != n || E->graph_f32 != (want_f32 ? 1 : 0)) {
      E->drop_graph();
      cudaGraph_t graph = nullptr;
      SDW_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      const int rc = E->run(st);
      const cudaError_t ce = cudaStreamEndCapture(st, &graph);
      if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
      }
      SDW_CUDA_OK(ce);
      const cudaError_t ie = cudaGraphInstantiate(&E->graph, graph, 0);
      cudaGraphDestroy(graph);
      SDW_CUDA_OK(ie);
      E->graph_n = n;
      E->graph_f32 = want_f32 ? 1 : 0;
    }
    SDW_CUDA_OK(cudaGraphLaunch(E->graph, st));
  } else {
    if (int rc = E->run(st)) return rc;
  }
  SDW_CUDA_OK(cudaMemcpyAsync(out_u8, E->out_stage, out_elems, cudaMemcpyDeviceToDevice, st));
  if (out_f32) SDW_CUDA_OK(cudaMemcpyAsync(out_f32, E->f32_stage, out_elems * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int sdw_esrgan_launches(const sdw_esrgan* e, int* n) {
  const Esrgan* E = reinterpret_cast<const Esrgan*>(e);
  SDW_REQUIRE(E && n && !E->dry, "null / engine not bound");
  *n = static_cast<int>(E->ops.size());
  return 0;
}

}  // extern "C"
