/* sdwalk.h — C ABI of libsdwalk.so, the Blackwell-native (sm_100a) implementation of the
 * latent-walk hot path of nateraw/stable-diffusion-videos.
 *
 * The reference has no FFI: its hot path sits behind the Python class
 * StableDiffusionWalkPipeline (stable_diffusion_videos/stable_diffusion_pipeline.py:38).
 * This header is the boundary a maintainer binds with ctypes (see INTEGRATION.md); every entry
 * point cites the reference lines it replaces.
 *
 * Conventions
 *   - every function returns int: 0 = ok, 1 = invalid argument, 2 = CUDA/driver failure,
 *     3 = not initialised / wrong state. sdw_last_error() returns a thread-local message.
 *   - all buffers are caller-owned DEVICE pointers (torch tensors' data_ptr()), sizes explicit.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream).
 *   - no entry point synchronises the device or allocates device memory, except
 *     sdw_engine_create (records sizes only) — the arena is supplied by the caller.
 *   - one engine per (process, device); an engine is not thread-safe (mirrors the reference:
 *     mutable scheduler state, stable_diffusion_pipeline.py:394).
 */
#ifndef SDWALK_H_
#define SDWALK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDW_ABI_VERSION 2

const char* sdw_last_error(void);
int sdw_abi_version(void);
/* tooling: validate launch plans (shapes, TMA alignment) without a CUDA driver; nothing can be launched while on */
void sdw_debug_plan_only(int on);

/* ------------------------------------------------------------------------------------------
 * Interpolation inputs — replaces generate_inputs' per-frame torch.lerp + numpy slerp
 * (stable_diffusion_pipeline.py:466-468, utils.py:42-66) with one batched fp32 kernel.
 *   lat_a, lat_b : [n_lat] fp16 or fp32 (dtype_is_f16) keyframe latents
 *   emb_a, emb_b : [n_emb] same dtype, keyframe text embeddings
 *   t            : [n_frames] fp32 interpolation weights on device
 *   out_lat      : [n_frames][n_lat], out_emb : [n_frames][n_emb], same dtype
 *   dot_threshold: 0.9995 in the reference (utils.py:42)
 * ---------------------------------------------------------------------------------------- */
int sdw_slerp_lerp_batch(const void* lat_a, const void* lat_b, const void* emb_a, const void* emb_b,
                         const float* t, int n_frames, int64_t n_lat, int64_t n_emb, int dtype_is_f16,
                         float dot_threshold, void* out_lat, void* out_emb, void* stream);

/* ------------------------------------------------------------------------------------------
 * Classifier-free guidance + scheduler update — replaces stable_diffusion_pipeline.py:421-426
 * (noise_pred chunk/combine and scheduler.step) and :414-415 (cat + scale_model_input) for
 * every linear-multistep scheduler the reference accepts (PNDM/PLMS, DDIM, LMS).
 *   eps_nhwc  : [2F][H][W][C] fp32 UNet output, first F = unconditional, last F = conditional
 *               (or [F] when guidance is off: has_uncond = 0)
 *   x         : [F][C][H][W] fp32 latents (updated in place)
 *   x_base    : [F][C][H][W] fp32 PLMS `cur_sample` slot
 *   hist      : [4][F][C][H][W] fp32 ring of previous combined eps, hist_slot[k] picks the slot
 *   coef      : see sdw_step_coef
 *   next_in   : [2F or F][H][W][Cpad] fp16 NHWC model input for the NEXT step (x * next_in_scale, duplicated
 *               for the uncond/cond halves); may be null on the last step
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_step_coef {
  float guidance;      /* g in u + g (c - u) */
  float c_x;           /* coefficient on the sample */
  float c_e[5];        /* coefficients on {current eps, hist[slot0], hist[slot1], hist[slot2], hist[slot3]} */
  int32_t hist_slot[4];
  int32_t use_x_base;  /* 1: sample := x_base (PLMS second step) */
  int32_t save_x_base; /* 1: x_base := sample before the update (PLMS first step) */
  int32_t push_slot;   /* >=0: store push_e * e + push_x * s into hist[push_slot] */
  float next_in_scale; /* scale_model_input factor for the next UNet call */
  float push_e, push_x; /* what the history keeps: (1, 0) = the combined eps (PLMS / LMS); DPM-Solver++ keeps the data
                         * prediction x0 = s / alpha_t - (sigma_t / alpha_t) e */
} sdw_step_coef;
/* update: e = u + g (c - u);  s = use_x_base ? x_base : x;  x' = c_x s + c_e[0] e + sum_j c_e[1+j] hist[hist_slot[j]];
 * covers PNDM/PLMS (warm-up, cur_sample step, 4-term Adams-Bashforth), DDIM eps / v-prediction (eta = 0), LMS, Euler
 * and DPM-Solver++(2M) (history of x0) exactly; coefficients are computed on the host in fp64 (see schedulers.py). */

int sdw_cfg_sched_step(const void* eps_nhwc, int has_uncond, float* x, float* x_base, float* hist,
                       const sdw_step_coef* coef, int F, int C, int H, int W, void* next_in, int next_in_cpad,
                       void* stream);

/* latents [F][C][H][W] (fp16/fp32) -> fp32 state * sigma and the first NHWC fp16 model input */
int sdw_latents_init(const void* latents, int dtype_is_f16, float init_noise_sigma, float in_scale, float* x,
                     void* model_in, int model_in_cpad, int dup, int F, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------
 * Engine: the whole per-frame sampler (stable_diffusion_pipeline.py:412-438, 450) for `frames` frames per call.
 * Life cycle: create(cfg) -> arena_bytes -> bind(arena) -> load_param xN -> set_schedule -> sample xN -> destroy.
 * Parameter names are the diffusers state-dict keys of the UNet; VAE decoder keys carry a "vae." prefix
 * ("vae.decoder.conv_in.weight", "vae.post_quant_conv.weight", attention as to_q/to_k/to_v/to_out.0).
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_engine sdw_engine;

typedef struct sdw_engine_config {
  /* UNet2DConditionModel (config.json of the checkpoint) */
  int32_t in_channels, out_channels;
  int32_t num_levels;
  int32_t block_out_channels[4];
  int32_t layers_per_block;
  int32_t attention_heads[4];      /* diffusers' `attention_head_dim` = NUMBER of heads per level */
  int32_t cross_attention_dim, ctx_tokens;
  int32_t norm_num_groups;
  float norm_eps;
  /* AutoencoderKL decoder */
  int32_t vae_num_levels;
  int32_t vae_block_out_channels[4];
  int32_t vae_layers_per_block;
  int32_t vae_norm_num_groups;
  int32_t vae_out_channels;
  int32_t vae_scale;               /* 2^(vae_num_levels-1) = pipeline.vae_scale_factor */
  float vae_scaling_factor;        /* 0.18215, hard-coded at stable_diffusion_pipeline.py:432 */
  /* problem */
  int32_t latent_h, latent_w;
  int32_t frames;                  /* frames per sample call (the reference's batch_size) */
  int32_t guidance;                /* 1: classifier-free guidance -> UNet batch 2*frames (P:414) */
  int32_t max_steps;
  int32_t tiled;                   /* 1: every 3x3 conv pads circularly (from_pretrained(tiled=True), P:841-858) */
} sdw_engine_config;

int sdw_engine_create(const sdw_engine_config* cfg, sdw_engine** out);
void sdw_engine_destroy(sdw_engine* e);
int sdw_engine_arena_bytes(const sdw_engine* e, uint64_t* bytes);
int sdw_engine_bind(sdw_engine* e, void* arena, uint64_t bytes);
int sdw_engine_num_params(const sdw_engine* e);
int sdw_engine_param_info(const sdw_engine* e, int index, const char** name, int64_t* numel);
/* src: fp16 device tensor in the checkpoint's own layout (OIHW conv / [out,in] linear / vectors) */
int sdw_engine_load_param(sdw_engine* e, const char* name, const void* src_f16, int64_t numel, void* stream);
int sdw_engine_missing_params(const sdw_engine* e, const char** first_missing);
/* timesteps: host fp32 [n_steps]; coefs: host [n_steps] */
int sdw_engine_set_schedule(sdw_engine* e, int n_steps, const float* timesteps, const sdw_step_coef* coefs,
                            float init_noise_sigma, float first_in_scale, void* stream);
/* latents fp32 [F][4][h][w] (already interpolated, unscaled), cond fp16 [F][tokens][D], uncond fp16 [1][tokens][D]
 * -> out_u8 [F][8h][8w][3] uint8 NHWC; out_latents (optional) fp32 [F][4][h][w] final latents. */
int sdw_engine_sample(sdw_engine* e, const float* latents_f32, const void* cond_f16, const void* uncond_f16,
                      uint8_t* out_u8, float* out_latents, float* out_raw_f32, int use_graph, void* stream);
/* use_graph = 1 captures the whole call into a CUDA graph on first use: `stream` must then be a real stream, not
 * the legacy default stream 0.  out_raw_f32 (optional): fp32 [F][8h][8w][3] decoder output BEFORE (x/2+0.5).clamp(0,1) — the float image of P:435 */
/* per-sample negative prompts (P:318-358 with a list `negative_prompt`): n = frames makes `uncond_f16` of the sample calls
 * a [frames][tokens][D] batch, n = 1 (default) one embedding shared by all frames */
int sdw_engine_set_uncond_batch(sdw_engine* e, int n);
int sdw_engine_launches(const sdw_engine* e, int* prologue, int* unet_per_step, int* vae);
/* The same sampler in three segments, for per-step callbacks (stable_diffusion_pipeline.py:429-430): `begin` stages the
 * inputs and runs the prologue (context assembly, cross-attention K/V, first model input); `steps` runs denoise steps
 * [s0, s1) eagerly and copies the current latents (fp32 [F][4][h][w]) to out_latents when non-null; `end` decodes.
 * sdw_engine_sample == begin + steps(0, n_steps) + end under one CUDA graph. */
int sdw_engine_sample_begin(sdw_engine* e, const float* latents_f32, const void* cond_f16, const void* uncond_f16,
                            void* stream);
int sdw_engine_sample_steps(sdw_engine* e, int s0, int s1, float* out_latents, void* stream);
int sdw_engine_sample_end(sdw_engine* e, uint8_t* out_u8, float* out_latents, float* out_raw_f32, void* stream);
/* the two model calls of the hot loop as stand-alone entry points: one UNet forward on an explicit [Bn] batch (Bn = 2F with
 * guidance: x fp32 [Bn][4][h][w], ctx fp16 [Bn][tokens][D] -> eps fp32 NHWC [Bn][h][w][4]; reference P:418) and one VAE
 * decode + post-process of fp32 [F][4][h][w] latents (division by the scaling factor inside) -> uint8 NHWC frames and,
 * optionally, the pre-clamp fp32 decoder output (reference P:432-438) */
int sdw_unet_forward(sdw_engine* e, const float* x_nchw, int step, const void* ctx_f16, float* eps_nhwc_out, void* stream);
int sdw_vae_decode_u8(sdw_engine* e, const float* latents_nchw, uint8_t* out_u8, float* out_f32_nhwc, void* stream);
/* parity hooks: one UNet forward on an explicit [Bn] batch / one VAE decode */
int sdw_engine_debug_unet(sdw_engine* e, const float* x_nchw, int step, const void* ctx_f16, float* eps_nhwc_out,
                          void* stream);
int sdw_engine_debug_vae(sdw_engine* e, const float* latents_nchw, uint8_t* out_u8, float* out_f32_nhwc, void* stream);
/* tooling: CUDA-event time of every op of one UNet forward and of the VAE decode, written as TSV to `path` */
int sdw_engine_debug_profile(sdw_engine* e, const char* path, void* stream);

/* ------------------------------------------------------------------------------------------
 * Low-level tensor-core op (tests / tooling): one implicit GEMM on the tcgen05 kernel.
 * Covers Conv2d 3x3 (stride 1/2, nearest-up x2 fused), 1x1, Linear and batched matmul.
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_gemm_desc {
  const void* A;             /* fp16 NHWC lattice base */
  int32_t C, W, H, B;
  int64_t sW, sH, sB;        /* element strides */
  int32_t conv;              /* 0: 1x1; 1: 3x3 s1 p1; 2: 3x3 s2 p1; 3: nearest-up2 + 3x3 for one output parity,
                                folded to a 2x2 conv (Wt = the parity's sdw_pack_weight_up4 block) */
  int32_t up_px, up_py;
  const void* Wt;            /* fp16 [N][taps*Cp] K-major, Cp = ceil64(C) */
  int32_t N;
  int64_t ldb, Kb;
  int32_t b_batched;
  int64_t sBh, sBb;
  const float* bias;
  const float* rowvec;
  int32_t rowvec_ld;
  const void* resid;
  int64_t ldr;
  void* out;
  int64_t ldc;
  int64_t o_sW, o_sH, o_sB;
  int32_t mode;              /* 0 plain, 1 GEGLU, 2 QKV with V^T scatter */
  int32_t act;               /* 0 none, 1 SiLU, 2 LeakyReLU(0.2) (applied after bias, before the residual) */
  float alpha;
  int32_t vt_col0, vt_d, vt_heads, vt_ntok;
  void* vt;
  int64_t vt_ld;
  int32_t bn;                /* BLOCK_N: 0 auto, 32/64/128/160/256 (32 and 64: one-CTA kernel only) */
  int32_t ver;               /* 0 auto, 1: one CTA per 128xBN tile, 2: persistent CTA pairs (256xBN) */
  int32_t nsub;              /* 0 auto, 1 / 2: accumulators per activation tile in the CTA-pair kernel */
  int32_t ew;                /* 0 auto, 2 / 4: epilogue warps per TMEM lane quarter of the CTA-pair kernel (4: needs the TMA epilogue) */
  int32_t tr;                /* 0 auto, 1 never, 2 require: 3x3 taps reuse one activation box in shared memory */
  int32_t et;                /* 0 auto, 1 never, 2 require: TMA-store epilogue with a TMA-fed residual ring.  With mode 2 the
                              * V^T rows are written through TMA, which clips the token extent at 16-byte granularity: the
                              * vt_ld padding up to the next multiple of 8 tokens may receive finite filler values */
  int32_t reserved0;         /* must be 0 */
} sdw_gemm_desc;

int sdw_gemm(const sdw_gemm_desc* desc, void* stream);
/* the same GEMM with a second, scaled residual on the first residual's strides (plain mode, `resid` set):
 * out = res2_scale * (epilogue result including resid) + resid2 — Real-ESRGAN's RRDB exit 0.2 * (0.2 * (acc + b) + x) + x0 */
int sdw_gemm_res2(const sdw_gemm_desc* desc, const void* resid2, float res2_scale, void* stream);
/* planner introspection, host only (also in plan-only mode): out = {kernel version, BLOCK_N, accumulators, epilogue warps
 * per lane quarter, tap reuse, TMA epilogue, pipeline stages, 0, grid size, tile w, tile h, tile b} */
int sdw_debug_plan(const sdw_gemm_desc* desc, int32_t out[12]);

/* fused attention on tcgen05 (tests / tooling): O = softmax(Q K^T d^-1/2) V per (batch, head).
 * q [B][Nq][q_ld], k [B][Nk][k_ld] with head h at columns h*d; vt [B][heads][d][vt_ld] = V transposed;
 * out [B][Nq][out_ld]; all fp16; d a multiple of 8 in 8..160. */
int sdw_attention(const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* vt, int64_t vt_ld, int B,
                  int Nq, int Nk, int heads, int d, void* out, int64_t out_ld, void* stream);

/* normalisation layers (tests / tooling).  x, y: fp16 [B][P][ld] NHWC views (ld = channel pitch, multiple of 8);
 * GroupNorm over (P pixels x C/G channels) per sample with optional SiLU; LayerNorm over the C channels of each row.
 * gamma / beta fp32 [C]. */
int sdw_groupnorm(const void* x, int64_t ldx, int B, int64_t P, int C, int G, const float* gamma, const float* beta,
                  float eps, int silu, void* y, int64_t ldy, void* stream);
int sdw_layernorm(const void* x, int64_t ldx, int64_t rows, int C, const float* gamma, const float* beta, float eps,
                  void* y, int64_t ldy, void* stream);

/* attention planner introspection, host only: out = {kernel variant, query tiles per CTA, grid x, y, z} */
int sdw_debug_attention_plan(int B, int Nq, int Nk, int heads, int d, int32_t out[5]);
/* tooling: device buffer of 2 x 4096 x 8 int64 that CTA 0 of the two-tile attention kernel fills with clock64 stamps per
 * KV tile (wait start, S ready, row in registers, max done, MUFU token held, burst issued, P stored) for query tiles A and B; NULL switches it off */
void sdw_debug_attention_trace(void* buf);

/* pack an OIHW fp16 conv / [N][K] linear weight into the kernel's K-major [N][taps][Cp] layout */
int sdw_pack_weight(const void* w_oihw, int N, int C, int kh, int kw, int geglu_interleave, void* out, void* stream);
/* upsampler (nearest x2 + 3x3) weights folded to four 2x2 parity convs: out = 4 blocks of [N][4][ceil64(C)];
 * block (py*2+px) is the weight operand of a conv = 3 GEMM with up_py/up_px = (py, px) */
int sdw_pack_weight_up4(const void* w_oihw, int N, int C, void* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * CLIP text tower: replaces `self.text_encoder(input_ids)[0]` of embed_text (stable_diffusion_pipeline.py:809-820) and of
 * the unconditional "" encode (P:341-348).  Parameter names are transformers' CLIPTextModel state-dict keys
 * ("text_model.embeddings.token_embedding.weight", "text_model.encoder.layers.{i}.self_attn.q_proj.weight", ...,
 * "text_model.final_layer_norm.bias"); all tensors are handed over as fp16.  Life cycle as the sampler engine:
 * create -> arena_bytes -> bind(arena: caller-owned device memory, 256-byte aligned) -> load_param x N -> forward x M.
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_clip sdw_clip;
typedef struct sdw_clip_config {
  int32_t vocab, max_positions, hidden, layers, heads, intermediate;
  int32_t act_gelu_erf; /* 0: quick-GELU x sigmoid(1.702 x) (SD-1.x ViT-L/14); 1: erf GELU (SD-2.x OpenCLIP-H) */
  float eps;            /* LayerNorm epsilon (1e-5) */
  int32_t max_batch;    /* prompts per forward call the activation buffers are sized for */
} sdw_clip_config;
int sdw_clip_create(const sdw_clip_config* cfg, sdw_clip** out);
void sdw_clip_destroy(sdw_clip* e);
int sdw_clip_arena_bytes(const sdw_clip* e, uint64_t* bytes);
int sdw_clip_bind(sdw_clip* e, void* arena, uint64_t bytes);
int sdw_clip_num_params(const sdw_clip* e);
int sdw_clip_param_info(const sdw_clip* e, int index, const char** name, int64_t* numel);
int sdw_clip_load_param(sdw_clip* e, const char* name, const void* data_f16, int64_t numel, void* stream);
int sdw_clip_missing_params(const sdw_clip* e, const char** first_missing);
/* ids: device int32 [B][max_positions] (token ids, already padded / truncated by the tokenizer);
 * out: device fp16 [B][max_positions][hidden] = last_hidden_state after the final LayerNorm */
int sdw_clip_forward(sdw_clip* e, const int32_t* ids, int B, void* out_f16, void* stream);

/* ------------------------------------------------------------------------------------------
 * Real-ESRGAN 4x upsampler: replaces RealESRGANModel.forward (upsampling.py:30-55; basicsr RRDBNet x4plus under
 * RealESRGANer.enhance with tile = 0, pre_pad = 0, outscale = 4) for `frames` frames per call.  Parameter names are
 * basicsr's RRDBNet state-dict keys ("conv_first.weight", "body.{i}.rdb{1,2,3}.conv{1..5}.weight", "conv_body.*",
 * "conv_up1.*", "conv_up2.*", "conv_hr.*", "conv_last.*"), handed over as fp16 in their own (OIHW / vector) layout.
 * Life cycle as the CLIP tower: create -> arena_bytes -> bind(arena: caller-owned device memory, 4096-byte aligned; all
 * launches are planned here) -> load_param x N -> forward x M -> destroy.
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_esrgan sdw_esrgan;
typedef struct sdw_esrgan_config {
  int32_t num_in_ch, num_out_ch;  /* 3, 3 */
  int32_t num_feat, num_block, num_grow_ch;  /* 64, 23, 32 for RealESRGAN_x4plus */
  int32_t scale;                  /* 4 only */
  int32_t height, width;          /* input frame size */
  int32_t frames;                 /* frames per forward call the activation buffers are sized for */
} sdw_esrgan_config;
int sdw_esrgan_create(const sdw_esrgan_config* cfg, sdw_esrgan** out);
void sdw_esrgan_destroy(sdw_esrgan* e);
int sdw_esrgan_arena_bytes(const sdw_esrgan* e, uint64_t* bytes);
int sdw_esrgan_bind(sdw_esrgan* e, void* arena, uint64_t bytes);
int sdw_esrgan_num_params(const sdw_esrgan* e);
int sdw_esrgan_param_info(const sdw_esrgan* e, int index, const char** name, int64_t* numel);
int sdw_esrgan_load_param(sdw_esrgan* e, const char* name, const void* src_f16, int64_t numel, void* stream);
int sdw_esrgan_missing_params(const sdw_esrgan* e, const char** first_missing);
/* in_u8 [n][H][W][3] RGB (n <= frames) -> out_u8 [n][4H][4W][3] = round(clamp(model(in / 255), 0, 1) * 255);
 * out_f32 (optional): fp32 [n][4H][4W][3] model output before the clamp.  use_graph = 1 replays the whole forward as one
 * CUDA graph (captured on first use per n; `stream` must then be a real stream, not the legacy default stream 0). */
int sdw_esrgan_forward(sdw_esrgan* e, const uint8_t* in_u8, int n, uint8_t* out_u8, float* out_f32, int use_graph,
                       void* stream);
/* number of kernel launches (and copies) of one forward, as planned at bind */
int sdw_esrgan_launches(const sdw_esrgan* e, int* n);

/* ------------------------------------------------------------------------------------------
 * Frame-sharded walk over the GPUs of one box (one process per GPU): the three exchanges of the path, as thin NCCL
 * wrappers (NCCL bound at run time with dlopen; no collective exists inside the sampler — frames are independent).
 * Replaces what the reference's Flax twin does with replicate / shard / unshard
 * (flax_stable_diffusion_pipeline.py:546, 568-578, 594-597, 898-902, 935).
 *   rank 0: sdw_nccl_unique_id(id) -> the 128 bytes travel to every rank by the host's own means (torch.distributed
 *   object broadcast in parallel.py) -> every rank: sdw_nccl_init(id, rank, world) with its CUDA device current.
 * ---------------------------------------------------------------------------------------- */
typedef struct sdw_comm sdw_comm;
int sdw_nccl_unique_id(void* id128);
int sdw_nccl_init(const void* id128, int rank, int world, sdw_comm** out);
void sdw_nccl_destroy(sdw_comm* c);
/* in place: `root`'s bytes reach every rank (the flat fp16 weight buffer, once per pipeline) */
int sdw_nccl_broadcast_weights(sdw_comm* c, void* buf, uint64_t bytes, int root, void* stream);
/* every rank sends `bytes_per_rank` bytes (its padded uint8 frame block); `root` receives [world][bytes_per_rank] in
 * `recv` (ignored elsewhere): one grouped ncclSend / ncclRecv round over NVLink */
int sdw_nccl_gather_frames(sdw_comm* c, const void* send, void* recv, uint64_t bytes_per_rank, int root, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDWALK_H_ */
