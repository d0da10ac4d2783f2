"""StableDiffusionWalkPipeline — host-side mirror of the reference class
(stable_diffusion_videos/stable_diffusion_pipeline.py:38) whose hot path runs in libsdwalk.so.

Same method names, argument meaning and error behaviour as the reference for the path §8b of SURVEY.md lists:
`__call__` (P:192), `generate_inputs` (P:457), `make_clip_frames` (P:481), `walk` (P:556), `embed_text` (P:809),
`init_noise` (P:822), `from_pretrained(tiled=)` (P:841), plus the duck-typed attributes callers read.
What differs is WHERE the arithmetic runs: lerp/slerp, the denoise loop (UNet, CFG, scheduler step) and the VAE
decode + uint8 post-process are native sm_100a kernels behind the C ABI.  There is no diffusers dependency and no
CPU fallback: without the CUDA library this class raises.
"""
import json
import math
import time
from pathlib import Path
from types import SimpleNamespace
from typing import Callable, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _native
from .configs import UNetConfig, VAEConfig, random_state_dict, unet_param_shapes, vae_param_shapes
from .engine import Engine
from .schedulers import SCHEDULERS, PNDMScheduler


class StableDiffusionPipelineOutput(dict):
    """dict-like + attribute access, as callers index `["images"]` (P:548) or `.images`."""

    def __init__(self, images, nsfw_content_detected=None):
        super().__init__(images=images, nsfw_content_detected=nsfw_content_detected)
        self.images = images
        self.nsfw_content_detected = nsfw_content_detected


class NativeUNet:
    """Weights + config holder standing in for `UNet2DConditionModel` (attributes read at P:173, 268, 367)."""

    def __init__(self, config: UNetConfig, state_dict):
        self.cfg = config
        self.config = SimpleNamespace(sample_size=config.sample_size, in_channels=config.in_channels,
                                      attention_head_dim=config.attention_head_dim,
                                      cross_attention_dim=config.cross_attention_dim)
        self.in_channels = config.in_channels
        self.state = state_dict

    def set_attention_slice(self, slice_size):  # flash-style tiling makes slicing moot; kept for API parity
        pass


class NativeVAE:
    def __init__(self, config: VAEConfig, state_dict):
        self.cfg = config
        self.config = SimpleNamespace(block_out_channels=tuple(config.block_out_channels),
                                      latent_channels=config.latent_channels)
        self.state = state_dict


class SyntheticTokenizer:
    """Offline stand-in for CLIPTokenizer (no vocab files in this image): a prompt maps to a deterministic key."""

    model_max_length = 77

    def __call__(self, text, padding=None, max_length=None, truncation=None, return_tensors=None):
        if isinstance(text, str):
            text = [text]
        ids = torch.zeros((len(text), self.model_max_length), dtype=torch.long)
        for i, s in enumerate(text):
            if s == "":
                key = -1
            elif s.strip().lstrip("-").isdigit():
                key = int(s)
            else:
                key = sum((j + 1) * b for j, b in enumerate(s.encode())) % 1_000_000
            ids[i, 0] = key
        return SimpleNamespace(input_ids=ids)

    def batch_decode(self, ids):
        return [str(int(r[0])) for r in ids]


class SyntheticTextEncoder:
    """Synthetic prompt embeddings (BASELINE.json: "synthetic prompt embeddings"): randn([77, D]) from a CPU
    generator seeded 1000 + key, 999 for the empty prompt (SURVEY.md §8d)."""

    def __init__(self, dim=768, dtype=torch.float16, device="cpu"):
        self.dim, self.dtype, self.device = dim, dtype, torch.device(device)

    def to(self, device):
        self.device = torch.device(device)
        return self

    def __call__(self, input_ids):
        outs = []
        for row in input_ids.cpu():
            key = int(row[0])
            seed = 999 if key < 0 else 1000 + key
            g = torch.Generator(device="cpu").manual_seed(seed)
            outs.append(torch.randn((1, row.shape[0], self.dim), generator=g, dtype=torch.float32))
        return (torch.cat(outs).to(self.dtype).to(self.device),)


class _FrameSink:
    """Frame sink of a clip (SURVEY.md §8f row 1): device uint8 frames -> `frame%06d.png` files (P:550-554) without
    stalling the sampler.  Two pinned host buffers alternate: the D2H copy of batch k runs on a side stream while the
    GPU renders batch k+1, and PNG encoding runs on a worker pool (the reference encodes serially on the main thread)."""

    def __init__(self, save_path, ext, batch_shape, device, workers=8):
        from concurrent.futures import ThreadPoolExecutor

        self.save_path, self.ext = save_path, ext
        self.host = [torch.empty(batch_shape, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.events = [None, None]
        self.pending_writes = [[], []]
        self.stream = torch.cuda.Stream(device=device)
        self.pool = ThreadPoolExecutor(max_workers=workers)
        self.k = 0
        self.inflight = None  # (slot, n, first_index) whose copy has been issued but not handed to the workers
        self.bytes_d2h = 0

    def _save(self, arr, path):
        from PIL import Image

        Image.fromarray(arr).save(path)

    def _flush(self):
        if self.inflight is None:
            return
        slot, n, first = self.inflight
        self.events[slot].synchronize()
        for i in range(n):
            path = self.save_path / (f"frame%06d{self.ext}" % (first + i))
            self.pending_writes[slot].append(self.pool.submit(self._save, self.host[slot][i].numpy(), path))
        self.inflight = None

    def push(self, frames_u8, n, first_index):
        slot = self.k & 1
        for fut in self.pending_writes[slot]:  # the workers are done reading this host buffer
            fut.result()
        self.pending_writes[slot] = []
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.host[slot][:n].copy_(frames_u8[:n], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        frames_u8.record_stream(self.stream)
        self.events[slot] = ev
        self.bytes_d2h += n * frames_u8[0].numel()
        self._flush()  # the PREVIOUS batch: its copy overlapped this batch's rendering
        self.inflight = (slot, n, first_index)
        self.k += 1

    def close(self):
        self._flush()
        for slot in (0, 1):
            for fut in self.pending_writes[slot]:
                fut.result()
        self.pool.shutdown()


class StableDiffusionWalkPipeline:
    _optional_components = ["safety_checker", "feature_extractor"]

    def __init__(self, vae, text_encoder, tokenizer, unet, scheduler, safety_checker=None, feature_extractor=None,
                 requires_safety_checker: bool = True):
        if safety_checker is not None and feature_extractor is None:
            raise ValueError(  # P:122-126
                "Make sure to define a feature extractor when loading {self.__class__} if you want to use the safety"
                " checker. If you do not want to use the safety checker, you can pass `'safety_checker=None'` instead.")
        if safety_checker is not None:
            raise NotImplementedError("the native hot path has no safety checker (None in every reference test/example)")
        self.vae, self.text_encoder, self.tokenizer, self.unet = vae, text_encoder, tokenizer, unet
        self.scheduler = scheduler
        self.safety_checker, self.feature_extractor = None, feature_extractor
        self.vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1)  # P:158
        self.device = torch.device("cpu")
        self.tiled = False
        self.upsampler = None
        self._engines = {}
        self._uncond_cache = {}
        self._dist = None  # (rank, world) when frames are sharded across GPUs

    # ------------------------------------------------------------------------------------------
    # construction
    # ------------------------------------------------------------------------------------------
    @classmethod
    def from_random(cls, unet_config: UNetConfig = None, vae_config: VAEConfig = None, scheduler="pndm", seed=0,
                    device="cuda"):
        """Random-init weights of the named architecture + synthetic prompt embeddings (no network, no checkpoint)."""
        ucfg, vcfg = unet_config or UNetConfig.sd14(), vae_config or VAEConfig()
        unet = NativeUNet(ucfg, random_state_dict(unet_param_shapes(ucfg), seed))
        vae = NativeVAE(vcfg, random_state_dict(vae_param_shapes(vcfg), seed + 1))
        sch = SCHEDULERS[scheduler](prediction_type=ucfg.prediction_type) if isinstance(scheduler, str) else scheduler
        pipe = cls(vae, SyntheticTextEncoder(ucfg.cross_attention_dim), SyntheticTokenizer(), unet, sch)
        return pipe.to(device)

    @classmethod
    def from_pretrained(cls, path, *args, tiled=False, torch_dtype=None, safety_checker=None, **kwargs):
        """Load a LOCAL diffusers-layout checkpoint directory (unet/, vae/, text_encoder/, tokenizer/, scheduler/)."""
        from safetensors.torch import load_file

        root = Path(path)
        if not root.is_dir():
            raise FileNotFoundError(f"{path}: from_pretrained needs a local checkpoint directory (no network here)")

        def _cfg(sub):
            return json.loads((root / sub / "config.json").read_text())

        uc = _cfg("unet")
        ucfg = UNetConfig(in_channels=uc["in_channels"], out_channels=uc["out_channels"],
                          block_out_channels=tuple(uc["block_out_channels"]), layers_per_block=uc["layers_per_block"],
                          attention_head_dim=uc["attention_head_dim"] if isinstance(uc["attention_head_dim"], int)
                          else tuple(uc["attention_head_dim"]),
                          cross_attention_dim=uc["cross_attention_dim"], norm_num_groups=uc.get("norm_num_groups", 32),
                          norm_eps=uc.get("norm_eps", 1e-5), sample_size=uc.get("sample_size", 64),
                          use_linear_projection=uc.get("use_linear_projection", False))
        vc = _cfg("vae")
        vcfg = VAEConfig(latent_channels=vc["latent_channels"], out_channels=vc["out_channels"],
                         block_out_channels=tuple(vc["block_out_channels"]), layers_per_block=vc["layers_per_block"],
                         norm_num_groups=vc.get("norm_num_groups", 32))

        def _sd(sub):
            for fn in ("diffusion_pytorch_model.fp16.safetensors", "diffusion_pytorch_model.safetensors"):
                if (root / sub / fn).exists():
                    return load_file(str(root / sub / fn))
            raise FileNotFoundError(f"no safetensors weights under {root / sub}")

        sc = json.loads((root / "scheduler" / "scheduler_config.json").read_text())
        kinds = {"PNDMScheduler": "pndm", "DDIMScheduler": "ddim", "LMSDiscreteScheduler": "lms",
                 "EulerDiscreteScheduler": "euler", "DPMSolverMultistepScheduler": "dpm"}
        if sc["_class_name"] not in kinds:
            raise NotImplementedError(f"scheduler {sc['_class_name']} has no native plan (deterministic linear multistep "
                                      f"rules only: {sorted(kinds)}); stochastic samplers (Euler ancestral, "
                                      "DPM-Solver SDE variants) are not implemented")
        kind = kinds[sc["_class_name"]]
        # scheduler_config.json fields beyond the beta schedule: the reference itself forces steps_offset = 1 and
        # clip_sample = False on whatever the checkpoint says (P:85-110), so those are applied, not read; anything this
        # implementation cannot honour is an error, never silently ignored
        if sc.get("trained_betas") is not None:
            raise NotImplementedError("scheduler_config.json: trained_betas is not supported (scaled_linear schedule only)")
        if sc.get("set_alpha_to_one", False):
            raise NotImplementedError("scheduler_config.json: set_alpha_to_one=True is not supported (Stable Diffusion "
                                      "checkpoints ship False; the final alpha is alphas_cumprod[0])")
        if kind == "pndm" and not sc.get("skip_prk_steps", True):
            raise NotImplementedError("PNDM with Runge-Kutta warm-up steps (skip_prk_steps=False) is not supported")
        if sc.get("prediction_type", "epsilon") not in ("epsilon", "v_prediction"):
            raise NotImplementedError(f"prediction_type {sc['prediction_type']!r} is not supported")
        ucfg.prediction_type = sc.get("prediction_type", "epsilon")
        sch = SCHEDULERS[kind](num_train_timesteps=sc.get("num_train_timesteps", 1000),
                               beta_start=sc.get("beta_start", 0.00085), beta_end=sc.get("beta_end", 0.012),
                               beta_schedule=sc.get("beta_schedule", "scaled_linear"),
                               prediction_type=ucfg.prediction_type)
        from transformers import CLIPTextModel, CLIPTokenizer

        # transformers is the checkpoint READER only: the tower that runs is the native one (clip.py, sdw_clip_*)
        from .clip import NativeCLIPTextEncoder

        hf_text = CLIPTextModel.from_pretrained(str(root / "text_encoder"), torch_dtype=torch_dtype)
        text_encoder = NativeCLIPTextEncoder.from_hf_model(hf_text)
        del hf_text
        tokenizer = CLIPTokenizer.from_pretrained(str(root / "tokenizer"))
        pipe = cls(NativeVAE(vcfg, _sd("vae")), text_encoder, tokenizer, NativeUNet(ucfg, _sd("unet")), sch)
        pipe.tiled = tiled
        return pipe

    def to(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise _native.SdwError("StableDiffusionWalkPipeline (native) runs on CUDA only — there is no CPU path; "
                                   "the CPU restatement lives in oracle/ as test infrastructure")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self._uncond_cache = {}  # embeddings live on the previous device / came from the previous encoder
        if hasattr(self.text_encoder, "to"):
            self.text_encoder = self.text_encoder.to(device)
        return self

    def enable_attention_slicing(self, slice_size="auto"):  # P:161-180 — memory knob, moot here
        pass

    def disable_attention_slicing(self):  # P:182-189
        pass

    def enable_xformers_memory_efficient_attention(self, *a, **k):  # examples/make_music_video.py:22
        pass

    def set_frame_sharding(self, rank, world):
        """frames of every clip are split into contiguous per-rank blocks (SURVEY.md §8e)."""
        self._dist = (int(rank), int(world))

    # ------------------------------------------------------------------------------------------
    def _engine(self, h, w, frames, guidance):
        key = (h, w, frames, guidance, bool(self.tiled))
        eng = self._engines.get(key)
        if eng is None:
            eng = Engine(self.unet.cfg, self.vae.cfg, (h, w), frames, guidance=guidance,
                         ctx_tokens=self.tokenizer.model_max_length, device=self.device, tiled=bool(self.tiled))
            eng.load_state_dict(self.unet.state, self.vae.state)
            self._engines = {key: eng}  # one resident engine (each carries its own packed weights)
        return eng

    def _plan_key(self, num_inference_steps, guidance_scale):
        """identity of the native coefficient plan + captured graph: scheduler instance AND its configuration"""
        sc = self.scheduler.config
        return (type(self.scheduler).__name__, id(self.scheduler), sc.num_train_timesteps, sc.beta_start, sc.beta_end,
                sc.prediction_type, sc.steps_offset, int(num_inference_steps), float(guidance_scale))

    def _uncond(self, uncond_tokens):
        key = tuple(uncond_tokens)
        if key not in self._uncond_cache:  # the reference re-encodes "" every call (P:341-348); the result is constant
            ids = self.tokenizer(list(uncond_tokens), padding="max_length",
                                 max_length=self.tokenizer.model_max_length, truncation=True,
                                 return_tensors="pt").input_ids
            with torch.no_grad():
                self._uncond_cache[key] = self.text_encoder(ids.to(self.device))[0]
        return self._uncond_cache[key]

    # ------------------------------------------------------------------------------------------
    # the sampler  (reference P:191-455)
    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def __call__(self, prompt: Optional[Union[str, List[str]]] = None, height: Optional[int] = None,
                 width: Optional[int] = None, num_inference_steps: int = 50, guidance_scale: float = 7.5,
                 negative_prompt: Optional[Union[str, List[str]]] = None, num_images_per_prompt: Optional[int] = 1,
                 eta: float = 0.0, generator: Optional[torch.Generator] = None,
                 latents: Optional[torch.FloatTensor] = None, output_type: Optional[str] = "pil",
                 return_dict: bool = True, callback: Optional[Callable] = None, callback_steps: Optional[int] = 1,
                 text_embeddings: Optional[torch.FloatTensor] = None, **kwargs):
        height = height or self.unet.config.sample_size * self.vae_scale_factor
        width = width or self.unet.config.sample_size * self.vae_scale_factor
        if height % 8 != 0 or width % 8 != 0:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if (callback_steps is None) or (not isinstance(callback_steps, int) or callback_steps <= 0):
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps} of type"
                             f" {type(callback_steps)}.")
        if eta != 0.0 and not isinstance(self.scheduler, PNDMScheduler) and type(self.scheduler).__name__.startswith("DDIM"):
            raise NotImplementedError("stochastic DDIM (eta > 0) is not implemented; eta = 0 is the reference default")

        prompt_given = text_embeddings is None
        if text_embeddings is None:
            if isinstance(prompt, str):
                batch_size = 1
            elif isinstance(prompt, list):
                batch_size = len(prompt)
            else:
                raise ValueError(f"`prompt` has to be of type `str` or `list` but is {type(prompt)}")
            ids = self.tokenizer(prompt, padding="max_length", max_length=self.tokenizer.model_max_length,
                                 return_tensors="pt").input_ids
            if ids.shape[-1] > self.tokenizer.model_max_length:
                ids = ids[:, : self.tokenizer.model_max_length]
            text_embeddings = self.text_encoder(ids.to(self.device))[0]
        else:
            batch_size = text_embeddings.shape[0]
        bs_embed, seq_len, _ = text_embeddings.shape
        text_embeddings = text_embeddings.repeat(1, num_images_per_prompt, 1)
        text_embeddings = text_embeddings.view(bs_embed * num_images_per_prompt, seq_len, -1)

        do_cfg = guidance_scale > 1.0
        uncond = None
        if do_cfg:
            if negative_prompt is None:
                uncond_tokens = [""]
            elif prompt_given and type(prompt) is not type(negative_prompt):
                raise TypeError(f"`negative_prompt` should be the same type to `prompt`, but got"
                                f" {type(negative_prompt)} != {type(prompt)}.")
            elif isinstance(negative_prompt, str):
                uncond_tokens = [negative_prompt]
            elif batch_size != len(negative_prompt):
                raise ValueError(f"`negative_prompt`: {negative_prompt} has batch size {len(negative_prompt)}, but"
                                 f" `prompt`: {prompt} has batch size {batch_size}. Please make sure that passed"
                                 " `negative_prompt` matches the batch size of `prompt`.")
            else:
                uncond_tokens = negative_prompt
            uncond = self._uncond(uncond_tokens)  # [1, ...] shared, or one per prompt (P:331-336)
            if uncond.shape[0] > 1:  # P:352-355: duplicated per image of a prompt
                uncond = uncond.repeat(1, num_images_per_prompt, 1).view(uncond.shape[0] * num_images_per_prompt,
                                                                         uncond.shape[1], -1)

        B = batch_size * num_images_per_prompt
        latents_shape = (B, self.unet.in_channels, height // 8, width // 8)
        latents_dtype = text_embeddings.dtype
        if latents is None:
            latents = torch.randn(latents_shape, generator=generator, device=self.device, dtype=latents_dtype)
        else:
            if latents.shape != latents_shape:
                raise ValueError(f"Unexpected latents shape, got {latents.shape}, expected {latents_shape}")
            latents = latents.to(self.device)

        want_float = output_type != "pil"
        frames_u8, raw = self._sample_device(latents, text_embeddings, uncond, height, width, num_inference_steps,
                                             guidance_scale, want_raw=want_float, callback=callback,
                                             callback_steps=callback_steps)
        if output_type == "pil":
            from PIL import Image

            arr = frames_u8.cpu().numpy()
            image = [Image.fromarray(a) for a in arr]
        else:
            image = (raw / 2 + 0.5).clamp(0, 1).cpu().numpy()  # float32 NHWC in [0,1] (P:435-438)
        if not return_dict:
            return (image, None)
        return StableDiffusionPipelineOutput(images=image, nsfw_content_detected=None)

    def _sample_device(self, latents, text_embeddings, uncond, height, width, num_inference_steps, guidance_scale,
                       want_raw=False, callback=None, callback_steps=1):
        """native hot path: set-up (P:394-401), loop (P:412-430), decode + post-process (P:432-438, 450).
        Returns (uint8 NHWC frames on the device, pre-clamp fp32 decoder output or None)."""
        B = latents.shape[0]
        eng = self._engine(height // 8, width // 8, B, guidance_scale > 1.0)
        plan_key = self._plan_key(num_inference_steps, guidance_scale)
        if eng._plan_key != plan_key:
            eng.set_scheduler(self.scheduler, num_inference_steps, guidance_scale)
            eng._plan_key = plan_key
        res = eng.sample(latents, text_embeddings.to(self.device), uncond, use_graph=True, return_raw=want_raw,
                         callback=callback, callback_steps=callback_steps)
        return res if want_raw else (res, None)

    # ------------------------------------------------------------------------------------------
    # interpolation inputs (reference P:457-479)
    # ------------------------------------------------------------------------------------------
    def generate_inputs(self, prompt_a, prompt_b, seed_a, seed_b, noise_shape, T, batch_size):
        embeds_a = self.embed_text(prompt_a)
        embeds_b = self.embed_text(prompt_b)
        latents_dtype = embeds_a.dtype
        latents_a = self.init_noise(seed_a, noise_shape, latents_dtype)
        latents_b = self.init_noise(seed_b, noise_shape, latents_dtype)
        T = np.asarray(T, dtype=np.float64)
        n = T.shape[0]
        if n == 0:
            return
        # one batched native kernel for the whole clip instead of a per-frame device->host->device slerp (U:48-64)
        t_dev = torch.tensor(T, dtype=torch.float32, device=self.device)
        noise_all, embeds_all = _native.slerp_lerp_batch(latents_a, latents_b, embeds_a, embeds_b, t_dev)
        batch_idx = 0
        for i0 in range(0, n, batch_size):
            yield batch_idx, embeds_all[i0:i0 + batch_size], noise_all[i0:i0 + batch_size]
            batch_idx += 1

    def make_clip_frames(self, prompt_a: str, prompt_b: str, seed_a: int, seed_b: int,
                         num_interpolation_steps: int = 5, save_path: Union[str, Path] = "outputs/",
                         num_inference_steps: int = 50, guidance_scale: float = 7.5, eta: float = 0.0,
                         height: Optional[int] = None, width: Optional[int] = None, upsample: bool = False,
                         batch_size: int = 1, image_file_ext: str = ".png", T: np.ndarray = None, skip: int = 0,
                         negative_prompt: str = None, step: Optional[Tuple[int, int]] = None):
        height = height or self.unet.config.sample_size * self.vae_scale_factor
        width = width or self.unet.config.sample_size * self.vae_scale_factor
        save_path = Path(save_path)
        save_path.mkdir(parents=True, exist_ok=True)
        T = T if T is not None else np.linspace(0.0, 1.0, num_interpolation_steps)
        if T.shape[0] != num_interpolation_steps:
            raise ValueError(f"Unexpected T shape, got {T.shape}, expected dim 0 to be {num_interpolation_steps}")
        if upsample:
            if self.upsampler is None:
                raise ValueError("upsample=True needs a Real-ESRGAN upsampler: set "
                                 "`pipe.upsampler = RealESRGANModel.from_pretrained(local_path)` (a local "
                                 "RealESRGAN_x4plus.pth; nothing is downloaded)")
            if self.tiled:
                raise NotImplementedError("upsample=True with tiled=True (a circularly padded upsampler) is not "
                                          "implemented")
        if height % 8 != 0 or width % 8 != 0:  # raised by __call__ in the reference (P:271-272)
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if eta != 0.0 and type(self.scheduler).__name__.startswith("DDIM"):
            raise NotImplementedError("stochastic DDIM (eta > 0) is not implemented; eta = 0 is the reference default")
        from . import parallel

        rank, world = self._dist if self._dist is not None else (0, 1)
        Tk = T[skip:]
        lo, hi = parallel.frame_block(Tk.shape[0], world, rank)  # contiguous per-rank block of the frames still to render
        h8, w8 = height // 8, width // 8
        do_cfg = guidance_scale > 1.0
        uncond = self._uncond([negative_prompt if negative_prompt is not None else ""]) if do_cfg else None
        # decoded frame size = latent size x vae_scale_factor (the reference hard-codes // 8 for the latents, P:368)
        out_h, out_w = h8 * self.vae_scale_factor, w8 * self.vae_scale_factor
        if upsample:  # every rank upsamples its own frames on its device, before the gather and the sink
            self.upsampler.to(self.device)
            out_h, out_w = 4 * out_h, 4 * out_w
        sink = _FrameSink(save_path, image_file_ext, (batch_size, out_h, out_w, self.vae.cfg.out_channels),
                          self.device) if rank == 0 else None
        mine = []  # this rank's frames, on the device, when they have to travel to rank 0
        frame_index = skip + lo
        gen = self.generate_inputs(prompt_a, prompt_b, seed_a, seed_b, (1, self.unet.in_channels, h8, w8), Tk[lo:hi],
                                   batch_size)
        for batch_idx, embeds_batch, noise_batch in gen:
            nb = embeds_batch.shape[0]
            if nb < batch_size:  # keep ONE engine shape per walk: pad the tail batch, drop the padding
                pad = batch_size - nb
                embeds_batch = torch.cat([embeds_batch, embeds_batch[-1:].expand(pad, -1, -1)])
                noise_batch = torch.cat([noise_batch, noise_batch[-1:].expand(pad, -1, -1, -1)])
            frames_u8, _ = self._sample_device(noise_batch, embeds_batch, uncond, height, width, num_inference_steps,
                                               guidance_scale)
            if upsample:
                frames_u8 = self.upsampler.upsample_frames(frames_u8[:nb])
            if world > 1:
                mine.append(frames_u8[:nb].clone())
            else:
                sink.push(frames_u8, nb, frame_index)  # async D2H + PNG workers; the GPU goes on with the next batch
            frame_index += nb
        if world > 1:
            # decoded frames travel to rank 0 over NCCL (NVLink); rank 0 alone writes files (reference layout P:550-554)
            shape = (0, out_h, out_w, self.vae.cfg.out_channels)
            local = torch.cat(mine) if mine else torch.empty(shape, dtype=torch.uint8, device=self.device)
            allf = parallel.gather_frames(local, Tk.shape[0], dst=0)
            if rank == 0:
                for i0 in range(0, allf.shape[0], batch_size):
                    chunk = allf[i0:i0 + batch_size]
                    sink.push(chunk, chunk.shape[0], skip + i0)
        if sink is not None:
            sink.close()  # joins every write, re-raises I/O errors
        if world > 1:
            parallel.barrier()  # nobody starts the next clip (or muxes) before this clip's files exist


    # ------------------------------------------------------------------------------------------
    # walk (reference P:556-807)
    # ------------------------------------------------------------------------------------------
    def walk(self, prompts: Optional[List[str]] = None, seeds: Optional[List[int]] = None,
             num_interpolation_steps: Optional[Union[int, List[int]]] = 5, output_dir: Optional[str] = "./dreams",
             name: Optional[str] = None, image_file_ext: Optional[str] = ".png", fps: Optional[int] = 30,
             num_inference_steps: Optional[int] = 50, guidance_scale: Optional[float] = 7.5,
             eta: Optional[float] = 0.0, height: Optional[int] = None, width: Optional[int] = None,
             upsample: Optional[bool] = False, batch_size: Optional[int] = 1, resume: Optional[bool] = False,
             audio_filepath: str = None, audio_start_sec: Optional[Union[int, float]] = None,
             margin: Optional[float] = 1.0, smooth: Optional[float] = 0.0, negative_prompt: Optional[str] = None,
             make_video: Optional[bool] = True):
        height = height or self.unet.config.sample_size * self.vae_scale_factor
        width = width or self.unet.config.sample_size * self.vae_scale_factor
        # one process per GPU under torchrun: frames of every clip are sharded over the ranks (SURVEY.md §8e; the
        # reference's only multi-device precedent pads / shards / unshards inside the pipeline the same way,
        # flax_stable_diffusion_pipeline.py:546,568-578,594-597,935); rank 0 gathers the frames and is the only writer
        from . import parallel

        if self._dist is None and parallel.world_size() > 1:
            self.set_frame_sharding(parallel.rank(), parallel.world_size())
        rank, world = self._dist if self._dist is not None else (0, 1)
        output_path = Path(output_dir)
        if name is None:
            name = time.strftime("%Y%m%d-%H%M%S")
            if world > 1:
                name = parallel.broadcast_object(name)  # every rank must agree on the run directory
        save_path_root = output_path / name
        save_path_root.mkdir(parents=True, exist_ok=True)
        output_filepath = save_path_root / f"{name}.mp4"
        if not resume and isinstance(num_interpolation_steps, int):
            num_interpolation_steps = [num_interpolation_steps] * (len(prompts) - 1)
        if not resume:
            audio_start_sec = audio_start_sec or 0
        prompt_config_path = save_path_root / "prompt_config.json"
        if not resume and rank != 0:
            pass  # rank 0 writes the config
        elif not resume:
            prompt_config_path.write_text(json.dumps(dict(
                prompts=prompts, seeds=seeds, num_interpolation_steps=num_interpolation_steps, fps=fps,
                num_inference_steps=num_inference_steps, guidance_scale=guidance_scale, eta=eta, upsample=upsample,
                height=height, width=width, audio_filepath=audio_filepath, audio_start_sec=audio_start_sec,
                negative_prompt=negative_prompt), indent=2, sort_keys=False))
        else:
            data = json.load(open(prompt_config_path))
            prompts, seeds = data["prompts"], data["seeds"]
            num_interpolation_steps, fps = data["num_interpolation_steps"], data["fps"]
            num_inference_steps, guidance_scale, eta = data["num_inference_steps"], data["guidance_scale"], data["eta"]
            upsample, height, width = data["upsample"], data["height"], data["width"]
            audio_filepath, audio_start_sec = data["audio_filepath"], data["audio_start_sec"]
            negative_prompt = data.get("negative_prompt", None)

        for i, (prompt_a, prompt_b, seed_a, seed_b, num_step) in enumerate(
                zip(prompts, prompts[1:], seeds, seeds[1:], num_interpolation_steps)):
            save_path = save_path_root / f"{name}_{i:06d}"
            step_output_filepath = save_path / f"{name}_{i:06d}.mp4"
            skip = 0
            if world > 1:
                parallel.barrier()  # rank 0's file operations of the previous clip are visible before anyone globs
            if resume:
                if step_output_filepath.exists():
                    print(f"Skipping {save_path} because frames already exist")
                    continue
                existing_frames = sorted(save_path.glob(f"*{image_file_ext}"))
                if existing_frames:
                    skip = int(existing_frames[-1].stem[-6:]) + 1
                    if skip + 1 >= num_step:
                        print(f"Skipping {save_path} because frames already exist")
                        continue
                    print(f"Resuming {save_path.name} from frame {skip}")
            audio_offset = audio_start_sec + sum(num_interpolation_steps[:i]) / fps
            audio_duration = num_step / fps
            T = None
            if audio_filepath:
                from .utils import get_timesteps_arr

                T = get_timesteps_arr(audio_filepath, offset=audio_offset, duration=audio_duration, fps=fps,
                                      margin=margin, smooth=smooth)
            self.make_clip_frames(prompt_a, prompt_b, seed_a, seed_b, num_interpolation_steps=num_step,
                                  save_path=save_path, num_inference_steps=num_inference_steps,
                                  guidance_scale=guidance_scale, eta=eta, height=height, width=width,
                                  upsample=upsample, batch_size=batch_size, T=T, skip=skip,
                                  negative_prompt=negative_prompt, step=(i, len(prompts) - 1))
            if make_video and rank == 0:
                from .utils import make_video_pyav

                make_video_pyav(save_path, audio_filepath=audio_filepath, fps=fps,
                                output_filepath=step_output_filepath, glob_pattern=f"*{image_file_ext}",
                                audio_offset=audio_offset, audio_duration=audio_duration, sr=44100)
        if world > 1:
            parallel.barrier()
        if make_video and rank == 0:
            from .utils import make_video_pyav

            return make_video_pyav(save_path_root, audio_filepath=audio_filepath, fps=fps,
                                   audio_offset=audio_start_sec, audio_duration=sum(num_interpolation_steps) / fps,
                                   output_filepath=output_filepath, glob_pattern=f"**/*{image_file_ext}", sr=44100)

    # ------------------------------------------------------------------------------------------
    def embed_text(self, text, negative_prompt=None):
        """Helper to embed some text (reference P:809-820)."""
        text_input = self.tokenizer(text, padding="max_length", max_length=self.tokenizer.model_max_length,
                                    truncation=True, return_tensors="pt")
        with torch.no_grad():
            embed = self.text_encoder(text_input.input_ids.to(self.device))[0]
        return embed

    def init_noise(self, seed, noise_shape, dtype):
        """Helper to initialize noise (reference P:822-838): seeded torch.randn ON the pipeline device."""
        return torch.randn(noise_shape, device=self.device,
                           generator=torch.Generator(device=self.device).manual_seed(seed), dtype=dtype)
