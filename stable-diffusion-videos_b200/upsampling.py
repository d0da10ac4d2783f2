"""Native 4x Real-ESRGAN upsampler (sdw_esrgan_* in include/sdwalk.h) behind the reference's `RealESRGANModel`
(upsampling.py): basicsr's RRDBNet x4plus under `RealESRGANer.enhance` with tile = 0, pre_pad = 0, outscale = 4, in fp16
storage with fp32 accumulation on sm_100a.  Weights come from a local `RealESRGAN_x4plus.pth` (`from_pretrained`) or a
seeded random init (`from_random`); nothing is downloaded and nothing runs on the CPU.
"""
import ctypes as C
import logging
from pathlib import Path

import numpy as np
import torch

from . import _native as N
from .configs import ESRGANConfig, esrgan_param_shapes, esrgan_random_state_dict

logger = logging.getLogger(__name__)


class ESRGANEngineConfig(C.Structure):
    _fields_ = [("num_in_ch", C.c_int32), ("num_out_ch", C.c_int32), ("num_feat", C.c_int32),
                ("num_block", C.c_int32), ("num_grow_ch", C.c_int32), ("scale", C.c_int32),
                ("height", C.c_int32), ("width", C.c_int32), ("frames", C.c_int32)]


class ESRGANEngine:
    """One native RRDBNet forward for a fixed input size and up to `frames` frames per call (its own arena)."""

    def __init__(self, cfg: ESRGANConfig, height, width, frames, device):
        self.cfg, self.height, self.width, self.frames = cfg, int(height), int(width), int(frames)
        self.device = torch.device(device)
        lib = N.lib()
        lib.sdw_esrgan_destroy.restype = None
        c = ESRGANEngineConfig(cfg.num_in_ch, cfg.num_out_ch, cfg.num_feat, cfg.num_block, cfg.num_grow_ch, cfg.scale,
                               self.height, self.width, self.frames)
        self._h = C.c_void_p()
        N.check(lib.sdw_esrgan_create(C.byref(c), C.byref(self._h)))
        nbytes = C.c_uint64()
        N.check(lib.sdw_esrgan_arena_bytes(self._h, C.byref(nbytes)))
        self.arena_bytes = int(nbytes.value)
        with torch.cuda.device(self.device):
            self.arena = torch.empty(self.arena_bytes + 4096, dtype=torch.uint8, device=self.device)
            base = (self.arena.data_ptr() + 4095) // 4096 * 4096
            N.check(lib.sdw_esrgan_bind(self._h, C.c_void_p(base), C.c_uint64(self.arena_bytes)))
            self.stream = torch.cuda.Stream(device=self.device)  # graph capture needs a real stream

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                N.lib().sdw_esrgan_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def load_state_dict(self, sd):
        lib = N.lib()
        want = esrgan_param_shapes(self.cfg)
        unexpected = sorted(set(sd) - set(want))
        if unexpected:
            raise N.SdwError(f"unexpected Real-ESRGAN parameter {unexpected[0]} (RRDBNet x{self.cfg.scale} keys expected)")
        keep = []
        with torch.cuda.device(self.device):
            for name, t in sd.items():
                if tuple(t.shape) != tuple(want[name]):
                    raise N.SdwError(f"shape mismatch for {name}: {tuple(t.shape)}, expected {want[name]}")
                th = t.detach().to(device=self.device, dtype=torch.float16).contiguous()
                keep.append(th)
                N.check(lib.sdw_esrgan_load_param(self._h, name.encode(), N.ptr(th), C.c_int64(th.numel()),
                                                  N.stream_ptr()))
            torch.cuda.current_stream().synchronize()
        first = C.c_char_p()
        missing = lib.sdw_esrgan_missing_params(self._h, C.byref(first))
        if missing:
            raise N.SdwError(f"{missing} Real-ESRGAN parameters not loaded (first: {first.value.decode()})")

    def forward(self, frames_u8, out=None, out_f32=None, use_graph=True):
        """frames_u8: CUDA uint8 [n, H, W, 3], n <= frames -> uint8 [n, 4H, 4W, 3] (and the fp32 pre-clamp output into
        `out_f32` when given)."""
        n = frames_u8.shape[0]
        s = self.cfg.scale
        if out is None:
            out = torch.empty((n, s * self.height, s * self.width, self.cfg.num_out_ch), dtype=torch.uint8,
                              device=self.device)
        x = frames_u8.contiguous()
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            N.check(N.lib().sdw_esrgan_forward(self._h, N.ptr(x), C.c_int(n), N.ptr(out), N.ptr(out_f32),
                                               C.c_int(int(use_graph)), C.c_void_p(self.stream.cuda_stream)))
        cur.wait_stream(self.stream)
        for t in (x, out, out_f32):
            if t is not None:
                t.record_stream(self.stream)
        return out


class RealESRGANModel:
    """The reference's `RealESRGANModel(model_path, tile=0, tile_pad=10, pre_pad=0, fp32=False)`, natively.

    `model(image)` upsamples one float RGB array in [0, 1] (or an image path) as the reference does; `model(frames)` with
    a CUDA uint8 tensor [n, H, W, 3] is the batched device path the walk uses (uint8 [n, 4H, 4W, 3] out, on the device).
    """

    def __init__(self, model_path=None, tile=0, tile_pad=10, pre_pad=0, fp32=False, state_dict=None, max_frames=8,
                 device=None):
        if tile and tile > 0:
            raise NotImplementedError("tiled Real-ESRGAN (tile > 0) is not implemented: the whole frame runs at once")
        if pre_pad and pre_pad > 0:
            raise NotImplementedError("pre_pad > 0 is not implemented")
        if fp32:
            raise NotImplementedError("fp32=True is not implemented: the native upsampler stores fp16 activations "
                                      "(the reference's default, half=not fp32)")
        if state_dict is None:
            if model_path is None:
                raise ValueError("model_path (a local RealESRGAN_x4plus.pth) or state_dict is required")
            state_dict = load_pth(model_path)
        self.cfg = _config_from_state_dict(state_dict)
        self.state = {k: v.detach().to("cpu", torch.float16) for k, v in state_dict.items()}
        self.max_frames = int(max_frames)
        self.device = torch.device(device) if device is not None else None
        self._engine = None

    @classmethod
    def from_pretrained(cls, model_name_or_path="RealESRGAN_x4plus.pth", **kwargs):
        """A LOCAL RealESRGAN_x4plus.pth (or a directory holding one).  Nothing is downloaded: a missing path raises
        FileNotFoundError."""
        p = Path(model_name_or_path)
        if p.is_dir():
            p = p / "RealESRGAN_x4plus.pth"
        if not p.exists():
            raise FileNotFoundError(f"{model_name_or_path}: from_pretrained needs a local RealESRGAN_x4plus.pth "
                                    "(no Hugging Face Hub download here)")
        return cls(str(p), **kwargs)

    @classmethod
    def from_random(cls, seed=0, num_block=23, **kwargs):
        """Seeded random weights with basicsr's initialisation (configs.esrgan_random_state_dict)."""
        return cls(state_dict=esrgan_random_state_dict(ESRGANConfig(num_block=num_block), seed), **kwargs)

    def to(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise N.SdwError("the native Real-ESRGAN upsampler runs on CUDA only (no CPU path)")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device != self.device:
            self.device, self._engine = device, None
        return self

    def engine(self, height, width):
        """The native engine for height x width inputs (one resident engine; rebuilt when the size changes)."""
        if self.device is None:
            self.to("cuda")
        e = self._engine
        if e is None or (e.height, e.width) != (height, width):
            self._engine = None
            e = ESRGANEngine(self.cfg, height, width, self.max_frames, self.device)
            e.load_state_dict(self.state)
            self._engine = e
        return e

    def upsample_frames(self, frames_u8, out_f32=None):
        """CUDA uint8 [n, H, W, 3] -> CUDA uint8 [n, 4H, 4W, 3], in chunks of at most `max_frames` frames."""
        if frames_u8.dtype != torch.uint8 or frames_u8.dim() != 4 or frames_u8.shape[-1] != 3:
            raise NotImplementedError("the device path takes uint8 RGB frames [n, H, W, 3]")
        if self.device is None:
            self.to(frames_u8.device if frames_u8.is_cuda else "cuda")
        x = frames_u8.to(self.device)
        n, H, W, _ = x.shape
        e = self.engine(H, W)
        s = self.cfg.scale
        out = torch.empty((n, s * H, s * W, 3), dtype=torch.uint8, device=self.device)
        for i0 in range(0, n, self.max_frames):
            i1 = min(n, i0 + self.max_frames)
            e.forward(x[i0:i1], out=out[i0:i1], out_f32=None if out_f32 is None else out_f32[i0:i1])
        return out

    def __call__(self, image, outscale=4, convert_to_pil=True):
        """Upsample an RGB image (float array in [0, 1], HWC) or an image path, as the reference's forward
        (upsampling.py:30-55).  A CUDA uint8 tensor [n, H, W, 3] takes the batched device path instead."""
        if outscale != 4:
            raise NotImplementedError("outscale != 4 (resampling after the x4 model) is not implemented")
        if isinstance(image, torch.Tensor) and image.is_cuda:
            return self.upsample_frames(image)
        if isinstance(image, (str, Path)):
            from PIL import Image

            im = Image.open(image)
            if im.mode != "RGB":
                raise NotImplementedError(f"{image}: image mode {im.mode}; only 8-bit RGB inputs are supported "
                                          "(no grayscale / alpha / 16-bit path)")
            img = np.asarray(im, dtype=np.uint8)
        else:
            arr = np.asarray(image)
            if arr.ndim != 3 or arr.shape[2] != 3:
                raise NotImplementedError(f"image of shape {arr.shape}: only RGB HxWx3 inputs are supported")
            img = (arr * 255).round().astype("uint8")  # upsampling.py:46
        out = self.upsample_frames(torch.from_numpy(np.ascontiguousarray(img))[None].to(self.device or "cuda"))
        out = out[0].cpu().numpy()
        if convert_to_pil:
            from PIL import Image

            return Image.fromarray(out)
        return out[:, :, ::-1]  # the reference returns enhance's BGR array when not converting to PIL

    def upsample_imagefolder(self, in_dir, out_dir, suffix="out", outfile_ext=".png", recursive=False, force=False):
        """Upsample every .png / .jpg / .jpeg under in_dir into out_dir (reference upsampling.py:81-99)."""
        in_dir, out_dir = Path(in_dir), Path(out_dir)
        if not in_dir.exists():
            raise FileNotFoundError(f"Provided input directory {in_dir} does not exist")
        out_dir.mkdir(exist_ok=True, parents=True)
        generator = in_dir.rglob("*") if recursive else in_dir.glob("*")
        image_paths = [x for x in generator if x.suffix.lower() in [".png", ".jpg", ".jpeg"]]
        n_img = len(image_paths)
        for i, image in enumerate(image_paths):
            out_filepath = out_dir / (str(image.relative_to(in_dir).with_suffix("")) + suffix + outfile_ext)
            if not force and out_filepath.exists():
                logger.info(f"[{i}/{n_img}] {out_filepath} already exists, skipping. To avoid skipping, pass force=True.")
                continue
            logger.info(f"[{i}/{n_img}] upscaling {image}")
            im = self(str(image))
            out_filepath.parent.mkdir(parents=True, exist_ok=True)
            im.save(out_filepath)


def load_pth(path):
    """State dict of a Real-ESRGAN .pth: `params_ema`, else `params`, else the file itself (RealESRGANer's order)."""
    p = Path(path)
    if not p.exists():
        raise FileNotFoundError(f"{path}: no such Real-ESRGAN weights file")
    obj = torch.load(str(p), map_location="cpu", weights_only=True)
    if isinstance(obj, dict) and "params_ema" in obj:
        obj = obj["params_ema"]
    elif isinstance(obj, dict) and "params" in obj:
        obj = obj["params"]
    if not isinstance(obj, dict) or "conv_first.weight" not in obj:
        raise ValueError(f"{path}: not an RRDBNet state dict (no conv_first.weight)")
    return obj


def _config_from_state_dict(sd):
    """RRDBNet x4 configuration read off the tensor shapes; anything but an RGB x4 model is refused."""
    w0 = sd["conv_first.weight"]
    nf, cin = int(w0.shape[0]), int(w0.shape[1])
    if cin != 3:
        raise NotImplementedError(f"conv_first takes {cin} channels: only RGB x4 models are supported (x2 / x1 models "
                                  "use pixel_unshuffle inputs)")
    if "conv_up1.weight" not in sd or "conv_up2.weight" not in sd:
        raise NotImplementedError("only x4 RRDBNet models (conv_up1 and conv_up2) are supported")
    blocks = [int(k.split(".")[1]) for k in sd if k.startswith("body.")]
    nb = 1 + max(blocks) if blocks else 0
    if nb < 1:
        raise ValueError("state dict has no RRDB blocks")
    g = int(sd["body.0.rdb1.conv1.weight"].shape[0])
    cout = int(sd["conv_last.weight"].shape[0])
    if cout != 3:
        raise NotImplementedError(f"conv_last outputs {cout} channels: only RGB models are supported")
    cfg = ESRGANConfig(num_feat=nf, num_block=nb, num_grow_ch=g)
    want = esrgan_param_shapes(cfg)
    got = set(sd)
    if got != set(want):
        extra, missing = sorted(got - set(want)), sorted(set(want) - got)
        raise ValueError(f"not an RRDBNet x4 state dict: unexpected {extra[:3]}, missing {missing[:3]}")
    return cfg
