"""Real-ESRGAN upsampler without a GPU: the oracle's architecture (parameter count and basicsr key set), the native
engine's dry-run plan at 512x512 / 8 frames (every launch plans, registry = oracle keys, arena size), and the host logic
of RealESRGANModel / make_clip_frames(upsample=True)."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import esrgan as OE  # noqa: E402


def _basicsr_keys(num_block=23):
    keys = ["conv_first"]
    keys += [f"body.{i}.rdb{r}.conv{k}" for i in range(num_block) for r in (1, 2, 3) for k in range(1, 6)]
    keys += ["conv_body", "conv_up1", "conv_up2", "conv_hr", "conv_last"]
    return {f"{k}.{s}" for k in keys for s in ("weight", "bias")}


def test_oracle_x4plus_parameter_count_and_keys():
    shapes = OE.param_shapes()
    assert OE.num_params(shapes) == 16_697_987
    assert set(shapes) == _basicsr_keys()
    assert shapes["body.22.rdb3.conv5.weight"] == (64, 192, 3, 3)
    assert shapes["body.0.rdb1.conv4.weight"] == (32, 160, 3, 3)
    from stable_diffusion_videos_b200.configs import ESRGANConfig, esrgan_param_shapes

    assert esrgan_param_shapes(ESRGANConfig()) == shapes


def test_oracle_small_instance_runs_and_is_not_saturated():
    from stable_diffusion_videos_b200.configs import ESRGANConfig, esrgan_random_state_dict

    sd = {k: v.float() for k, v in esrgan_random_state_dict(ESRGANConfig(num_block=2), 0).items()}
    frames = np.load(os.path.join(ROOT, "tests", "golden", "cfg1_frames_u8.npy"))[:1, :16, :16]
    u8, raw = OE.enhance(sd, frames)
    assert u8.shape == (1, 64, 64, 3) and raw.shape == (1, 64, 64, 3)
    assert ((u8 == 0) | (u8 == 255)).mean() < 0.05


def _esrgan_cfg(frames=8, hw=(512, 512), num_block=23):
    from stable_diffusion_videos_b200.upsampling import ESRGANEngineConfig

    return ESRGANEngineConfig(3, 3, 64, num_block, 32, 4, hw[0], hw[1], frames)


def test_engine_dry_run_plans_512_f8():
    from stable_diffusion_videos_b200 import _native

    lib = _native.lib()
    lib.sdw_debug_plan_only(1)
    try:
        c = _esrgan_cfg()
        h = C.c_void_p()
        _native.check(lib.sdw_esrgan_create(C.byref(c), C.byref(h)))
        n = C.c_uint64()
        _native.check(lib.sdw_esrgan_arena_bytes(h, C.byref(n)))
        # 8 frames: 37 MB packed weights + 268 MB conv_first features + the shared trunk / tail region, which the
        # two 2048x2048x64 fp16 tail buffers set (2 x 4.29 GB; the trunk's three 512x512x192 dense buffers need 2.4 GB)
        assert 8.8e9 < n.value < 9.0e9, n.value
        _native.check(lib.sdw_esrgan_bind(h, C.c_void_p(1 << 40), n))  # fake, aligned, never dereferenced
        launches = C.c_int()
        _native.check(lib.sdw_esrgan_launches(h, C.byref(launches)))
        # conv_first + copy into the dense buffer, 23 x 3 x 5 trunk GEMMs, conv_body, 2 x 4 parity GEMMs, conv_hr, conv_last
        assert launches.value == 2 + 23 * 15 + 1 + 8 + 1 + 1
        got = {}
        name, numel = C.c_char_p(), C.c_int64()
        for i in range(lib.sdw_esrgan_num_params(h)):
            _native.check(lib.sdw_esrgan_param_info(h, i, C.byref(name), C.byref(numel)))
            got[name.value.decode()] = numel.value
        assert got == {k: math.prod(s) for k, s in OE.param_shapes().items()}
        first = C.c_char_p()
        assert lib.sdw_esrgan_missing_params(h, C.byref(first)) == len(got)
        lib.sdw_esrgan_destroy(h)
        # other frame counts / sizes plan too
        for frames, hw in ((30, (512, 512)), (1, (64, 64)), (2, (64, 96)), (3, (24, 40))):
            c = _esrgan_cfg(frames, hw)
            _native.check(lib.sdw_esrgan_create(C.byref(c), C.byref(h)))
            _native.check(lib.sdw_esrgan_arena_bytes(h, C.byref(n)))
            _native.check(lib.sdw_esrgan_bind(h, C.c_void_p(1 << 40), n))
            lib.sdw_esrgan_destroy(h)
    finally:
        lib.sdw_debug_plan_only(0)


def test_engine_rejects_unsupported_configs():
    from stable_diffusion_videos_b200 import _native

    lib = _native.lib()
    h = C.c_void_p()
    c = _esrgan_cfg()
    c.scale = 2
    assert lib.sdw_esrgan_create(C.byref(c), C.byref(h)) == 1
    assert b"x4" in lib.sdw_last_error()
    c = _esrgan_cfg()
    c.num_in_ch = 4
    assert lib.sdw_esrgan_create(C.byref(c), C.byref(h)) == 1


def _random_sd(num_block=1):
    from stable_diffusion_videos_b200.configs import ESRGANConfig, esrgan_random_state_dict

    return esrgan_random_state_dict(ESRGANConfig(num_block=num_block), 0)


@pytest.mark.parametrize("wrap", ["params_ema", "params", None])
def test_from_pretrained_reads_local_pth(tmp_path, wrap):
    from stable_diffusion_videos_b200 import RealESRGANModel

    sd = _random_sd(2)
    obj = {wrap: sd} if wrap else sd
    if wrap == "params":  # RealESRGANer prefers params_ema; a file with only `params` uses those
        obj["other"] = {"x": torch.zeros(1)}
    path = tmp_path / "RealESRGAN_x4plus.pth"
    torch.save(obj, path)
    m = RealESRGANModel.from_pretrained(str(path))
    assert m.cfg.num_block == 2 and m.cfg.num_feat == 64 and m.cfg.num_grow_ch == 32
    assert set(m.state) == set(sd)
    assert torch.equal(m.state["conv_first.weight"], sd["conv_first.weight"])
    m2 = RealESRGANModel.from_pretrained(str(tmp_path))  # a directory holding the file
    assert set(m2.state) == set(sd)


def test_from_pretrained_prefers_params_ema(tmp_path):
    from stable_diffusion_videos_b200 import RealESRGANModel

    a, b = _random_sd(1), {k: v + 1 for k, v in _random_sd(1).items()}
    torch.save({"params": a, "params_ema": b}, tmp_path / "w.pth")
    m = RealESRGANModel.from_pretrained(str(tmp_path / "w.pth"))
    assert torch.equal(m.state["conv_last.bias"], b["conv_last.bias"])


def test_from_pretrained_missing_path_raises(tmp_path):
    from stable_diffusion_videos_b200 import RealESRGANModel

    with pytest.raises(FileNotFoundError):
        RealESRGANModel.from_pretrained(str(tmp_path / "nope.pth"))
    with pytest.raises(FileNotFoundError):
        RealESRGANModel.from_pretrained("nateraw/real-esrgan")  # a hub id is not a local file: no download


@pytest.mark.parametrize("kw", [dict(tile=256), dict(pre_pad=10), dict(fp32=True)])
def test_unsupported_constructor_options_raise(kw):
    from stable_diffusion_videos_b200 import RealESRGANModel

    with pytest.raises(NotImplementedError):
        RealESRGANModel(state_dict=_random_sd(), **kw)


def test_unsupported_call_options_raise(tmp_path):
    from PIL import Image

    from stable_diffusion_videos_b200 import RealESRGANModel

    m = RealESRGANModel(state_dict=_random_sd())
    with pytest.raises(NotImplementedError):
        m(np.zeros((8, 8, 3), np.float32), outscale=2)
    with pytest.raises(NotImplementedError):
        m(np.zeros((8, 8), np.float32))  # grayscale
    with pytest.raises(NotImplementedError):
        m(np.zeros((8, 8, 4), np.float32))  # alpha
    Image.new("RGBA", (8, 8)).save(tmp_path / "a.png")
    with pytest.raises(NotImplementedError):
        m(str(tmp_path / "a.png"))
    with pytest.raises(NotImplementedError):
        m.upsample_frames(torch.zeros((1, 8, 8, 4), dtype=torch.uint8))


def test_non_x4_or_foreign_state_dicts_raise():
    from stable_diffusion_videos_b200 import RealESRGANModel

    sd = _random_sd()
    x2 = dict(sd, **{"conv_first.weight": torch.zeros(64, 12, 3, 3)})  # x2 models read pixel_unshuffle'd 12 channels
    with pytest.raises(NotImplementedError):
        RealESRGANModel(state_dict=x2)
    with pytest.raises(ValueError):
        RealESRGANModel(state_dict=dict(sd, extra=torch.zeros(1)))


def _bare_pipe():
    from stable_diffusion_videos_b200.configs import UNetConfig, VAEConfig
    from stable_diffusion_videos_b200.pipeline import (NativeUNet, NativeVAE, StableDiffusionWalkPipeline,
                                                       SyntheticTokenizer)

    return StableDiffusionWalkPipeline(NativeVAE(VAEConfig(), {}), None, SyntheticTokenizer(),
                                       NativeUNet(UNetConfig(), {}), None)


def test_upsample_without_upsampler_raises_documented_error(tmp_path):
    pipe = _bare_pipe()
    with pytest.raises(ValueError, match=r"pipe\.upsampler = RealESRGANModel\.from_pretrained"):
        pipe.make_clip_frames("a", "b", 1, 2, num_interpolation_steps=2, save_path=tmp_path, upsample=True)


def test_upsample_with_tiled_raises(tmp_path):
    from stable_diffusion_videos_b200 import RealESRGANModel

    pipe = _bare_pipe()
    pipe.tiled = True
    pipe.upsampler = RealESRGANModel(state_dict=_random_sd())
    with pytest.raises(NotImplementedError, match="tiled"):
        pipe.make_clip_frames("a", "b", 1, 2, num_interpolation_steps=2, save_path=tmp_path, upsample=True)
