"""The C-ABI library loads without a GPU and exports every symbol include/sdwalk.h declares; the engine's
dry-run planner sizes the arena for the real SD-1.4 configuration (no compute calls)."""
import ctypes as C

import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported():
    from stable_diffusion_videos_b200 import _native

    lib = _native.lib()
    hdr = open(os.path.join(ROOT, "include", "sdwalk.h")).read()
    names = set(re.findall(r"\b(sdw_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
    assert lib.sdw_abi_version() == 2


def test_engine_dry_run_sizes_sd14_arena():
    from stable_diffusion_videos_b200 import _native
    from stable_diffusion_videos_b200.configs import UNetConfig, VAEConfig
    from stable_diffusion_videos_b200.engine import EngineConfig

    lib = _native.lib()
    c = EngineConfig()
    u, v = UNetConfig.sd14(), VAEConfig()
    c.in_channels, c.out_channels, c.num_levels, c.layers_per_block = 4, 4, 4, 2
    for i, ch in enumerate(u.block_out_channels):
        c.block_out_channels[i] = ch
        c.attention_heads[i] = 8
    c.cross_attention_dim, c.ctx_tokens, c.norm_num_groups, c.norm_eps = 768, 77, 32, 1e-5
    c.vae_num_levels, c.vae_layers_per_block, c.vae_norm_num_groups = 4, 2, 32
    for i, ch in enumerate(v.block_out_channels):
        c.vae_block_out_channels[i] = ch
    c.vae_out_channels, c.vae_scale, c.vae_scaling_factor = 3, 8, 0.18215
    c.latent_h = c.latent_w = 64
    c.frames, c.guidance, c.max_steps = 4, 1, 64
    h = C.c_void_p()
    _native.check(lib.sdw_engine_create(C.byref(c), C.byref(h)))
    n = C.c_uint64()
    _native.check(lib.sdw_engine_arena_bytes(h, C.byref(n)))
    # 1.72 GB UNet + 0.1 GB VAE weights (+ K padding) plus activations with build-time liveness (scratch scopes, VAE
    # ping-pong): 3.6 GB at 4 frames; the bump-only allocator needed 16 GB here (and 110 GB at 30 frames)
    assert 2e9 < n.value < 6e9
    from stable_diffusion_videos_b200.configs import unet_param_shapes, vae_param_shapes
    import math

    want = {k: math.prod(s) for k, s in unet_param_shapes(u).items()}
    want.update({"vae." + k: math.prod(s) for k, s in vae_param_shapes(v).items()})
    got = {}
    name, numel = C.c_char_p(), C.c_int64()
    for i in range(lib.sdw_engine_num_params(h)):
        _native.check(lib.sdw_engine_param_info(h, i, C.byref(name), C.byref(numel)))
        got[name.value.decode()] = numel.value
    assert got == want  # the engine's registry IS the diffusers key set (859,520,964 + 49,490,199 parameters)
    assert sum(got.values()) == 859_520_964 + 49_490_199
    a, b, d = C.c_int(), C.c_int(), C.c_int()
    _native.check(lib.sdw_engine_launches(h, C.byref(a), C.byref(b), C.byref(d)))
    assert b.value > 300 and d.value > 50
    lib.sdw_engine_destroy(h)
    # invalid configuration -> error code + message, no crash
    c.frames = 0
    assert lib.sdw_engine_create(C.byref(c), C.byref(h)) == 1
    assert b"bad sizes" in lib.sdw_last_error()


def _cfg(u, v, hw, frames):
    from stable_diffusion_videos_b200.engine import EngineConfig

    c = EngineConfig()
    c.in_channels, c.out_channels, c.num_levels, c.layers_per_block = 4, 4, len(u.block_out_channels), u.layers_per_block
    for i, ch in enumerate(u.block_out_channels):
        c.block_out_channels[i] = ch
        c.attention_heads[i] = u.heads(i)
    c.cross_attention_dim, c.ctx_tokens, c.norm_num_groups, c.norm_eps = u.cross_attention_dim, 77, u.norm_num_groups, 1e-5
    c.vae_num_levels, c.vae_layers_per_block, c.vae_norm_num_groups = len(v.block_out_channels), v.layers_per_block, v.norm_num_groups
    for i, ch in enumerate(v.block_out_channels):
        c.vae_block_out_channels[i] = ch
    c.vae_out_channels, c.vae_scale, c.vae_scaling_factor = 3, 2 ** (len(v.block_out_channels) - 1), 0.18215
    c.latent_h, c.latent_w = hw
    c.frames, c.guidance, c.max_steps = frames, 1, 64
    return c


def test_launch_plans_validate_without_a_gpu():
    """every GEMM of the SD-1.4 / SD-2.1 / test configurations passes the planner's shape + TMA-alignment checks
    (plan-only mode: tensor maps are validated, not encoded; nothing is launched)."""
    from _helpers import MID_UNET, MID_VAE, TINY_UNET, TINY_VAE, product_cfgs
    from stable_diffusion_videos_b200 import _native
    from stable_diffusion_videos_b200.configs import UNetConfig, VAEConfig

    lib = _native.lib()
    lib.sdw_debug_plan_only(1)
    try:
        cases = [(UNetConfig.sd14(), VAEConfig(), (64, 64), 2), (UNetConfig.sd21(), VAEConfig(), (96, 96), 1),
                 (UNetConfig.sd14(), VAEConfig(), (8, 8), 2), (UNetConfig.sd14(), VAEConfig(), (64, 64), 30),
                 (UNetConfig.sd14(), VAEConfig(), (64, 64), 16)]
        cases += [product_cfgs(TINY_UNET, TINY_VAE) + ((8, 8), 2), product_cfgs(TINY_UNET, TINY_VAE) + ((16, 8), 1),
                  product_cfgs(MID_UNET, MID_VAE) + ((16, 16), 1)]
        for u, v, hw, frames in cases:
            c = _cfg(u, v, hw, frames)
            h = C.c_void_p()
            _native.check(lib.sdw_engine_create(C.byref(c), C.byref(h)))
            n = C.c_uint64()
            _native.check(lib.sdw_engine_arena_bytes(h, C.byref(n)))
            _native.check(lib.sdw_engine_bind(h, C.c_void_p(1 << 40), n))  # fake, aligned, never dereferenced
            lib.sdw_engine_destroy(h)
    finally:
        lib.sdw_debug_plan_only(0)
