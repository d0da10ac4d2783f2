"""Model configurations and parameter-shape tables of the native engine.

The shapes are the published `unet/config.json` / `vae/config.json` architectures of the checkpoints the reference
loads with `from_pretrained` (stable_diffusion_pipeline.py:856): SD-1.x (CompVis/stable-diffusion-v1-4,
tests/test_pipeline.py:21) and SD-2.1.  Key names are the diffusers state-dict keys (SURVEY.md A.6), so a real
checkpoint's tensors can be handed to `Engine.load_state_dict` unchanged.
"""
from dataclasses import dataclass, field
from typing import Dict, Tuple, Union


@dataclass
class UNetConfig:
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    layers_per_block: int = 2
    attention_head_dim: Union[int, Tuple[int, ...]] = 8  # diffusers' name for the NUMBER of heads
    cross_attention_dim: int = 768
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    sample_size: int = 64
    use_linear_projection: bool = False
    prediction_type: str = "epsilon"

    @staticmethod
    def sd14():
        return UNetConfig()

    @staticmethod
    def sd21():
        return UNetConfig(attention_head_dim=(5, 10, 20, 20), cross_attention_dim=1024, use_linear_projection=True,
                          sample_size=96, prediction_type="v_prediction")

    def heads(self, level):
        a = self.attention_head_dim
        return a if isinstance(a, int) else a[level]


@dataclass
class VAEConfig:
    latent_channels: int = 4
    out_channels: int = 3
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: int = 2
    norm_num_groups: int = 32
    scaling_factor: float = 0.18215  # hard-coded in the reference (stable_diffusion_pipeline.py:432)


def _resnet(p, cin, cout, temb, out):
    out[p + ".norm1.weight"] = (cin,)
    out[p + ".norm1.bias"] = (cin,)
    out[p + ".conv1.weight"] = (cout, cin, 3, 3)
    out[p + ".conv1.bias"] = (cout,)
    if temb:
        out[p + ".time_emb_proj.weight"] = (cout, temb)
        out[p + ".time_emb_proj.bias"] = (cout,)
    out[p + ".norm2.weight"] = (cout,)
    out[p + ".norm2.bias"] = (cout,)
    out[p + ".conv2.weight"] = (cout, cout, 3, 3)
    out[p + ".conv2.bias"] = (cout,)
    if cin != cout:
        out[p + ".conv_shortcut.weight"] = (cout, cin, 1, 1)
        out[p + ".conv_shortcut.bias"] = (cout,)


def _transformer(p, c, ctx, linear, out):
    out[p + ".norm.weight"] = (c,)
    out[p + ".norm.bias"] = (c,)
    pshape = (c, c) if linear else (c, c, 1, 1)
    out[p + ".proj_in.weight"] = pshape
    out[p + ".proj_in.bias"] = (c,)
    t = p + ".transformer_blocks.0"
    for n in ("norm1", "norm2", "norm3"):
        out[f"{t}.{n}.weight"] = (c,)
        out[f"{t}.{n}.bias"] = (c,)
    for a, kd in (("attn1", c), ("attn2", ctx)):
        out[f"{t}.{a}.to_q.weight"] = (c, c)
        out[f"{t}.{a}.to_k.weight"] = (c, kd)
        out[f"{t}.{a}.to_v.weight"] = (c, kd)
        out[f"{t}.{a}.to_out.0.weight"] = (c, c)
        out[f"{t}.{a}.to_out.0.bias"] = (c,)
    out[t + ".ff.net.0.proj.weight"] = (8 * c, c)
    out[t + ".ff.net.0.proj.bias"] = (8 * c,)
    out[t + ".ff.net.2.weight"] = (c, 4 * c)
    out[t + ".ff.net.2.bias"] = (c,)
    out[p + ".proj_out.weight"] = pshape
    out[p + ".proj_out.bias"] = (c,)


def unet_param_shapes(cfg: UNetConfig) -> Dict[str, tuple]:
    """name -> shape of every UNet2DConditionModel parameter (diffusers key names)."""
    o: Dict[str, tuple] = {}
    ch = cfg.block_out_channels
    nlev, L = len(ch), cfg.layers_per_block
    temb = ch[0] * 4
    o["conv_in.weight"] = (ch[0], cfg.in_channels, 3, 3)
    o["conv_in.bias"] = (ch[0],)
    o["time_embedding.linear_1.weight"] = (temb, ch[0])
    o["time_embedding.linear_1.bias"] = (temb,)
    o["time_embedding.linear_2.weight"] = (temb, temb)
    o["time_embedding.linear_2.bias"] = (temb,)
    cout = ch[0]
    for i in range(nlev):
        cin, cout = cout, ch[i]
        last = i == nlev - 1
        for j in range(L):
            _resnet(f"down_blocks.{i}.resnets.{j}", cin if j == 0 else cout, cout, temb, o)
            if not last:
                _transformer(f"down_blocks.{i}.attentions.{j}", cout, cfg.cross_attention_dim,
                             cfg.use_linear_projection, o)
        if not last:
            o[f"down_blocks.{i}.downsamplers.0.conv.weight"] = (cout, cout, 3, 3)
            o[f"down_blocks.{i}.downsamplers.0.conv.bias"] = (cout,)
    c = ch[-1]
    _resnet("mid_block.resnets.0", c, c, temb, o)
    _transformer("mid_block.attentions.0", c, cfg.cross_attention_dim, cfg.use_linear_projection, o)
    _resnet("mid_block.resnets.1", c, c, temb, o)
    rev = list(reversed(ch))
    cout = rev[0]
    for i in range(nlev):
        prev, cout = cout, rev[i]
        cin = rev[min(i + 1, nlev - 1)]
        for j in range(L + 1):
            skip = cin if j == L else cout
            rin = prev if j == 0 else cout
            _resnet(f"up_blocks.{i}.resnets.{j}", rin + skip, cout, temb, o)
            if i > 0:
                _transformer(f"up_blocks.{i}.attentions.{j}", cout, cfg.cross_attention_dim,
                             cfg.use_linear_projection, o)
        if i < nlev - 1:
            o[f"up_blocks.{i}.upsamplers.0.conv.weight"] = (cout, cout, 3, 3)
            o[f"up_blocks.{i}.upsamplers.0.conv.bias"] = (cout,)
    o["conv_norm_out.weight"] = (ch[0],)
    o["conv_norm_out.bias"] = (ch[0],)
    o["conv_out.weight"] = (cfg.out_channels, ch[0], 3, 3)
    o["conv_out.bias"] = (cfg.out_channels,)
    return o


def vae_param_shapes(cfg: VAEConfig) -> Dict[str, tuple]:
    """name -> shape of `post_quant_conv` + `decoder.*` of AutoencoderKL (keys WITHOUT the engine's "vae." prefix)."""
    o: Dict[str, tuple] = {}
    ch = cfg.block_out_channels
    lc, top = cfg.latent_channels, ch[-1]
    o["post_quant_conv.weight"] = (lc, lc, 1, 1)
    o["post_quant_conv.bias"] = (lc,)
    o["decoder.conv_in.weight"] = (top, lc, 3, 3)
    o["decoder.conv_in.bias"] = (top,)
    _resnet("decoder.mid_block.resnets.0", top, top, 0, o)
    a = "decoder.mid_block.attentions.0"
    o[a + ".group_norm.weight"] = (top,)
    o[a + ".group_norm.bias"] = (top,)
    for n in ("to_q", "to_k", "to_v", "to_out.0"):
        o[f"{a}.{n}.weight"] = (top, top)
        o[f"{a}.{n}.bias"] = (top,)
    _resnet("decoder.mid_block.resnets.1", top, top, 0, o)
    rev = list(reversed(ch))
    cout = rev[0]
    for i in range(len(ch)):
        cin, cout = cout, rev[i]
        for j in range(cfg.layers_per_block + 1):
            _resnet(f"decoder.up_blocks.{i}.resnets.{j}", cin if j == 0 else cout, cout, 0, o)
        if i < len(ch) - 1:
            o[f"decoder.up_blocks.{i}.upsamplers.0.conv.weight"] = (cout, cout, 3, 3)
            o[f"decoder.up_blocks.{i}.upsamplers.0.conv.bias"] = (cout,)
    o["decoder.conv_norm_out.weight"] = (ch[0],)
    o["decoder.conv_norm_out.bias"] = (ch[0],)
    o["decoder.conv_out.weight"] = (cfg.out_channels, ch[0], 3, 3)
    o["decoder.conv_out.bias"] = (cfg.out_channels,)
    return o


# older diffusers VAE checkpoints name the attention projections query/key/value/proj_attn
VAE_KEY_ALIASES = {"query": "to_q", "key": "to_k", "value": "to_v", "proj_attn": "to_out.0"}


def random_state_dict(shapes: Dict[str, tuple], seed: int, dtype=None, device="cpu"):
    """Random-init weights with torch's default Conv2d/Linear scale (U(-1/sqrt(fan_in), 1/sqrt(fan_in))) and
    identity norm affines, generated name-by-name in sorted order from one CPU generator (deterministic)."""
    import torch

    g = torch.Generator(device="cpu").manual_seed(seed)
    sd = {}
    for name in sorted(shapes):
        shp = shapes[name]
        leaf = name.rsplit(".", 2)[-2] if name.count(".") >= 1 else name
        is_norm = "norm" in leaf
        if is_norm:
            t = torch.ones(shp) if name.endswith("weight") else torch.zeros(shp)
        else:
            if name.endswith("weight"):
                fan_in = 1
                for s in shp[1:]:
                    fan_in *= s
            else:
                w = shapes[name[:-4] + "weight"]
                fan_in = 1
                for s in w[1:]:
                    fan_in *= s
            bound = fan_in ** -0.5
            t = (torch.rand(shp, generator=g) * 2 - 1) * bound
        sd[name] = t.to(dtype or torch.float16).to(device)
    return sd


@dataclass
class ESRGANConfig:
    """basicsr RRDBNet as RealESRGANModel builds it (the reference's upsampling.py:25): RealESRGAN_x4plus."""
    num_in_ch: int = 3
    num_out_ch: int = 3
    num_feat: int = 64
    num_block: int = 23
    num_grow_ch: int = 32
    scale: int = 4


def esrgan_param_shapes(cfg: ESRGANConfig) -> Dict[str, tuple]:
    """name -> shape of every RRDBNet parameter (basicsr state-dict keys, as in RealESRGAN_x4plus.pth)."""
    o: Dict[str, tuple] = {}
    nf, g = cfg.num_feat, cfg.num_grow_ch

    def conv(name, cout, cin):
        o[name + ".weight"] = (cout, cin, 3, 3)
        o[name + ".bias"] = (cout,)

    conv("conv_first", nf, cfg.num_in_ch)
    for i in range(cfg.num_block):
        for r in (1, 2, 3):
            for k in range(4):
                conv(f"body.{i}.rdb{r}.conv{k + 1}", g, nf + k * g)
            conv(f"body.{i}.rdb{r}.conv5", nf, nf + 4 * g)
    for name in ("conv_body", "conv_up1", "conv_up2", "conv_hr"):
        conv(name, nf, nf)
    conv("conv_last", cfg.num_out_ch, nf)
    return o


def esrgan_random_state_dict(cfg: ESRGANConfig, seed: int, dtype=None, device="cpu"):
    """Random RRDBNet weights initialised as basicsr does: the dense-block convs get `default_init_weights(scale=0.1)`
    (Kaiming-normal fan-in weights x 0.1, zero bias), every other conv torch's Conv2d default
    (U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for weight and bias).  Generated name-by-name in sorted order from one CPU
    generator (deterministic).  One departure: `conv_last` gets half-scale weights and a bias of 0.5, so the untrained
    model's image sits mid-range, as a trained model's does, instead of a third of its pixels clamping at 0 — parity
    fixtures built on it then compare unsaturated pixels."""
    import torch

    shapes = esrgan_param_shapes(cfg)
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd = {}
    for name in sorted(shapes):
        shp = shapes[name]
        wshp = shapes[name.rsplit(".", 1)[0] + ".weight"]
        fan_in = wshp[1] * wshp[2] * wshp[3]
        if name.startswith("body."):
            if name.endswith("weight"):
                t = torch.randn(shp, generator=g) * (2.0 / fan_in) ** 0.5 * 0.1
            else:
                t = torch.zeros(shp)
        else:
            t = (torch.rand(shp, generator=g) * 2 - 1) * fan_in ** -0.5
            if name == "conv_last.weight":
                t = t * 0.5
            elif name == "conv_last.bias":
                t = torch.full(shp, 0.5)
        sd[name] = t.to(dtype or torch.float16).to(device)
    return sd
