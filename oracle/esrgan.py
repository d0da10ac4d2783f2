"""ORACLE — fp32 restatement of the reference's Real-ESRGAN upsampler (RealESRGANModel, upsampling.py).  TEST
INFRASTRUCTURE ONLY.

The model is basicsr's `RRDBNet(num_in_ch=3, num_out_ch=3, num_feat=64, num_block=23, num_grow_ch=32, scale=4)`
(upsampling.py:25) written in torch.nn.functional over a basicsr-keyed state dict; `enhance` restates
`RealESRGANer.enhance` for tile = 0, pre_pad = 0, outscale = 4 on an RGB uint8 frame (the reference's two BGR flips,
upsampling.py:47,52 and the pair inside `enhance`, cancel out, so the network sees RGB).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F


def param_shapes(num_in_ch=3, num_out_ch=3, num_feat=64, num_block=23, num_grow_ch=32):
    """name -> shape of every RRDBNet x4 parameter (basicsr key names)."""
    o = {}

    def conv(name, cout, cin):
        o[name + ".weight"] = (cout, cin, 3, 3)
        o[name + ".bias"] = (cout,)

    conv("conv_first", num_feat, num_in_ch)
    for i in range(num_block):
        for r in (1, 2, 3):
            for k in range(4):
                conv(f"body.{i}.rdb{r}.conv{k + 1}", num_grow_ch, num_feat + k * num_grow_ch)
            conv(f"body.{i}.rdb{r}.conv5", num_feat, num_feat + 4 * num_grow_ch)
    conv("conv_body", num_feat, num_feat)
    conv("conv_up1", num_feat, num_feat)
    conv("conv_up2", num_feat, num_feat)
    conv("conv_hr", num_feat, num_feat)
    conv("conv_last", num_out_ch, num_feat)
    return o


def _lrelu(x):
    return F.leaky_relu(x, 0.2)


def rrdbnet_forward(sd, x, num_block=None, store=None):
    """RRDBNet x4 on x [B, 3, H, W] (fp32, in [0, 1]) -> [B, 3, 4H, 4W], before any clamp.

    `store` (optional): applied to every conv output and block exit — e.g. an fp16 rounding to emulate fp16 storage."""
    store = store or (lambda t: t)
    if num_block is None:
        num_block = 1 + max(int(k.split(".")[1]) for k in sd if k.startswith("body."))

    def conv(name, t):
        return F.conv2d(t, sd[name + ".weight"].float(), sd[name + ".bias"].float(), padding=1)

    feat = store(conv("conv_first", x))
    h = feat
    for i in range(num_block):
        x0 = h
        for r in (1, 2, 3):
            p = f"body.{i}.rdb{r}."
            xs = [h]
            for k in range(1, 5):
                xs.append(store(_lrelu(conv(p + f"conv{k}", torch.cat(xs, 1)))))
            x5 = conv(p + "conv5", torch.cat(xs, 1))
            h = x5 * 0.2 + h
            if r < 3:
                h = store(h)
        h = store(h * 0.2 + x0)
    feat = store(conv("conv_body", h) + feat)
    feat = store(_lrelu(conv("conv_up1", F.interpolate(feat, scale_factor=2, mode="nearest"))))
    feat = store(_lrelu(conv("conv_up2", F.interpolate(feat, scale_factor=2, mode="nearest"))))
    return conv("conv_last", store(_lrelu(conv("conv_hr", feat))))


def to_uint8(out):
    """RealESRGANer.enhance's post-process: clamp(0, 1) * 255, round, uint8; NCHW -> NHWC numpy."""
    return (out.clamp(0, 1) * 255.0).round().to(torch.uint8).permute(0, 2, 3, 1).numpy()


def enhance(sd, frames_u8, num_block=None, store=None):
    """uint8 RGB frames [n, H, W, 3] -> (uint8 [n, 4H, 4W, 3], fp32 pre-clamp output NHWC)."""
    x = torch.from_numpy(np.ascontiguousarray(frames_u8)).permute(0, 3, 1, 2).float() / 255.0
    with torch.no_grad():
        out = rrdbnet_forward(sd, x, num_block, store)
    return to_uint8(out), out.permute(0, 2, 3, 1).contiguous().numpy()


def num_params(shapes):
    return sum(math.prod(s) for s in shapes.values())
