"""GPU tests of the native 4x Real-ESRGAN upsampler: the small-N GEMM shapes of a residual dense block (channel-prefix
input, channel-slice output, LeakyReLU, scaled residuals) against TF32-free torch fp32 convs; the full x4plus forward
against the committed oracle fixture (calibrated tolerance, tests/golden/make_golden_esrgan.py); graph replay vs eager;
a one-block engine against the oracle; and walk(upsample=True) against the upsampler applied to the plain walk's frames.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

TOL_X = 1.25  # native-vs-oracle error allowed as a multiple of the calibrated fp16-storage spread (as test_golden_full_gpu)
FLOOR = {"raw_rel_l2": 0.0, "frames_mean_lsb": 0.0, "frames_p999_lsb": 1.0}


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.float16).cuda()


def _tol(ref):
    return float(ref.abs().max()) * 2.0 ** -9 + 1e-3


@pytest.mark.parametrize("N", [32, 64])
@pytest.mark.parametrize("Cin", [64, 96, 128, 160, 192])
@pytest.mark.parametrize("case", ["leaky", "dense_exit", "rrdb_exit"])
def test_small_n_conv_on_dense_buffer(N, Cin, case):
    """conv over channels [0, Cin) of a [B][H][W][192] concat buffer, written into channels [c0, c0 + N) of another
    192-wide buffer: conv1..4 (LeakyReLU), the dense-block exit 0.2 (acc + b) + x and the RRDB exit
    0.2 (0.2 (acc + b) + x) + x0 (second residual through sdw_gemm_res2)."""
    import ctypes as C

    from stable_diffusion_videos_b200 import _native as n

    B, H, W, ld = 2, 24, 40, 192
    buf = _rand(B, H, W, ld, seed=1)
    x = buf[..., :Cin]
    w = _rand(N, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=2)
    b = _rand(N, seed=3).float()
    dst = torch.full((B, H, W, ld), float("nan"), dtype=torch.float16, device="cuda")
    c0 = 96 if N == 32 else 0
    out = dst[..., c0:c0 + N]
    resid = buf[..., :N]
    x0 = _rand(B, H, W, ld, seed=4)[..., :N]
    wp = n.pack_weight(w)
    d = n.GemmDesc()
    d.A = x.data_ptr()
    d.C, d.W, d.H, d.B = Cin, W, H, B
    d.sW, d.sH, d.sB = x.stride(2), x.stride(1), x.stride(0)
    d.conv = 1
    d.Wt = wp.data_ptr()
    d.N = N
    d.out, d.ldc = out.data_ptr(), ld
    d.alpha = 1.0
    ref = Fn.conv2d(x.float().permute(0, 3, 1, 2), w.float(), padding=1).permute(0, 2, 3, 1)
    if case == "leaky":
        d.bias = b.data_ptr()
        d.act = 2
        ref = Fn.leaky_relu(ref + b, 0.2)
    else:
        bs = (0.2 * b).contiguous()  # the engine's bias pre-scale
        d.bias = bs.data_ptr()
        d.alpha = 0.2
        d.resid, d.ldr = resid.data_ptr(), ld
        ref = 0.2 * ref + bs + resid.float()
    if case == "rrdb_exit":
        ref = 0.2 * ref + x0.float()
        n.check(n.lib().sdw_gemm_res2(C.byref(d), C.c_void_p(x0.data_ptr()), C.c_float(0.2), n.stream_ptr()))
    else:
        n.gemm(d)
    torch.cuda.synchronize()
    got = out.float()
    assert torch.isfinite(got).all()
    err = (got - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))
    rest = torch.cat([dst[..., :c0], dst[..., c0 + N:]], -1)
    assert torch.isnan(rest.float()).all()  # nothing outside the slice was written


@pytest.mark.parametrize("act", [1, 2])
def test_leaky_and_silu_on_the_cta_pair_kernel(act):
    """act = 2 on the 2-CTA kernel's TMA epilogue (N >= 128) and its classic epilogue (TMA epilogue off)."""
    sys.path.insert(0, HERE)
    from test_gemm_gpu import ref_conv, run_conv

    x = _rand(2, 16, 16, 128, seed=8)
    w = _rand(128, 128, 3, 3, scale=(9 * 128) ** -0.5, seed=9)
    bias = _rand(128, seed=10).float()
    ref = ref_conv(x, w, 1, bias=bias)
    ref = Fn.silu(ref) if act == 1 else Fn.leaky_relu(ref, 0.2)
    for et in (2, 1):
        out = run_conv(x, w, 1, bias=bias, act=act, ver=2, et=et)
        assert (out.float() - ref).abs().max().item() <= _tol(ref), et


def _golden_model(num_block=23):
    from stable_diffusion_videos_b200 import RealESRGANModel
    from stable_diffusion_videos_b200.configs import ESRGANConfig, esrgan_random_state_dict

    return RealESRGANModel(state_dict=esrgan_random_state_dict(ESRGANConfig(num_block=num_block), 0), max_frames=2)


def test_x4plus_matches_golden_fixture():
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_golden_esrgan as mg

    gold = np.load(os.path.join(HERE, "golden", "esrgan_x4plus_f2.npz"))
    cal = json.load(open(os.path.join(HERE, "golden", "esrgan_calibration.json")))["esrgan_x4plus_f2"]
    assert cal["saturated_frac"] < 0.05
    frames = np.load(os.path.join(HERE, "golden", "cfg1_frames_u8.npy"))
    m = _golden_model().to("cuda")
    x = torch.from_numpy(frames).cuda()
    raw = torch.empty((2, 256, 256, 3), dtype=torch.float32, device="cuda")
    u8 = m.upsample_frames(x, out_f32=raw)
    torch.cuda.synchronize()
    u8, raw = u8.cpu().numpy(), raw.cpu().numpy()[:, ::mg.RAW_STRIDE, ::mg.RAW_STRIDE]
    gf, gr = gold["frames"], gold["raw"]
    assert np.isfinite(raw).all()
    d = np.abs(u8.astype(np.int32) - gf.astype(np.int32))
    got = {"raw_rel_l2": float(np.linalg.norm(raw - gr) / np.linalg.norm(gr)), "frames_mean_lsb": float(d.mean()),
           "frames_p999_lsb": float(np.quantile(d, 0.999)), "frames_max_lsb": int(d.max())}
    print(json.dumps({"native_vs_fp32_oracle": got, "fp16_storage_oracle_vs_fp32_oracle": cal}))  # shown with -s / -rA
    for k, floor in FLOOR.items():
        limit = max(TOL_X * cal[k], floor)
        assert got[k] <= limit, (k, got[k], "limit", limit, "calibrated spread", cal[k])


def test_graph_replay_equals_eager():
    m = _golden_model(num_block=2).to("cuda")
    frames = torch.from_numpy(np.load(os.path.join(HERE, "golden", "cfg1_frames_u8.npy"))).cuda()
    e = m.engine(64, 64)
    g1 = e.forward(frames, use_graph=True)
    g2 = e.forward(frames, use_graph=True)  # replay of the captured graph
    ea = e.forward(frames, use_graph=False)
    one = e.forward(frames[1:], use_graph=True)  # n < frames: its own plan and graph
    torch.cuda.synchronize()
    assert torch.equal(g1, ea) and torch.equal(g2, ea)
    assert torch.equal(one[0], ea[1])


def test_one_block_engine_matches_oracle():
    """num_block = 1 with torch-default-scale weights and non-zero biases everywhere (every epilogue term matters)."""
    from oracle import esrgan as OE
    from stable_diffusion_videos_b200 import RealESRGANModel

    g = torch.Generator().manual_seed(7)
    sd = {}
    for k, s in OE.param_shapes(num_block=1).items():
        fan_in = s[1] * 9 if len(s) == 4 else None
        bound = (fan_in if fan_in else 64 * 9) ** -0.5
        sd[k] = ((torch.rand(s, generator=g) * 2 - 1) * bound).half()
    sd["conv_last.bias"] = sd["conv_last.bias"] + 0.5
    frames = np.load(os.path.join(HERE, "golden", "cfg1_frames_u8.npy"))[:, :32, :48]
    ref_u8, ref_raw = OE.enhance({k: v.float() for k, v in sd.items()}, frames)
    m = RealESRGANModel(state_dict=sd, max_frames=2).to("cuda")
    raw = torch.empty((2, 128, 192, 3), dtype=torch.float32, device="cuda")
    u8 = m.upsample_frames(torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out_f32=raw).cpu().numpy()
    raw = raw.cpu().numpy()
    dev = ref_raw - 0.5
    rel = float(np.linalg.norm(raw - ref_raw) / np.linalg.norm(dev))
    assert rel < 4e-3, rel  # relative to the signal around the 0.5 offset
    d = np.abs(u8.astype(np.int32) - ref_u8.astype(np.int32))
    assert d.max() <= 2 and d.mean() < 0.1, (d.max(), d.mean())


def test_walk_upsample_equals_upsampler_on_plain_walk(tmp_path):
    """3 frames in batches of 2 (the tail batch padded and dropped): the 4x PNGs of walk(upsample=True) equal the
    upsampler applied to the PNGs of the same walk without upsampling."""
    from PIL import Image

    from _helpers import TINY_UNET, TINY_VAE, product_cfgs
    from stable_diffusion_videos_b200 import RealESRGANModel
    from stable_diffusion_videos_b200.pipeline import StableDiffusionWalkPipeline

    sys.path.insert(0, HERE)
    ucfg, vcfg = product_cfgs(TINY_UNET, TINY_VAE)
    pipe = StableDiffusionWalkPipeline.from_random(ucfg, vcfg, seed=0)
    up = _golden_model(num_block=2)
    kw = dict(prompts=["a", "b"], seeds=[1, 2], num_interpolation_steps=3, num_inference_steps=3, height=64, width=64,
              batch_size=2, make_video=False)
    pipe.walk(output_dir=str(tmp_path), name="plain", upsample=False, **kw)
    pipe.upsampler = up
    pipe.walk(output_dir=str(tmp_path), name="up", upsample=True, **kw)
    plain = sorted((tmp_path / "plain" / "plain_000000").glob("*.png"))
    ups = sorted((tmp_path / "up" / "up_000000").glob("*.png"))
    assert len(plain) == 3 and [p.name for p in ups] == [p.name for p in plain]
    frames = torch.from_numpy(np.stack([np.asarray(Image.open(p)) for p in plain])).cuda()
    want = up.upsample_frames(frames).cpu().numpy()
    for i, p in enumerate(ups):
        got = np.asarray(Image.open(p))
        assert got.shape == (4 * frames.shape[1], 4 * frames.shape[2], 3)
        assert np.array_equal(got, want[i]), p.name
