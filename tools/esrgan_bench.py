"""Real-ESRGAN x4plus upsampler on one GPU: each 3x3 conv shape of a residual dense block at 512x512 timed alone
(CUDA events, L2 flushed before every launch) against its max(FLOP / peak, bytes / bandwidth) floor; the whole
512x512 -> 2048x2048 forward in frames/s at F = 8 and F = 30 frames per call against the ~6.6 ms per frame floor
computed from the same shapes; and walk(upsample=True) frames/s with PNG files (host PNG encoding included; for
information).  Prints one JSON document; `--out FILE` also writes it there.

    python tools/esrgan_bench.py [--frames 8 30] [--iters 10] [--walk-frames 16] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from stable_diffusion_videos_b200 import _native as n  # noqa: E402

PEAK_TFLOPS, PEAK_GBS = 1440.7, 6564.5  # sustained fp16 tensor rate and HBM bandwidth measured on the B200 (SURVEY.md)
# (name, Cin, N, residual reads): FLOP/px = 2 * 9 * Cin * N; bytes/px = 2 * (Cin + N + residual channels)
SHAPES = [("conv1", 64, 32, 0), ("conv2", 96, 32, 0), ("conv3", 128, 32, 0), ("conv4", 160, 32, 0),
          ("conv5", 192, 64, 64)]


def floor_s(flop, nbytes):
    t_c, t_m = flop / (PEAK_TFLOPS * 1e12), nbytes / (PEAK_GBS * 1e9)
    return max(t_c, t_m), "tensor" if t_c >= t_m else "memory"


def forward_floor_s(H=512, W=512, nf=64, g=32, blocks=23):
    """sum of per-conv floors of one frame: the 69 dense blocks, conv_body, the two folded up-convs, conv_hr, conv_last"""
    P = H * W
    t = 0.0
    for _, cin, nn, r in SHAPES:
        t += blocks * 3 * floor_s(2 * 9 * cin * nn * P, 2 * (cin + nn + r) * P)[0]
    t += floor_s(2 * 9 * nf * nf * P, 2 * 3 * nf * P)[0]                           # conv_body (+ feat)
    t += floor_s(2 * 4 * nf * nf * 4 * P, 2 * (nf + 4 * nf) * P)[0]                # conv_up1: 4 parities x 2x2 taps
    t += floor_s(2 * 4 * nf * nf * 16 * P, 2 * (4 * nf + 16 * nf) * P)[0]          # conv_up2
    t += floor_s(2 * 9 * nf * nf * 16 * P, 2 * 2 * nf * 16 * P)[0]                 # conv_hr
    t += floor_s(2 * 9 * nf * 3 * 16 * P, (2 * nf + 3) * 16 * P)[0]                # conv_last (uint8 out)
    return t


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


def bench_shapes(F, iters):
    H = W = 512
    ld = 192
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    buf = (torch.randn(F, H, W, ld, device="cuda") * 0.5).half()
    dst = torch.empty_like(buf)
    out = []
    for name, cin, nn, r in SHAPES:
        w = (torch.randn(nn, cin, 3, 3, device="cuda") * (9 * cin) ** -0.5).half()
        wp = n.pack_weight(w)
        b = torch.randn(nn, device="cuda")
        d = n.GemmDesc()
        d.A = buf.data_ptr()
        d.C, d.W, d.H, d.B = cin, W, H, F
        d.sW, d.sH, d.sB = ld, ld * W, ld * W * H
        d.conv, d.Wt, d.N, d.bias = 1, wp.data_ptr(), nn, b.data_ptr()
        d.out, d.ldc = dst.data_ptr() + 2 * (cin if nn == 32 else 0), ld
        d.alpha = 0.2 if r else 1.0
        d.act = 0 if r else 2
        if r:
            d.resid, d.ldr = buf.data_ptr(), ld
        def timed():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
            for _ in range(2):
                n.gemm(d)
            for e0, e1 in ev:
                flush.zero_()
                e0.record()
                n.gemm(d)
                e1.record()
            torch.cuda.synchronize()
            return sorted(e0.elapsed_time(e1) for e0, e1 in ev)[iters // 2]

        ms = timed()
        alt = {}
        if nn == 32:  # A/B: the same GEMM on BLOCK_N = 64 tiles (half of each MMA and weight tile is padding)
            d.bn = 64
            alt["us_bn64"] = round(timed() * 1e3, 1)
            d.bn = 0
        P = F * H * W
        flop, nbytes = 2 * 9 * cin * nn * P, 2 * (cin + nn + r) * P
        fl, bound = floor_s(flop, nbytes)
        out.append(dict(shape=f"{name} {cin}->{nn}" + (" +res" if r else ""), frames=F, us=round(ms * 1e3, 1),
                        tflops=round(flop / ms / 1e9, 1), floor_us=round(fl * 1e6, 1), floor_bound=bound,
                        frac_of_floor=round(fl * 1e3 / ms, 3), **alt))
    del flush, buf, dst
    return out


def bench_forward(F, iters):
    from stable_diffusion_videos_b200 import RealESRGANModel

    m = RealESRGANModel.from_random(0, max_frames=F).to("cuda")
    e = m.engine(512, 512)
    x = torch.randint(0, 256, (F, 512, 512, 3), dtype=torch.uint8, device="cuda")
    y = torch.empty((F, 2048, 2048, 3), dtype=torch.uint8, device="cuda")
    for _ in range(2):
        e.forward(x, out=y)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        e.forward(x, out=y)
    torch.cuda.synchronize()
    s = (time.perf_counter() - t0) / iters
    fl = forward_floor_s()
    res = dict(frames_per_call=F, ms_per_call=round(s * 1e3, 2), frames_per_s=round(F / s, 2),
               ms_per_frame=round(s * 1e3 / F, 3), floor_ms_per_frame=round(fl * 1e3, 3),
               frac_of_floor=round(fl * F / s, 3), arena_gb=round(e.arena_bytes / 1e9, 2))
    lib = n.lib()
    import ctypes as C

    k = C.c_int()
    n.check(lib.sdw_esrgan_launches(e._h, C.byref(k)))
    res["launches_per_call"] = k.value
    del m, e, x, y
    torch.cuda.empty_cache()
    return res


def bench_walk(frames, batch):
    from stable_diffusion_videos_b200 import RealESRGANModel
    from stable_diffusion_videos_b200.configs import UNetConfig, VAEConfig
    from stable_diffusion_videos_b200.pipeline import StableDiffusionWalkPipeline

    pipe = StableDiffusionWalkPipeline.from_random(UNetConfig.sd14(), VAEConfig(), seed=0)
    pipe.upsampler = RealESRGANModel.from_random(0, max_frames=batch)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for up in (False, True):
            kw = dict(prompts=["a", "b"], seeds=[1, 2], num_interpolation_steps=frames, num_inference_steps=50,
                      height=512, width=512, batch_size=batch, make_video=False, upsample=up)
            pipe.walk(output_dir=tmp, name=f"warm{int(up)}", **dict(kw, num_interpolation_steps=batch))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe.walk(output_dir=tmp, name=f"run{int(up)}", **kw)
            torch.cuda.synchronize()
            out["upsample" if up else "plain"] = round(frames / (time.perf_counter() - t0), 3)
    return dict(frames=frames, batch_size=batch, steps=50, frames_per_s=out,
                note="SD-1.4 random weights, PNDM 50 steps, 512x512 PNGs (plain) vs 2048x2048 PNGs (upsample); "
                     "includes host PNG encoding")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, nargs="+", default=[8, 30])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--walk-frames", type=int, default=16, help="0 skips the walk measurement")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("esrgan_bench needs a CUDA GPU")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    res = dict(gpu=gpu_info(), peaks=dict(tflops=PEAK_TFLOPS, gbs=PEAK_GBS),
               shapes=bench_shapes(8, a.iters),
               forward=[bench_forward(F, a.iters) for F in a.frames])
    if a.walk_frames:
        res["walk"] = bench_walk(a.walk_frames, 8)
    res["gpu_after"] = gpu_info()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
