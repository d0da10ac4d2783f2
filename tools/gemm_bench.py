"""Micro-benchmark of the tcgen05 implicit-GEMM kernel on representative SD-1.4 shapes (CUDA events, warm).
Prints TFLOP/s per shape; used to steer kernel work and to produce profiles/*_gemm_shapes.txt."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stable_diffusion_videos_b200 import _native as n  # noqa: E402


def bench(B, H, W, C, N, conv, iters=20, bn=0, ver=0, epi=False, nsub=0, tr=0):
    x = torch.randn(B, H, W, C, device="cuda").half()
    k = 3 if conv else 1
    w = (torch.randn(N, C, k, k, device="cuda") * (C * k * k) ** -0.5).half()
    wp = n.pack_weight(w)
    out = torch.empty(B, H, W, N, device="cuda", dtype=torch.float16)
    d = n.GemmDesc()
    d.A = x.data_ptr(); d.C, d.W, d.H, d.B = C, W, H, B
    d.sW, d.sH, d.sB = C, W * C, H * W * C
    d.conv = 1 if conv else 0
    d.Wt = wp.data_ptr(); d.N = N
    d.out = out.data_ptr(); d.ldc = N
    d.alpha = 1.0; d.bn = bn; d.ver = ver; d.nsub = nsub; d.tr = tr
    if epi:  # bias + residual epilogue, as the ResBlock conv2 / attention out-projections run
        bias = torch.randn(N, device="cuda")
        resid = torch.randn(B, H, W, N, device="cuda").half()
        d.bias = bias.data_ptr(); d.resid = resid.data_ptr(); d.ldr = N
    for _ in range(3):
        n.gemm(d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        n.gemm(d)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    flop = 2.0 * B * H * W * N * C * k * k
    return ms, flop / ms / 1e9


if __name__ == "__main__":
    F = int(os.environ.get("F", "8"))
    Bn = 2 * F
    shapes = [
        ("conv3x3 64x64 320->320", Bn, 64, 64, 320, 320, 1),
        ("conv3x3 64x64 640->320", Bn, 64, 64, 640, 320, 1),
        ("conv3x3 32x32 640->640", Bn, 32, 32, 640, 640, 1),
        ("conv3x3 16x16 1280->1280", Bn, 16, 16, 1280, 1280, 1),
        ("conv3x3 8x8 1280->1280", Bn, 8, 8, 1280, 1280, 1),
        ("conv3x3 8x8 2560->1280", Bn, 8, 8, 2560, 1280, 1),
        ("linear 64x64 320->2560 (geglu N)", Bn, 64, 64, 320, 2560, 0),
        ("linear 64x64 1280->320 (ff.out)", Bn, 64, 64, 1280, 320, 0),
        ("linear 32x32 640->1920 (qkv)", Bn, 32, 32, 640, 1920, 0),
        ("vae conv3x3 256x256 256->256", F, 256, 256, 256, 256, 1),
        ("vae conv3x3 512x512 128->128", F, 512, 512, 128, 128, 1),
    ]
    for name, B, H, W, C, N, conv in shapes:
        for ver in ((1, 2) if os.environ.get('BOTH') else (2,)):
            variants = ((0, 0, 0), (160, 1, 1), (256, 1, 1))
            if conv and W % 16 == 0 and H % 8 == 0:  # tr: 1 = per-tap activation tiles, 2 = tap-reuse mainloop
                variants = ((0, 0, 0), (0, 0, 1), (128, 1, 1), (128, 1, 2), (160, 1, 1), (160, 1, 2), (192, 1, 2),
                            (256, 1, 1), (256, 1, 2), (160, 2, 1))
            for bn, nsub, tr in variants:
                if ver == 1 and (bn in (192, 256) or tr == 2):  # CTA-pair-only tiles
                    continue
                for epi in (True,):
                    ms, tf = bench(B, H, W, C, N, conv, bn=bn, ver=ver, epi=epi, nsub=nsub, tr=tr)
                    print(f"{name:36s} B={B:3d} v{ver} bn={bn or 'auto':>4} nsub={nsub} tr={tr} "
                          f"epi={'bias+res' if epi else 'none':8s} {ms*1e3:9.1f} us {tf:8.1f} TFLOP/s", flush=True)
