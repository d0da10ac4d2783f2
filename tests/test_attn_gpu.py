"""GPU parity of the fused tcgen05 attention kernel (sdw_attention) against torch fp32 SDPA.
Tolerance: P is rounded to fp16 before the PV product and the output is rounded to fp16:
|err| <= 2^-8 * max|ref| + 1e-3 (calibrated in DESIGN.md §Parity)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(B, heads, Nq, Nk, d, seed=0, scale=1.0):
    from stable_diffusion_videos_b200 import _native as n

    g = torch.Generator().manual_seed(seed)
    Cc = heads * d
    q = (torch.randn(B, Nq, Cc, generator=g) * scale).half().cuda()
    k = (torch.randn(B, Nk, Cc, generator=g) * scale).half().cuda()
    v = torch.randn(B, Nk, Cc, generator=g).half().cuda()
    vt_ld = (Nk + 7) // 8 * 8
    vt = torch.zeros(B, heads, d, vt_ld, dtype=torch.float16, device="cuda")
    vt[..., :Nk] = v.reshape(B, Nk, heads, d).permute(0, 2, 3, 1)
    out = torch.full((B, Nq, Cc), float("nan"), dtype=torch.float16, device="cuda")
    n.check(n.lib().sdw_attention(n.ptr(q), C.c_int64(Cc), n.ptr(k), C.c_int64(Cc), n.ptr(vt), C.c_int64(vt_ld),
                                  B, Nq, Nk, heads, d, n.ptr(out), C.c_int64(Cc), n.stream_ptr()))
    torch.cuda.synchronize()
    qf = q.float().reshape(B, Nq, heads, d).transpose(1, 2)
    kf = k.float().reshape(B, Nk, heads, d).transpose(1, 2)
    vf = v.float().reshape(B, Nk, heads, d).transpose(1, 2)
    ref = torch.softmax(qf @ kf.transpose(-1, -2) * d ** -0.5, -1) @ vf
    ref = ref.transpose(1, 2).reshape(B, Nq, Cc)
    return out.float(), ref


@pytest.mark.parametrize("B,heads,Nq,Nk,d", [
    (2, 8, 256, 256, 40),     # SD-1.4 64x64-level head dim (padded to 48 in the MMA)
    (1, 8, 4096, 4096, 40),   # full 64x64 self-attention: 32 KV tiles, online softmax
    (2, 8, 1024, 77, 40),     # cross attention: one ragged KV tile
    (2, 8, 1024, 1024, 80),
    (2, 8, 256, 256, 160),    # BKV = 64 variant
    (2, 8, 64, 64, 160),      # 8x8 level: half-empty query tile
    (2, 4, 64, 64, 8),
    (2, 4, 64, 77, 16),
    (1, 5, 300, 300, 64),     # SD-2.1 head dim, ragged both ways
    (3, 2, 129, 200, 32),
])
def test_flash_attention_matches_sdpa(B, heads, Nq, Nk, d):
    out, ref = _run(B, heads, Nq, Nk, d)
    assert torch.isfinite(out).all()
    err = float((out - ref).abs().max())
    assert err <= 2.0 ** -8 * float(ref.abs().max()) + 1e-3, (err, float(ref.abs().max()))


def test_flash_attention_peaky_scores():
    """large logits: running-max rescale path must engage and stay finite."""
    out, ref = _run(1, 4, 512, 512, 40, seed=3, scale=4.0)
    assert torch.isfinite(out).all()
    assert float((out - ref).abs().max()) <= 2.0 ** -7 * float(ref.abs().max()) + 2e-3


@pytest.mark.parametrize("B,heads,Nq,Nk,d", [
    (1, 4, 300, 700, 40),     # ragged query block (second 128-row tile of the last pair partly empty) and ragged keys
    (1, 2, 128, 1000, 32),    # query tile B entirely out of range
    (2, 3, 576, 576, 64),     # SD-2.1 at 24x24: 2.25 query pairs, 4.5 KV tiles
    (1, 2, 2048, 2048, 16),
    (3, 8, 1024, 1024, 40),   # several work items per CTA (persistent loop, Q refill, barrier phases across items)
])
def test_two_tile_kernel_rising_max_and_ragged(B, heads, Nq, Nk, d):
    """attn_pp_kernel: keys scaled so that the row max keeps rising along the KV loop (lazy rescale engages late too)."""
    from stable_diffusion_videos_b200 import _native as n

    g = torch.Generator().manual_seed(5)
    Cc = heads * d
    q = torch.randn(B, Nq, Cc, generator=g).half().cuda()
    k = (torch.randn(B, Nk, Cc, generator=g) * torch.linspace(0.2, 3.0, Nk)[None, :, None]).half().cuda()
    v = torch.randn(B, Nk, Cc, generator=g).half().cuda()
    vt_ld = (Nk + 7) // 8 * 8
    vt = torch.zeros(B, heads, d, vt_ld, dtype=torch.float16, device="cuda")
    vt[..., :Nk] = v.reshape(B, Nk, heads, d).permute(0, 2, 3, 1)
    out = torch.full((B, Nq, Cc), float("nan"), dtype=torch.float16, device="cuda")
    n.check(n.lib().sdw_attention(n.ptr(q), C.c_int64(Cc), n.ptr(k), C.c_int64(Cc), n.ptr(vt), C.c_int64(vt_ld),
                                  B, Nq, Nk, heads, d, n.ptr(out), C.c_int64(Cc), n.stream_ptr()))
    torch.cuda.synchronize()
    qf = q.float().reshape(B, Nq, heads, d).transpose(1, 2)
    kf = k.float().reshape(B, Nk, heads, d).transpose(1, 2)
    vf = v.float().reshape(B, Nk, heads, d).transpose(1, 2)
    ref = (torch.softmax(qf @ kf.transpose(-1, -2) * d ** -0.5, -1) @ vf).transpose(1, 2).reshape(B, Nq, Cc)
    assert torch.isfinite(out).all()
    err = float((out.float() - ref).abs().max())
    assert err <= 2.0 ** -8 * float(ref.abs().max()) + 1e-3, (err, float(ref.abs().max()))
