"""GPU parity tests of the tcgen05 implicit-GEMM kernel (sdw_gemm) against torch fp32 references.

Tolerance: inputs are fp16, accumulation fp32, output rounded once to fp16 -> |err| <= 2^-9 * max|ref| + 1e-3
(the per-kernel bound of SURVEY.md §8d).
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as Fn

pytestmark = pytest.mark.gpu


def _native():
    from stable_diffusion_videos_b200 import _native as n
    return n


def _tol(ref):
    return float(ref.abs().max()) * 2.0 ** -9 + 1e-3


def run_conv(x_nhwc, w_oihw, conv, bias=None, rowvec=None, resid=None, act=0, bn=0, mode=0, N_out=None, ver=0, nsub=0, ew=0, tr=0, et=0, out_buf=None, out_c0=0):
    """x: [B,H,W,C] fp16 cuda; returns NHWC fp16 output computed by the native kernel."""
    n = _native()
    B, H, W, Cc = x_nhwc.shape
    N = w_oihw.shape[0]
    wp = n.pack_weight_up4(w_oihw) if conv == 3 else n.pack_weight(w_oihw, geglu=(mode == 1))
    if conv == 2:
        OH, OW = H // 2, W // 2
    elif conv == 3:
        OH, OW = 2 * H, 2 * W
    else:
        OH, OW = H, W
    ncols = N // 2 if mode == 1 else N
    if out_buf is None:
        out = torch.full((B, OH, OW, ncols), float("nan"), dtype=torch.float16, device="cuda")
    else:  # channel slice [out_c0, out_c0 + ncols) of a wider NHWC buffer (the skip-concat destinations)
        out = out_buf[..., out_c0:out_c0 + ncols]
    parities = [(0, 0), (0, 1), (1, 0), (1, 1)] if conv == 3 else [(0, 0)]
    for (py, px) in parities:
        d = n.GemmDesc()
        d.A = x_nhwc.data_ptr()
        d.C, d.W, d.H, d.B = Cc, W, H, B
        d.sW, d.sH, d.sB = x_nhwc.stride(2), x_nhwc.stride(1), x_nhwc.stride(0)
        d.conv = conv
        d.up_px, d.up_py = px, py
        d.Wt = wp[py * 2 + px].data_ptr() if conv == 3 else wp.data_ptr()
        d.N = N
        d.bias = bias.data_ptr() if bias is not None else None
        if rowvec is not None:
            d.rowvec = rowvec.data_ptr()
            d.rowvec_ld = rowvec.shape[1]
        if resid is not None:
            d.resid = resid.data_ptr()
            d.ldr = resid.shape[-1]
        d.out = out.data_ptr()
        d.ldc = out.stride(2)
        d.mode = mode
        d.act = act
        d.alpha = 1.0
        d.bn = bn
        d.ver = ver
        d.nsub = nsub
        d.ew = ew
        d.tr = tr
        d.et = et
        n.gemm(d)
    torch.cuda.synchronize()
    return out


def ref_conv(x_nhwc, w, conv, bias=None, rowvec=None, resid=None, act=0):
    x = x_nhwc.float().permute(0, 3, 1, 2)
    wf = w.float()
    if conv == 0:
        y = Fn.conv2d(x, wf.reshape(wf.shape[0], wf.shape[1], 1, 1))
    elif conv == 1:
        y = Fn.conv2d(x, wf, padding=1)
    elif conv == 2:
        y = Fn.conv2d(x, wf, stride=2, padding=1)
    else:
        y = Fn.conv2d(Fn.interpolate(x, scale_factor=2.0, mode="nearest"), wf, padding=1)
    if bias is not None:
        y = y + bias.float()[None, :, None, None]
    if rowvec is not None:
        y = y + rowvec.float()[:, :, None, None]
    if act == 1:
        y = Fn.silu(y)
    y = y.permute(0, 2, 3, 1)
    if resid is not None:
        y = y + resid.float()
    return y


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.float16).cuda()


@pytest.mark.parametrize("M,N,K,bn", [(128, 128, 64, 128), (300, 320, 320, 0), (77 * 2, 640, 768, 128),
                                       (2, 1280, 320, 0), (1024, 64, 128, 64), (512, 512, 512, 256),
                                       (8192, 320, 2880, 160)])
def test_linear(M, N, K, bn):
    x = _rand(1, 1, M, K, seed=1)
    w = _rand(N, K, scale=K ** -0.5, seed=2)
    bias = _rand(N, seed=3).float()
    out = run_conv(x, w, 0, bias=bias, bn=bn)
    ref = ref_conv(x, w, 0, bias=bias)
    err = (out.float() - ref).abs().max().item()
    assert torch.isfinite(out.float()).all()
    assert err <= _tol(ref), (err, _tol(ref))


@pytest.mark.parametrize("B,H,W,Cc,N", [(2, 16, 16, 64, 128), (2, 8, 8, 320, 320), (1, 64, 64, 320, 320),
                                         (3, 4, 4, 128, 64), (2, 32, 32, 192, 160), (4, 2, 2, 64, 64),
                                         (2, 1, 1, 64, 64), (1, 24, 24, 64, 64)])
def test_conv3x3(B, H, W, Cc, N):
    x = _rand(B, H, W, Cc, seed=4)
    w = _rand(N, Cc, 3, 3, scale=(9 * Cc) ** -0.5, seed=5)
    bias = _rand(N, seed=6).float()
    rowvec = _rand(B, N, seed=7).float()
    out = run_conv(x, w, 1, bias=bias, rowvec=rowvec)
    ref = ref_conv(x, w, 1, bias=bias, rowvec=rowvec)
    err = (out.float() - ref).abs().max().item()
    assert torch.isfinite(out.float()).all()
    assert err <= _tol(ref), (err, _tol(ref))


def test_conv3x3_residual_silu():
    x = _rand(2, 16, 16, 128, seed=8)
    w = _rand(128, 128, 3, 3, scale=(9 * 128) ** -0.5, seed=9)
    resid = _rand(2, 16, 16, 128, seed=10)
    out = run_conv(x, w, 1, resid=resid, act=1)
    ref = ref_conv(x, w, 1, resid=resid, act=1)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


@pytest.mark.parametrize("B,H,W,Cc,N", [(2, 16, 16, 64, 128), (1, 64, 64, 320, 320), (2, 2, 2, 64, 64)])
def test_conv3x3_stride2(B, H, W, Cc, N):
    x = _rand(B, H, W, Cc, seed=11)
    w = _rand(N, Cc, 3, 3, scale=(9 * Cc) ** -0.5, seed=12)
    bias = _rand(N, seed=13).float()
    out = run_conv(x, w, 2, bias=bias)
    ref = ref_conv(x, w, 2, bias=bias)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


@pytest.mark.parametrize("B,H,W,Cc,N", [(2, 8, 8, 64, 128), (1, 32, 32, 128, 128), (2, 1, 1, 64, 64)])
def test_upsample_conv3x3(B, H, W, Cc, N):
    x = _rand(B, H, W, Cc, seed=14)
    w = _rand(N, Cc, 3, 3, scale=(9 * Cc) ** -0.5, seed=15)
    bias = _rand(N, seed=16).float()
    out = run_conv(x, w, 3, bias=bias)
    ref = ref_conv(x, w, 3, bias=bias)
    assert torch.isfinite(out.float()).all()
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


def test_geglu():
    M, K, Ch = 256, 128, 256  # Linear(K -> 2*Ch), out = a * gelu(g)
    x = _rand(1, 1, M, K, seed=17)
    w = _rand(2 * Ch, K, scale=K ** -0.5, seed=18)
    bias = _rand(2 * Ch, seed=19).float()
    n = _native()
    # bias must follow the same row interleave as the packed weight
    blk = torch.arange(2 * Ch, device="cuda")
    b64, within = blk // 64, blk % 64
    src = torch.where(within < 32, b64 * 32 + within, Ch + b64 * 32 + within - 32)
    out = run_conv(x, w, 0, bias=bias[src].contiguous(), mode=1)
    h = x.float().reshape(M, K) @ w.float().t() + bias
    a, g = h.chunk(2, dim=-1)
    ref = (a * Fn.gelu(g)).reshape(1, 1, M, Ch)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


def test_qkv_vt_and_batched_attention_matmuls():
    """QKV projection with V^T scatter, then S = Q K^T and O = P V as head-batched matmuls."""
    n = _native()
    Bn, Ntok, Cc, heads = 2, 256, 128, 4
    d = Cc // heads
    x = _rand(Bn, 1, Ntok, Cc, seed=20)
    wqkv = _rand(3 * Cc, Cc, scale=Cc ** -0.5, seed=21)
    wp = n.pack_weight(wqkv)
    qk = torch.zeros((Bn, Ntok, 2 * Cc), dtype=torch.float16, device="cuda")
    vt = torch.zeros((Bn, heads, d, Ntok), dtype=torch.float16, device="cuda")
    g = n.GemmDesc()
    g.A = x.data_ptr(); g.C, g.W, g.H, g.B = Cc, Ntok, 1, Bn
    g.sW, g.sH, g.sB = Cc, Ntok * Cc, Ntok * Cc
    g.Wt = wp.data_ptr(); g.N = 3 * Cc
    g.out = qk.data_ptr(); g.ldc = 2 * Cc
    g.mode = 2; g.alpha = 1.0
    g.vt_col0, g.vt_d, g.vt_heads, g.vt_ntok = 2 * Cc, d, heads, Ntok
    g.vt = vt.data_ptr(); g.vt_ld = Ntok
    n.gemm(g)
    torch.cuda.synchronize()
    ref = x.float().reshape(Bn, Ntok, Cc) @ wqkv.float().t()
    q_ref, k_ref, v_ref = ref.split(Cc, dim=-1)
    assert (qk.float() - torch.cat([q_ref, k_ref], -1)).abs().max().item() <= _tol(ref)
    vt_ref = v_ref.reshape(Bn, Ntok, heads, d).permute(0, 2, 3, 1)
    assert (vt.float() - vt_ref).abs().max().item() <= _tol(ref)

    # S[b,h] = Q[b,:,h,:] K[b,:,h,:]^T * d^-0.5 : lattice (C=d, W=tok, H=heads, B=b)
    S = torch.zeros((Bn, heads, Ntok, Ntok), dtype=torch.float16, device="cuda")
    g = n.GemmDesc()
    g.A = qk.data_ptr(); g.C, g.W, g.H, g.B = d, Ntok, heads, Bn
    g.sW, g.sH, g.sB = 2 * Cc, d, Ntok * 2 * Cc
    g.Wt = qk.data_ptr() + Cc * 2; g.N = Ntok; g.ldb = 2 * Cc; g.Kb = d
    g.b_batched = 1; g.sBh = d; g.sBb = Ntok * 2 * Cc
    g.out = S.data_ptr(); g.ldc = Ntok
    g.o_sW, g.o_sH, g.o_sB = Ntok, Ntok * Ntok, heads * Ntok * Ntok
    g.alpha = d ** -0.5
    n.gemm(g)
    torch.cuda.synchronize()
    q = qk[..., :Cc].float().reshape(Bn, Ntok, heads, d).permute(0, 2, 1, 3)
    k = qk[..., Cc:].float().reshape(Bn, Ntok, heads, d).permute(0, 2, 1, 3)
    S_ref = q @ k.transpose(-1, -2) * d ** -0.5
    assert (S.float() - S_ref).abs().max().item() <= _tol(S_ref)

    # O[b, tok, h*d + :] = P[b,h] V[b,h]  with P = softmax(S) (torch), V^T from the scatter above
    P = torch.softmax(S.float(), -1).to(torch.float16).contiguous()
    O = torch.zeros((Bn, Ntok, Cc), dtype=torch.float16, device="cuda")
    g = n.GemmDesc()
    g.A = P.data_ptr(); g.C, g.W, g.H, g.B = Ntok, Ntok, heads, Bn
    g.sW, g.sH, g.sB = Ntok, Ntok * Ntok, heads * Ntok * Ntok
    g.Wt = vt.data_ptr(); g.N = d; g.ldb = Ntok; g.Kb = Ntok
    g.b_batched = 1; g.sBh = d * Ntok; g.sBb = heads * d * Ntok
    g.out = O.data_ptr(); g.ldc = Cc
    g.o_sW, g.o_sH, g.o_sB = Cc, d, Ntok * Cc
    g.alpha = 1.0; g.bn = 64
    n.gemm(g)
    torch.cuda.synchronize()
    O_ref = (P.float() @ vt.float().transpose(-1, -2)).permute(0, 2, 1, 3).reshape(Bn, Ntok, Cc)
    assert (O.float() - O_ref).abs().max().item() <= _tol(O_ref)


# ---- the persistent 2-CTA (cta_group::2) kernel, forced ------------------------------------------------------
@pytest.mark.parametrize("M,N,K,bn", [(256, 256, 64, 256), (300, 320, 320, 160), (8192, 320, 2880, 160),
                                       (128, 128, 128, 128), (4096, 2560, 320, 0), (1000, 640, 1280, 0),
                                       (77 * 4, 1280, 768, 256), (20000, 512, 512, 256)])
def test_linear_2cta(M, N, K, bn):
    x = _rand(1, 1, M, K, seed=31)
    w = _rand(N, K, scale=K ** -0.5, seed=32)
    bias = _rand(N, seed=33).float()
    out = run_conv(x, w, 0, bias=bias, bn=bn, ver=2)
    ref = ref_conv(x, w, 0, bias=bias)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))


@pytest.mark.parametrize("B,H,W,Cc,N,conv", [(2, 16, 16, 64, 128, 1), (4, 64, 64, 320, 320, 1), (2, 8, 8, 320, 320, 1),
                                              (3, 4, 4, 128, 256, 1), (2, 32, 32, 192, 160, 1), (1, 24, 24, 64, 128, 1),
                                              (2, 16, 16, 64, 128, 2), (2, 64, 64, 320, 320, 2), (2, 8, 8, 64, 128, 3),
                                              (1, 32, 32, 128, 128, 3)])
def test_conv_2cta(B, H, W, Cc, N, conv):
    x = _rand(B, H, W, Cc, seed=34)
    w = _rand(N, Cc, 3, 3, scale=(9 * Cc) ** -0.5, seed=35)
    bias = _rand(N, seed=36).float()
    rowvec = _rand(B, N, seed=37).float() if conv == 1 else None
    resid = None
    out = run_conv(x, w, conv, bias=bias, rowvec=rowvec, ver=2)
    ref = ref_conv(x, w, conv, bias=bias, rowvec=rowvec)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))


def test_conv_residual_2cta_many_tiles():
    """more tiles than clusters: exercises the persistent loop, TMEM double buffering and barrier phase wrap."""
    x = _rand(8, 64, 64, 128, seed=38)
    w = _rand(256, 128, 3, 3, scale=(9 * 128) ** -0.5, seed=39)
    resid = _rand(8, 64, 64, 256, seed=40)
    bias = _rand(256, seed=41).float()
    out = run_conv(x, w, 1, bias=bias, resid=resid, ver=2, bn=128)
    ref = ref_conv(x, w, 1, bias=bias, resid=resid)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


def test_geglu_2cta():
    M, K, Ch = 1024, 320, 1280
    x = _rand(1, 1, M, K, seed=42)
    w = _rand(2 * Ch, K, scale=K ** -0.5, seed=43)
    bias = _rand(2 * Ch, seed=44).float()
    blk = torch.arange(2 * Ch, device="cuda")
    b64, within = blk // 64, blk % 64
    src = torch.where(within < 32, b64 * 32 + within, Ch + b64 * 32 + within - 32)
    out = run_conv(x, w, 0, bias=bias[src].contiguous(), mode=1, ver=2)
    h = x.float().reshape(M, K) @ w.float().t() + bias
    a, g = h.chunk(2, dim=-1)
    ref = (a * Fn.gelu(g)).reshape(1, 1, M, Ch)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


# ---- two accumulators per activation tile (256 x 320 tiles, single-buffered TMEM) --------------------------------
@pytest.mark.parametrize("B,H,W,Cc,N,conv", [(4, 64, 64, 320, 320, 1), (2, 32, 32, 640, 640, 1), (2, 16, 16, 128, 1280, 1),
                                              (1, 8, 8, 64, 480, 1), (2, 64, 64, 64, 320, 2), (2, 16, 16, 64, 640, 3),
                                              (1, 1, 5000, 1280, 960, 0)])
def test_gemm_2cta_two_accumulators(B, H, W, Cc, N, conv):
    x = _rand(B, H, W, Cc, seed=51)
    k = 3 if conv else 1
    w = _rand(N, Cc, k, k, scale=(k * k * Cc) ** -0.5, seed=52)
    bias = _rand(N, seed=53).float()
    oh, ow = (H // 2, W // 2) if conv == 2 else ((2 * H, 2 * W) if conv == 3 else (H, W))
    resid = _rand(B, oh, ow, N, seed=54)
    out = run_conv(x, w, conv, bias=bias, resid=resid, ver=2, bn=160, nsub=2)
    ref = ref_conv(x, w if conv else w.reshape(N, Cc), conv, bias=bias, resid=resid)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))


# ---- tap reuse: one 10-row activation box per (channel chunk, kx) feeds the three ky taps of a 3x3 stride-1 conv ---------
@pytest.mark.parametrize("B,H,W,Cc,N,bn,nsub", [(4, 64, 64, 320, 320, 160, 1), (2, 32, 32, 640, 640, 256, 1), (2, 16, 16, 128, 1280, 256, 1),
                                                 (3, 16, 16, 64, 480, 128, 1), (1, 8, 16, 72, 200, 192, 1),
                                                 (1, 128, 128, 128, 128, 128, 1), (1, 24, 48, 104, 320, 0, 0)])
def test_gemm_conv3x3_tap_reuse(B, H, W, Cc, N, bn, nsub):
    x = _rand(B, H, W, Cc, seed=71)
    w = _rand(N, Cc, 3, 3, scale=(9 * Cc) ** -0.5, seed=72)
    bias = _rand(N, seed=73).float()
    resid = _rand(B, H, W, N, seed=74)
    out = run_conv(x, w, 1, bias=bias, resid=resid, ver=2, bn=bn, nsub=nsub, tr=2)
    ref = ref_conv(x, w, 1, bias=bias, resid=resid)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))
    # and it must agree with the per-tap mainloop to accumulation-order noise
    out1 = run_conv(x, w, 1, bias=bias, resid=resid, ver=2, bn=bn, nsub=nsub, tr=1)
    assert (out.float() - out1.float()).abs().max().item() <= _tol(ref)


def test_gemm_tap_reuse_strided_input():
    """input view = channel slice of a wider NHWC buffer (skip-concat destination), SiLU epilogue"""
    big = _rand(2, 32, 32, 704, seed=75)
    x = big[..., 64:704]
    w = _rand(320, 640, 3, 3, scale=(9 * 640) ** -0.5, seed=76)
    bias = _rand(320, seed=77).float()
    out = run_conv(x, w, 1, bias=bias, act=1, ver=2, tr=2)
    ref = ref_conv(x, w, 1, bias=bias, act=1)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


# ---- TMA epilogue: bias in shared memory, residual through a TMA-fed ring, output slabs through TMA stores ---------------
@pytest.mark.parametrize("B,H,W,Cc,N,conv,bn,act,res", [
    (1, 1, 5000, 320, 320, 0, 160, 0, True),     # token lattice, ragged last tile, residual (attention out-projection)
    (1, 1, 4096, 1280, 320, 0, 0, 0, True),      # ff.out
    (2, 32, 32, 640, 640, 0, 160, 0, True),      # 1x1 conv on an image lattice (proj_out)
    (2, 16, 16, 128, 1280, 0, 256, 1, False),    # SiLU, no residual, BLOCK_N 256
    (3, 8, 8, 64, 200, 0, 128, 0, True),         # batch-folded tiles (bb = 2), ragged N, odd tile count
    (2, 64, 64, 64, 320, 2, 160, 0, True),       # stride-2 conv
    (2, 16, 16, 64, 640, 3, 160, 0, True),       # folded upsample: parity-scattered stores + residual reads
    (4, 64, 64, 320, 320, 1, 160, 0, True),      # 3x3 with tap reuse and the TMA epilogue together
    (1, 1, 300, 64, 768, 0, 192, 0, False),
])
def test_gemm_tma_epilogue(B, H, W, Cc, N, conv, bn, act, res):
    x = _rand(B, H, W, Cc, seed=81)
    k = 3 if conv else 1
    w = _rand(N, Cc, k, k, scale=(k * k * Cc) ** -0.5, seed=82)
    bias = _rand(N, seed=83).float()
    oh, ow = (H // 2, W // 2) if conv == 2 else ((2 * H, 2 * W) if conv == 3 else (H, W))
    resid = _rand(B, oh, ow, N, seed=84) if res else None
    out = run_conv(x, w, conv, bias=bias, resid=resid, act=act, ver=2, bn=bn, et=2)
    ref = ref_conv(x, w if conv else w.reshape(N, Cc), conv, bias=bias, resid=resid, act=act)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))
    out1 = run_conv(x, w, conv, bias=bias, resid=resid, act=act, ver=2, bn=bn, et=1)
    assert (out.float() - out1.float()).abs().max().item() <= _tol(ref)


def test_gemm_tma_epilogue_concat_slice_and_no_bias():
    """output = channel slice of a wider buffer; neighbours must stay untouched (TMA clipping at the column extent)"""
    x = _rand(2, 32, 32, 320, seed=85)
    w = _rand(320, 320, 1, 1, scale=320 ** -0.5, seed=86)
    buf = torch.full((2, 32, 32, 960), 7.0, dtype=torch.float16, device="cuda")
    out = run_conv(x, w, 0, ver=2, et=2, out_buf=buf, out_c0=320)
    ref = ref_conv(x, w.reshape(320, 320), 0)
    assert (out.float() - ref).abs().max().item() <= _tol(ref)
    assert (buf[..., :320] == 7.0).all() and (buf[..., 640:] == 7.0).all()


@pytest.mark.parametrize("M,K,Ch", [(1024, 320, 1280), (900, 640, 2560), (256, 1280, 5120)])
def test_geglu_tma_epilogue(M, K, Ch):
    x = _rand(1, 1, M, K, seed=87)
    w = _rand(2 * Ch, K, scale=K ** -0.5, seed=88)
    bias = _rand(2 * Ch, seed=89).float()
    blk = torch.arange(2 * Ch, device="cuda")
    b64, within = blk // 64, blk % 64
    src = torch.where(within < 32, b64 * 32 + within, Ch + b64 * 32 + within - 32)
    out = run_conv(x, w, 0, bias=bias[src].contiguous(), mode=1, ver=2, et=2)
    h = x.float().reshape(M, K) @ w.float().t() + bias
    a, g = h.chunk(2, dim=-1)
    ref = (a * Fn.gelu(g)).reshape(1, 1, M, Ch)
    assert torch.isfinite(out.float()).all()
    assert (out.float() - ref).abs().max().item() <= _tol(ref)


@pytest.mark.parametrize("Bn,Ntok,Cc,heads,et", [(2, 300, 320, 8, 2), (2, 300, 320, 8, 1), (3, 1024, 640, 8, 2), (1, 256, 1280, 8, 2)])
def test_qkv_vt_tma_epilogue(Bn, Ntok, Cc, heads, et):
    """fused QKV projection: Q|K columns through TMA row slabs, V columns transposed in shared memory -> V^T."""
    n = _native()
    d = Cc // heads
    ld = (Ntok + 7) // 8 * 8
    x = _rand(Bn, 1, Ntok, Cc, seed=91)
    wqkv = _rand(3 * Cc, Cc, scale=Cc ** -0.5, seed=92)
    bias = _rand(3 * Cc, seed=93).float()
    wp = n.pack_weight(wqkv)
    qk = torch.full((Bn, Ntok, 2 * Cc), 3.0, dtype=torch.float16, device="cuda")
    vt = torch.full((Bn, heads, d, ld), 5.0, dtype=torch.float16, device="cuda")
    g = n.GemmDesc()
    g.A = x.data_ptr(); g.C, g.W, g.H, g.B = Cc, Ntok, 1, Bn
    g.sW, g.sH, g.sB = Cc, Ntok * Cc, Ntok * Cc
    g.Wt = wp.data_ptr(); g.N = 3 * Cc
    g.bias = bias.data_ptr()
    g.out = qk.data_ptr(); g.ldc = 2 * Cc
    g.mode = 2; g.alpha = 1.0; g.ver = 2; g.et = et
    g.vt_col0, g.vt_d, g.vt_heads, g.vt_ntok = 2 * Cc, d, heads, Ntok
    g.vt = vt.data_ptr(); g.vt_ld = ld
    n.gemm(g)
    torch.cuda.synchronize()
    ref = x.float().reshape(Bn, Ntok, Cc) @ wqkv.float().t() + bias
    q_ref, k_ref, v_ref = ref.split(Cc, dim=-1)
    assert (qk.float() - torch.cat([q_ref, k_ref], -1)).abs().max().item() <= _tol(ref)
    vt_ref = v_ref.reshape(Bn, Ntok, heads, d).permute(0, 2, 3, 1)
    assert (vt[..., :Ntok].float() - vt_ref).abs().max().item() <= _tol(ref)
    # TMA clips the contiguous (token) extent at 16-byte granularity: the row padding up to the next multiple of 8 tokens
    # may receive finite filler values (sdwalk.h documents this); it must never be NaN / inf
    assert torch.isfinite(vt.float()).all()


# ---- epilogue width: 2 or 4 warps per TMEM lane quarter (the 640-thread kernel of the short-K GEMMs) --------------------
@pytest.mark.parametrize("ew", [2, 4])
@pytest.mark.parametrize("T,Cc,N,bn,mode,res", [
    (20000, 320, 960, 256, 0, False),     # QKV-like, 4 N tiles, ragged last M pair
    (19200, 320, 2560, 256, 1, False),    # GEGLU: one 64-column chunk per warp and tile
    (24000, 320, 640, 160, 0, True),      # residual ring, five 32-column chunks over four warps
    (19000, 64, 512, 128, 0, True),       # one K chunk
    (19000, 448, 480, 160, 0, False),     # seven K chunks, ragged last N tile (480 = 3 x 160)
    (40000, 320, 960, 0, 0, True),        # several tiles per cluster, auto BLOCK_N
    (9000, 1280, 320, 192, 0, True),      # ff.out-like: 20 K blocks
    (300, 320, 320, 160, 0, True),        # fewer tiles than clusters
])
def test_gemm_epilogue_width(T, Cc, N, bn, mode, res, ew):
    x = _rand(1, 1, T, Cc, seed=95)
    w = _rand(N, Cc, scale=Cc ** -0.5, seed=96)
    bias = _rand(N, seed=97).float()
    ncols = N // 2 if mode == 1 else N
    resid = _rand(1, 1, T, ncols, seed=98) if res else None
    if mode == 1:
        blk = torch.arange(N, device="cuda")
        b64, within = blk // 64, blk % 64
        src = torch.where(within < 32, b64 * 32 + within, ncols + b64 * 32 + within - 32)
        out = run_conv(x, w, 0, bias=bias[src].contiguous(), mode=1, ver=2, bn=bn, et=2, ew=ew)
        h = x.float().reshape(T, Cc) @ w.float().t() + bias
        a, g = h.chunk(2, dim=-1)
        ref = (a * Fn.gelu(g)).reshape(1, 1, T, ncols)
    else:
        out = run_conv(x, w.reshape(N, Cc, 1, 1), 0, bias=bias, resid=resid, ver=2, bn=bn, et=2, ew=ew)
        ref = ref_conv(x, w, 0, bias=bias, resid=resid)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(ref), (err, _tol(ref))
