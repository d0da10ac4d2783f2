"""plan_gemm decisions for the SD-1.4 layer shapes, checked without a GPU (plan-only mode: tensor maps are validated, not
encoded).  These pin the choices the measurements in profiles/ justified: tap reuse for 3x3 stride-1 convs, the TMA
epilogue wherever it is eligible, the shared-memory budget behind the pipeline depth."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def native():
    from stable_diffusion_videos_b200 import _native

    lib = _native.lib()
    lib.sdw_debug_plan_only(1)
    yield _native
    lib.sdw_debug_plan_only(0)


def _plan(n, B, H, W, Cc, N, conv, mode=0, resid=True, rowvec_ld=None, **kw):
    d = n.GemmDesc()
    base = 1 << 30  # fake, 16-byte aligned device addresses: nothing is dereferenced in plan-only mode
    d.A = base
    d.C, d.W, d.H, d.B = Cc, W, H, B
    d.sW, d.sH, d.sB = Cc, W * Cc, H * W * Cc
    d.conv = conv
    d.Wt = base + (1 << 28)
    d.N = N
    d.bias = base + (2 << 28)
    ncols = N // 2 if mode == 1 else N
    if resid:
        d.resid = base + (3 << 28)
        d.ldr = ncols
    if rowvec_ld is not None:
        d.rowvec = base + (5 << 28)
        d.rowvec_ld = rowvec_ld
    d.out = base + (4 << 28)
    d.ldc = ncols
    d.mode = mode
    d.alpha = 1.0
    for k, v in kw.items():
        setattr(d, k, v)
    out = (C.c_int32 * 12)()
    n.check(n.lib().sdw_debug_plan(C.byref(d), out))
    keys = ("ver", "bn", "nsub", "ew", "tr", "epi_tma", "nstages", "reserved", "grid", "bw", "bh", "bb")
    return dict(zip(keys, list(out)))


def test_conv3x3_uses_tap_reuse_and_cta_pairs(native):
    for (B, hw, c, nn) in [(32, 64, 320, 320), (60, 64, 640, 320), (32, 32, 640, 640), (32, 16, 1280, 1280), (16, 512, 128, 128)]:
        p = _plan(native, B, hw, hw, c, nn, 1)
        assert p["ver"] == 2 and p["tr"] == 1 and (p["bw"], p["bh"], p["bb"]) == (16, 8, 1), p
        assert p["bn"] in (128, 160, 192) and p["nsub"] == 1, p   # BLOCK_N 256 gains nothing with 3-tap stages
        assert p["grid"] == 148 and p["nstages"] >= 3, p
    # 8x8 level: two samples per tile, no tap reuse (geometry needs W % 16 == 0)
    p = _plan(native, 32, 8, 8, 1280, 1280, 1)
    assert p["tr"] == 0 and (p["bw"], p["bh"], p["bb"]) == (8, 8, 2), p


def test_tma_epilogue_is_the_default_where_eligible(native):
    p = _plan(native, 1, 1, 131072, 320, 320, 0)                       # attention out-projection + residual
    assert p["epi_tma"] == 1 and p["ver"] == 2 and p["bn"] == 160, p
    p = _plan(native, 1, 1, 131072, 320, 2560, 0, mode=1, resid=False)  # GEGLU
    assert p["epi_tma"] == 1 and p["bn"] == 256 and p["nstages"] >= 3, p
    p = _plan(native, 32, 64, 64, 320, 320, 1, rowvec_ld=0)            # conv1 of a ResBlock: time-embedding row, same for all samples
    assert p["epi_tma"] == 1, p
    p = _plan(native, 32, 64, 64, 320, 320, 1, rowvec_ld=320)          # per-sample row vector: classic epilogue
    assert p["epi_tma"] == 0, p
    p = _plan(native, 1, 1, 4096, 320, 320, 0, et=1)
    assert p["epi_tma"] == 0, p


def test_small_problems_fall_back_to_the_single_cta_kernel(native):
    p = _plan(native, 1, 1, 64, 320, 320, 0)      # one M tile
    assert p["ver"] == 1, p
    p = _plan(native, 1, 1, 4096, 320, 64, 0, resid=False)  # N < 128
    assert p["ver"] == 1 and p["bn"] == 64, p


def test_shared_memory_budget_bounds_the_pipeline_depth(native):
    # stages x (A + B) + epilogue buffers + barriers must fit 227 KB - 1 KB alignment slack
    for (conv, c, nn, mode, resid) in [(1, 320, 320, 0, True), (0, 320, 2560, 1, False), (0, 1280, 320, 0, True),
                                       (0, 320, 960, 0, False), (1, 2560, 1280, 0, True)]:
        hw = 64 if c <= 640 else 16
        p = _plan(native, 32, hw, hw, c, nn, conv, mode=mode, resid=resid)
        a = 20480 if p["tr"] else 16384
        b = (3 if p["tr"] else 1) * p["nsub"] * (p["bn"] // 2) * 128
        epi = ((32768 + 16384 + (65536 if resid else 0)) if p["ew"] == 4 else (32768 + 8192 + (32768 if resid else 0))) if p["epi_tma"] else 16384
        assert 2 <= p["nstages"] <= 8 and p["nstages"] * (a + b) + epi + 1024 <= 227 * 1024 - 1024, p


def test_opt_in_variants_are_refused_outside_their_domain(native):
    with pytest.raises(native.SdwError):
        _plan(native, 32, 8, 8, 1280, 1280, 1, tr=2)          # tap reuse needs W % 16 == 0
    with pytest.raises(native.SdwError):
        _plan(native, 32, 64, 64, 320, 320, 1, ew=4)           # the 16-warp epilogue belongs to the per-tap kernels
    with pytest.raises(native.SdwError):
        _plan(native, 32, 64, 64, 320, 320, 1, nsub=2, tr=2)   # two accumulators need the per-tap mainloop
    with pytest.raises(native.SdwError):
        _plan(native, 1, 1, 4096, 320, 320, 0, ver=1, bn=256)  # BLOCK_N 256 is a CTA-pair tile
    p = _plan(native, 1, 1, 131072, 320, 2560, 0, mode=1, resid=False, ew=4)
    assert p["ew"] == 4 and p["epi_tma"] == 1 and p["grid"] == 148, p
    p = _plan(native, 1, 1, 131072, 320, 2560, 0, mode=1, resid=False)      # short K: chosen automatically
    assert p["ew"] == 4, p
    p = _plan(native, 1, 1, 131072, 320, 2560, 0, mode=1, resid=False, ew=2)
    assert p["ew"] == 2, p


def _attn(n, B, Nq, Nk, heads, d):
    out = (C.c_int32 * 5)()
    n.check(n.lib().sdw_debug_attention_plan(B, Nq, Nk, heads, d, out))
    return dict(zip(("variant", "qt", "gx", "gy", "gz"), list(out)))


def test_attention_variants_for_the_sd14_head_dims(native):
    # head dims <= 64 with more than one KV tile: the two-query-tile persistent kernel (variants 8-11, one CTA per SM);
    # 80: the BKV = 64 P-in-TMEM tile; 160: double-buffered S
    assert _attn(native, 32, 4096, 4096, 8, 40)["variant"] == 10
    assert _attn(native, 32, 4096, 160, 8, 40)["variant"] == 10
    assert _attn(native, 32, 1024, 1024, 8, 80)["variant"] == 4
    assert _attn(native, 32, 256, 256, 8, 160)["variant"] == 5
    assert _attn(native, 16, 9216, 9216, 5, 64)["variant"] == 11   # SD-2.1, 96x96 latent
    assert _attn(native, 32, 4096, 77, 8, 40)["variant"] == 10      # single KV tile, >= 2 query tiles: the two-tile kernel too
    assert _attn(native, 32, 128, 77, 8, 40)["variant"] == 2        # one query tile: the one-tile kernel
    p = _attn(native, 32, 4096, 4096, 8, 40)
    assert (p["qt"], p["gx"], p["gy"], p["gz"]) == (2, 148, 1, 1)   # persistent: 148 CTAs over 32 * 8 * 16 work items
    p = _attn(native, 1, 576, 576, 5, 64)                           # fewer work items than SMs
    assert (p["gx"], p["gy"], p["gz"]) == (15, 1, 1)


def test_cross_attention_plans(native):
    p = _attn(native, 32, 1024, 77, 8, 80)     # head dim 80: BKV = 64, so 77 keys are two KV tiles — no query-tile loop
    assert p["variant"] == 4 and p["qt"] == 1 and p["gx"] == 8
    p = _attn(native, 32, 128, 77, 8, 40)      # one query tile: attn_fwd_kernel, all keys in one KV tile
    assert p["variant"] == 2 and p["gx"] * p["qt"] * 128 >= 128
    p = _attn(native, 32, 4096, 77, 8, 40)     # head dim 40: persistent two-tile kernel, one work item = 256 queries
    assert (p["variant"], p["qt"], p["gx"]) == (10, 2, 148)
    with pytest.raises(native.SdwError):
        _attn(native, 1, 64, 64, 1, 512)        # the VAE's d = 512 goes through the unfused path
