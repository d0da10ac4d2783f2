#!/usr/bin/env python
"""bench.py — frames/sec of the latent-walk hot path (BASELINE.json metric) on N B200s.

  python bench.py --gpus 1 --steps K --warmup W             native arm (libsdwalk.so)
  python bench.py --impl reference ...                       the reference's CPU path (oracle restatement), rank 0
  torchrun --nproc-per-node N bench.py --gpus N ...          one rank per GPU, frames sharded, NCCL gather
  python bench.py ... --dump-outputs DIR                     also write the last timed step's frames to DIR/frames.npy

Workload (config.workload): BASELINE.json configs[1] — SD-1.4 architecture, 512x512, fp16, PNDM 50 steps
(51 UNet calls), classifier-free guidance 7.5, frames interpolated between 2 synthetic prompts; random-init weights
and synthetic prompt embeddings (no network).  A *step* = one sample call of F frames through
slerp/lerp inputs -> 51 x {UNet, CFG, scheduler step} -> VAE decode -> uint8 frames.  Frames are independent and
cost-identical, so frames/s on K*F frames is the throughput of the 60-frame clip.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernels the roofline block names, taken from committed
# `ncu --set full` captures (profiles/roofline_traffic.json: bytes, the batch of the capture, the raw page they come from)
def _traffic(kernel, batch):
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))[kernel]
        return {"bytes": t["bytes"] * batch / t["batch"], "source": f"ncu capture {t['source']} at batch {t['batch']}, "
                                                                   f"scaled to batch {batch}"}
    except Exception:
        return {"bytes": None, "source": "no capture committed"}


FLOP_PER_FRAME = {"sd14": 2 * 51 * 0.8033e12 + 2.5145e12}  # SURVEY.md §8d algorithmic FLOPs (84.45 T)
UNET_FLOP_B1 = 0.8033e12
VAE_FLOP = 2.5145e12


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1440.7), d.get("hbm_gbs", 6564.5), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max((int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()), default=0)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference_leg(steps, warmup, budget_s=150.0):
    """time the oracle (restated diffusers CPU path, fp32) on a bounded sample: up to `steps` batch-2 UNet forwards at
    the 64x64 latent (after up to `warmup` untimed ones) + ONE VAE decode, all host cores; frame time = 51 * t_unet +
    t_vae (frames are cost-identical).  The sample stops early once `budget_s` of CPU time is spent; the number of
    forwards that really ran is reported."""
    import torch

    from oracle.unet import UNet2DConditionModel, UNetConfig
    from oracle.vae import AutoencoderKLDecoder, VAEConfig

    # BASELINE.md §3: all host cores, whatever OMP_NUM_THREADS the launcher exported (torchrun sets it to 1).  "All cores" =
    # the PHYSICAL cores this process may run on: with one thread per hyper-thread (os.cpu_count() = 128 on the GPU box) the
    # same forward took 88 s instead of 7.6 s (profiles/r02_bench_F30_db_attention.json vs BENCH_r01)
    try:
        import psutil

        physical = psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        physical = max(1, (os.cpu_count() or 2) // 2)
    try:
        physical = min(physical, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    threads = max(1, physical)
    torch.set_num_threads(threads)
    threads = torch.get_num_threads()
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.sd14()).eval()
    vae = AutoencoderKLDecoder(VAEConfig()).eval()
    x = torch.randn(2, 4, 64, 64)
    ctx = torch.randn(2, 77, 768)
    z = torch.randn(1, 4, 64, 64)
    with torch.no_grad():
        t_begin = time.perf_counter()
        warm_run = 0
        for _ in range(max(0, warmup)):
            unet(x, torch.tensor(981), ctx)
            warm_run += 1
            if time.perf_counter() - t_begin > budget_s / 4:
                break
        t0 = time.perf_counter()
        steps_run = 0
        for _ in range(max(1, steps)):
            unet(x, torch.tensor(981), ctx)
            steps_run += 1
            if time.perf_counter() - t_begin > budget_s:
                break
        t_unet = (time.perf_counter() - t0) / steps_run
        t0 = time.perf_counter()
        vae.decode(z)
        t_vae = time.perf_counter() - t0
    spf = 51 * t_unet + t_vae
    return {"value": 1.0 / spf, "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"{steps_run} timed (+{warm_run} warm-up) batch-2 UNet forwards (64x64 latent, fp32) + 1 VAE decode "
                      f"on {threads} threads; s/frame = 51*{t_unet:.3f} + {t_vae:.3f} = {spf:.1f}",
            "s_per_frame": spf, "t_unet_s": t_unet, "t_vae_s": t_vae, "steps_run": steps_run, "warmup_run": warm_run}


DUMP_BYTES = 64_000_000  # at most this much in --dump-outputs DIR


def dump_outputs(out_dir, frames):
    """Write the uint8 frames [n, H, W, 3] a timed step returned as out_dir/frames.npy in float32.  When all n frames
    exceed DUMP_BYTES, a fixed sample of whole frames is written: indices drawn without replacement by numpy's
    default_rng(0), ascending.  Returns the indices written."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    x = frames.cpu().numpy()
    n, keep = x.shape[0], (DUMP_BYTES - 128) // (x[0].size * 4)  # 128: the .npy header
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    np.save(os.path.join(out_dir, "frames.npy"), x[idx].astype(np.float32))
    return idx


def _stdout_to_stderr():
    """Route fd 1 to stderr while the benchmark runs: libraries (NCCL prints its version line from C) must not put
    anything on stdout next to the ONE JSON line."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _restore_stdout(saved):
    import ctypes

    sys.stdout.flush()
    try:
        ctypes.CDLL(None).fflush(None)  # C stdio buffers (NCCL's printf) drain to stderr, not into the JSON stream
    except Exception:
        pass
    os.dup2(saved, 1)
    os.close(saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--frames-per-call", type=int, default=int(os.environ.get("SDW_BENCH_F", "30")))
    ap.add_argument("--inference-steps", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames of the last one to DIR/frames.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    saved_stdout = _stdout_to_stderr()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    workload = ("SD-1.4 UNet+VAE, 512x512, fp16, PNDM 50 steps (51 UNet calls), CFG 7.5, 2 prompts x 60 interp "
                "frames (BASELINE configs[1]); random-init weights, synthetic embeddings")

    if a.impl == "reference":
        if rank != 0:
            return
        leg = cpu_reference_leg(max(1, a.steps), a.warmup)
        _restore_stdout(saved_stdout)
        print(json.dumps({
            "impl": "reference", "metric": "frames/sec at 512x512 50-step SD-1.4", "value": leg["value"],
            "unit": "frames/s", "n_gpus": a.gpus, "steps": leg["steps_run"], "warmup": leg["warmup_run"],
            "ms_per_step": leg["t_unet_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": workload, "reference_arm": leg["sample"],
                                            "step": "one batch-2 UNet forward of the restated diffusers CPU path; "
                                                    "frames/s = 1 / (51 x step + VAE decode)"},
            "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": leg["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    import torch.distributed as dist

    from stable_diffusion_videos_b200 import _native
    from stable_diffusion_videos_b200.configs import UNetConfig, VAEConfig
    from stable_diffusion_videos_b200.parallel import broadcast_state_dict, gather_frames, init_distributed
    from stable_diffusion_videos_b200.pipeline import StableDiffusionWalkPipeline

    rank, world, local = init_distributed()
    assert world == a.gpus or world == 1, f"--gpus {a.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    F, K, W = a.frames_per_call, a.steps, a.warmup

    # ---- model: random-init SD-1.4; rank 0 generates, one NCCL broadcast ships the weights -------------------
    from stable_diffusion_videos_b200.configs import random_state_dict, unet_param_shapes, vae_param_shapes
    from stable_diffusion_videos_b200.pipeline import NativeUNet, NativeVAE, SyntheticTextEncoder, SyntheticTokenizer
    from stable_diffusion_videos_b200.schedulers import PNDMScheduler

    ucfg, vcfg = UNetConfig.sd14(), VAEConfig()
    if rank == 0 or world == 1:
        usd = {k: v.to(dev) for k, v in random_state_dict(unet_param_shapes(ucfg), 0).items()}
        vsd = {k: v.to(dev) for k, v in random_state_dict(vae_param_shapes(vcfg), 1).items()}
    else:
        usd = {k: torch.empty(s, dtype=torch.float16, device=dev) for k, s in unet_param_shapes(ucfg).items()}
        vsd = {k: torch.empty(s, dtype=torch.float16, device=dev) for k, s in vae_param_shapes(vcfg).items()}
    usd, vsd = broadcast_state_dict(usd), broadcast_state_dict(vsd)
    pipe = StableDiffusionWalkPipeline(NativeVAE(vcfg, vsd), SyntheticTextEncoder(768), SyntheticTokenizer(),
                                       NativeUNet(ucfg, usd), PNDMScheduler()).to(dev)
    h = w = 64
    eng = pipe._engine(h, w, F, True)
    del usd, vsd
    pipe.unet.state, pipe.vae.state = None, None
    eng.set_scheduler(pipe.scheduler, a.inference_steps, 7.5)
    eng._plan_key = pipe._plan_key(a.inference_steps, 7.5)
    n_unet_calls = eng.n_steps

    # ---- inputs: one clip's worth of interpolated (embedding, latent) pairs, resident on the device ------------
    n_clip = max(F * (K + W), 60)
    ea, eb = pipe.embed_text("0"), pipe.embed_text("1")
    la, lb = pipe.init_noise(42, (1, 4, h, w), ea.dtype), pipe.init_noise(1337, (1, 4, h, w), ea.dtype)
    T = torch.linspace(0, 1, n_clip, device=dev)
    lat_all, emb_all = _native.slerp_lerp_batch(la, lb, ea, eb, T)
    unc = pipe._uncond([""])
    # per-rank offset so ranks render different frames (weak scaling: per-GPU work fixed)
    def batch(i):
        j = ((rank * 7 + i) * F) % (n_clip - F + 1)
        return lat_all[j:j + F], emb_all[j:j + F]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_step(i, gather=True):
        lat, emb = batch(i)
        u8 = eng.sample(lat, emb, unc, use_graph=not a.no_graph)
        if world > 1 and gather:
            u8 = gather_frames(u8, F * world)  # decoded frames to rank 0 over NCCL (None on the other ranks)
        return u8

    for i in range(W):
        run_step(i)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(K):
        out = run_step(W + i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        idx = dump_outputs(a.dump_outputs, out)
        print(f"dump: frames {idx.tolist()} of {out.shape[0]} of timed step {K} -> "
              f"{os.path.join(a.dump_outputs, 'frames.npy')}", file=sys.stderr)
    frames_total = K * F * world
    value = frames_total / (ms / 1e3)

    # ---- e2e: the public call (pipeline.__call__) with HOST inputs: H2D of latents+embeddings, D2H of frames ------
    lat_h = [batch(i)[0].cpu().pin_memory() for i in range(K + 1)]
    emb_h = [batch(i)[1].cpu().pin_memory() for i in range(K + 1)]
    pipe(latents=lat_h[K], text_embeddings=emb_h[K], num_inference_steps=a.inference_steps, guidance_scale=7.5, output_type="pil")
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        out = pipe(latents=lat_h[i], text_embeddings=emb_h[i], num_inference_steps=a.inference_steps,
                   guidance_scale=7.5, output_type="pil")
        assert len(out["images"]) == F
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    e2e_val = frames_total / e2e_s
    h2d = F * (4 * h * w + 77 * 768) * 2
    d2h = F * 512 * 512 * 3

    # ---- walk()-level throughput: the call users make (P:556), PNG files included (frame sink: pinned async D2H + workers)
    walk_leg = None
    if world == 1:
        import shutil
        import tempfile

        tmp = tempfile.mkdtemp(prefix="sdw_bench_walk_")
        n_walk = F * min(K, 3)
        kw = dict(output_dir=tmp, num_inference_steps=a.inference_steps, guidance_scale=7.5, batch_size=F, make_video=False)
        pipe.walk(["0", "1"], seeds=[42, 1337], num_interpolation_steps=F, name="warm", **kw)  # same engine shape, warm
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipe.walk(["0", "1"], seeds=[42, 1337], num_interpolation_steps=n_walk, name="timed", **kw)
        torch.cuda.synchronize()
        t_walk = time.perf_counter() - t0
        n_png = len([f for f in os.listdir(os.path.join(tmp, "timed", "timed_000000")) if f.endswith(".png")])
        assert n_png == n_walk, (n_png, n_walk)
        walk_leg = {"value": n_walk / t_walk, "unit": "frames/s", "frames": n_walk,
                    "note": "StableDiffusionWalkPipeline.walk(make_video=False): embed_text + init_noise + slerp/lerp + "
                            "sampler + D2H + PNG files on disk (tmpfs-independent: written under the system temp dir)"}
        shutil.rmtree(tmp, ignore_errors=True)

    # ---- rooflines, measured live at this run's UNet batch (2F), each kernel alone with L2 flushed between launches,
    #      CUDA events on the launch stream
    kern = None
    if rank == 0:
        import ctypes as C

        Bn = 2 * F
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

        def timed(fn, warm=2, reps=6):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                k0.record()
                fn()
                k1.record()
                torch.cuda.synchronize()
                tot += k0.elapsed_time(k1)
            return tot / reps * 1e3  # us

        # (1) dominant kernel by share of the step: self-attention at the 64x64 level (8 heads x 40)
        Cc, Nt = 320, 4096
        qa = torch.randn(Bn, Nt, Cc, device=dev).half()
        ka = torch.randn(Bn, Nt, Cc, device=dev).half()
        vta = torch.randn(Bn, 8, 40, Nt, device=dev).half()
        oa = torch.empty(Bn, Nt, Cc, device=dev, dtype=torch.float16)
        attn_us = timed(lambda: _native.check(_native.lib().sdw_attention(
            _native.ptr(qa), C.c_int64(Cc), _native.ptr(ka), C.c_int64(Cc), _native.ptr(vta), C.c_int64(Nt), Bn, Nt, Nt, 8,
            40, _native.ptr(oa), C.c_int64(Cc), _native.stream_ptr())))
        attn_flop = 4.0 * Bn * 8 * Nt * Nt * 40
        attn_exps = float(Bn) * 8 * Nt * Nt
        del qa, ka, vta, oa
        # (2) the 64x64-level ResBlock conv3x3 (320 -> 320, bias + residual): the tensor-bound GEMM family
        xk = torch.randn(Bn, 64, 64, 320, device=dev).half()
        wk = _native.pack_weight((torch.randn(320, 320, 3, 3, device=dev) * (2880 ** -0.5)).half())
        bk = torch.randn(320, device=dev)
        rk = torch.randn(Bn, 64, 64, 320, device=dev).half()
        ok = torch.empty(Bn, 64, 64, 320, device=dev, dtype=torch.float16)
        d = _native.GemmDesc()
        d.A = xk.data_ptr(); d.C, d.W, d.H, d.B = 320, 64, 64, Bn
        d.sW, d.sH, d.sB = 320, 64 * 320, 64 * 64 * 320
        d.conv = 1; d.Wt = wk.data_ptr(); d.N = 320
        d.bias = bk.data_ptr(); d.resid = rk.data_ptr(); d.ldr = 320
        d.out = ok.data_ptr(); d.ldc = 320; d.alpha = 1.0
        conv_us = timed(lambda: _native.gemm(d))
        kern = {"name": "gemm2_tc_kernel<160, tap-reuse> conv3x3 64x64 320->320 bias+residual", "batch": Bn,
                "flop_per_launch": 2.0 * Bn * 64 * 64 * 320 * 2880, "us_per_launch": conv_us}
        # (3) the short-K transformer linears (HBM / epilogue bound): attention out-projection 320 -> 320 + residual
        T = Bn * 4096
        wl = _native.pack_weight((torch.randn(320, 320, 1, 1, device=dev) * (320 ** -0.5)).half())
        dl = _native.GemmDesc()
        xl = xk.view(T, 320)
        dl.A = xl.data_ptr(); dl.C, dl.W, dl.H, dl.B = 320, T, 1, 1
        dl.sW = 320
        dl.Wt = wl.data_ptr(); dl.N = 320
        dl.bias = bk.data_ptr(); dl.resid = rk.data_ptr(); dl.ldr = 320
        dl.out = ok.data_ptr(); dl.ldc = 320; dl.alpha = 1.0
        lin_us = timed(lambda: _native.gemm(dl))
        lin_bytes = 2.0 * T * 320 * 3 + 2.0 * 320 * 320  # activations in, residual in, out; weights once
        del xk, wk, rk, ok, wl, flush

    if rank != 0:
        return
    peak_tf, peak_gbs, peak_src = _peaks()
    burst_tf = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops", 1736.7) \
        if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1590.0
    k_ach = kern["flop_per_launch"] / (kern["us_per_launch"] * 1e-6) / 1e12
    attn_tf = attn_flop / (attn_us * 1e-6) / 1e12
    # exponential floor of the attention kernel: one ex2 per score at 16 / clk / SM.  The kernel is timed ALONE (it then
    # runs near the maximum SM clock, not at the power-capped clock of the sampler), so the floor is taken at sm_max_mhz —
    # the smallest floor, i.e. xu_frac is a lower bound of how close the kernel is to it
    sm_hz = (clk["sm_max_mhz"] if clk and clk.get("sm_max_mhz") else 1965) * 1e6
    xu_floor_us = attn_exps / (16.0 * 148 * sm_hz) * 1e6
    tr_attn, tr_conv = _traffic("attention_self_64x64_d40", 2 * F), _traffic("conv3x3_64x64_320", 2 * F)
    achieved_tf = value * FLOP_PER_FRAME["sd14"] / 1e12 / world
    pro, per_step, vae_l = eng.launches()
    launches_per_call = pro + 1 + n_unet_calls * (per_step + 1) + vae_l
    res = {
        "metric": "frames/sec at 512x512 50-step SD-1.4", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": workload, "frames_per_step": F, "unet_calls_per_frame": n_unet_calls,
                   "unet_batch": 2 * F, "parallelism": f"frame-dp{world}", "cuda_graph": not a.no_graph,
                   "l2": "working set per step (1.8 GB weights + activations) exceeds the 126 MB L2"},
        "roofline": {
            "bound": "tensor", "achieved": attn_tf, "peak": burst_tf, "unit": "TFLOP/s", "frac": attn_tf / burst_tf,
            "traffic": tr_attn["bytes"], "traffic_source": tr_attn["source"],
            "kernel": "attn_pp_kernel self-attention 64x64, 8 heads x 40 (dominant kernel by share of the step)",
            "kernel_batch": 2 * F, "us_per_launch": attn_us,
            "xu_floor_us": xu_floor_us, "xu_frac": xu_floor_us / attn_us,
            "note": f"timed alone, L2 flushed between launches, vs {peak_src} burst fp16/bf16 peak; this kernel is bound by "
                    "one exponential per score (MUFU.EX2, 16/clk/SM; the kernel moves a quarter of them to the FMA pipe): "
                    "xu_frac = all-MUFU exponential floor at the maximum SM clock / time",
            "conv3x3": {"kernel": kern["name"], "kernel_batch": kern["batch"], "us_per_launch": kern["us_per_launch"],
                        "bound": "tensor", "achieved": k_ach, "peak": burst_tf, "unit": "TFLOP/s", "frac": k_ach / burst_tf,
                        "traffic": tr_conv["bytes"], "traffic_source": tr_conv["source"]},
            "short_k_linear": {"kernel": "gemm2_tc_kernel attention out-projection 64x64 320->320 bias+residual",
                               "kernel_batch": 2 * F, "us_per_launch": lin_us, "bound": "hbm",
                               "achieved": lin_bytes / (lin_us * 1e-6) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                               "frac": lin_bytes / (lin_us * 1e-6) / 1e9 / peak_gbs,
                               "note": "algorithmic bytes (activations in + residual in + out + weights) / time"},
            "whole_sampler": {"achieved": achieved_tf, "peak": peak_tf, "frac": achieved_tf / peak_tf, "unit": "TFLOP/s",
                              "note": "frames x 84.45 TFLOP / time / gpus vs sustained peak"}},
        "e2e": {"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches_per_call * K,
        "clocks": clk,
    }
    if walk_leg:
        res["walk"] = walk_leg
    if not a.no_cpu_baseline and world == 1:
        res["cpu_baseline"] = {k: v for k, v in cpu_reference_leg(2, 1).items()
                               if k in ("value", "unit", "cores", "kind", "sample")}
    _restore_stdout(saved_stdout)
    print(json.dumps(res), flush=True)
    saved_stdout = _stdout_to_stderr()  # teardown chatter stays off stdout too
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
