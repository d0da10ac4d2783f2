"""Golden fixture of the 4x Real-ESRGAN upsampler (RealESRGAN_x4plus architecture, 23 RRDB blocks), generated with the
fp32 ORACLE (oracle/esrgan.py), plus the tolerance calibration the native path is held to: the same oracle with
fp16-storage emulation (every conv output and block exit rounded to fp16 — what an fp16 pipeline stores), whose spread
against the fp32 oracle is the yardstick.  Run from the repo root (about a minute on 8 cores):

    python tests/golden/make_golden_esrgan.py

Input: the committed cfg1_frames_u8.npy (2 frames of 64x64).  Weights: configs.esrgan_random_state_dict(seed 0), fp16
as stored.  Output esrgan_x4plus_f2.npz: uint8 frames [2, 256, 256, 3] and the fp32 pre-clamp output at every
RAW_STRIDE-th row and column (fp32: fp16 rounding of the stored reference alone would use half the tolerance);
calibration in esrgan_calibration.json.
"""
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from oracle import esrgan as OE  # noqa: E402

CASE = "esrgan_x4plus_f2"
RAW_STRIDE = 2


def inputs():
    from stable_diffusion_videos_b200.configs import ESRGANConfig, esrgan_random_state_dict

    frames = np.load(os.path.join(HERE, "cfg1_frames_u8.npy"))
    sd = esrgan_random_state_dict(ESRGANConfig(), 0)
    return frames, sd


def spread(a, b):
    (fa, ra), (fb, rb) = a, b
    d = np.abs(fa.astype(np.int32) - fb.astype(np.int32))
    return {
        "raw_rel_l2": float(np.linalg.norm(ra - rb) / np.linalg.norm(rb)),
        "raw_max_abs_over_max": float(np.abs(ra - rb).max() / np.abs(rb).max()),
        "frames_mean_lsb": float(d.mean()), "frames_frac_within_2": float((d <= 2).mean()),
        "frames_p999_lsb": float(np.quantile(d, 0.999)), "frames_max_lsb": int(d.max()),
    }


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    frames, sd = inputs()
    sd32 = {k: v.float() for k, v in sd.items()}
    t0 = time.time()
    ref = OE.enhance(sd32, frames)
    t1 = time.time()
    emu = OE.enhance(sd32, frames, store=lambda t: t.half().float())
    ref = (ref[0], ref[1][:, ::RAW_STRIDE, ::RAW_STRIDE])
    emu = (emu[0], emu[1][:, ::RAW_STRIDE, ::RAW_STRIDE])
    u8, raw = ref
    sat = float(np.mean((u8 == 0) | (u8 == 255)))
    np.savez_compressed(os.path.join(HERE, CASE + ".npz"), frames=u8, raw=raw.astype(np.float32))
    cal = {}
    cal[CASE] = dict(spread(emu, ref), oracle_seconds=round(t1 - t0, 1), saturated_frac=sat,
                     raw_range=[float(raw.min()), float(raw.max())],
                     note="fp16-storage-emulated oracle vs fp32 oracle, same fp16-rounded weights")
    with open(os.path.join(HERE, "esrgan_calibration.json"), "w") as f:
        json.dump(cal, f, indent=1, sort_keys=True)
    print(CASE, json.dumps(cal[CASE]))


if __name__ == "__main__":
    main()
