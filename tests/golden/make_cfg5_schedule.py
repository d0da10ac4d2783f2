"""BASELINE.json configs[4] ("audio-driven walk (examples/make_music_video.py), 30 fps x 10 s"): the interpolation
schedule T the walk follows, computed from the reference's own fixture tests/samples/choice.wav (22 050 Hz mono, 10 s;
tests/test_pipeline.py:53-68) with this package's librosa-free `get_timesteps_arr` restatement and the example's
arguments (fps 30, margin 1.0, smooth 0.2, offset 0, duration 10 — examples/make_music_video.py:43-55).

The clip's PCM samples are committed as cfg5_choice_wav.npz (sr, int16 samples); T is computed from them.  Given the
path of a choice.wav, the script first refreshes cfg5_choice_wav.npz from it.
PARITY UNPINNED against librosa (not installable here): the fixture pins the restatement against regressions.

    python tests/golden/make_cfg5_schedule.py [path/to/choice.wav]
"""
import importlib.util
import os
import sys
import tempfile

import numpy as np
from scipy.io import wavfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CLIP = os.path.join(HERE, "cfg5_choice_wav.npz")


def schedule(wav):
    spec = importlib.util.spec_from_file_location("sdw_audio", os.path.join(ROOT, "stable-diffusion-videos_b200", "audio.py"))
    audio = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(audio)
    return audio.get_timesteps_arr(wav, offset=0, duration=10, fps=30, margin=1.0, smooth=0.2)


if __name__ == "__main__":
    if len(sys.argv) > 1:
        sr, samples = wavfile.read(sys.argv[1])
        np.savez_compressed(CLIP, sr=np.int32(sr), samples=samples)
    clip = np.load(CLIP)
    with tempfile.TemporaryDirectory() as tmp:
        wav = os.path.join(tmp, "choice.wav")
        wavfile.write(wav, int(clip["sr"]), clip["samples"])
        T = schedule(wav)
    np.save(os.path.join(HERE, "cfg5_choice_T.npy"), T.astype(np.float64))
    print(T.shape, T[:5], T[-3:], "monotone:", bool(np.all(np.diff(T) >= 0)))
