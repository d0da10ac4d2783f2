"""The librosa-free audio schedule (stable-diffusion-videos_b200/audio.py; reference utils.py:12-39 via librosa).
PARITY UNPINNED (no librosa in the image, no golden schedule in the reference): construction properties only."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def audio():
    spec = importlib.util.spec_from_file_location("sdw_audio", os.path.join(ROOT, "stable-diffusion-videos_b200", "audio.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _clicks(sr=22050, seconds=4.0, at=(0.5, 1.0, 3.0, 3.2, 3.4, 3.6)):
    rng = np.random.default_rng(0)
    t = np.arange(int(sr * seconds)) / sr
    y = 0.2 * np.sin(2 * np.pi * 220.0 * t)               # a steady tone: harmonic, must not drive the schedule
    for c in at:
        i = int(c * sr)
        if i + 256 > len(y):
            continue
        y[i:i + 256] += rng.standard_normal(256) * np.hanning(256) * 0.9   # broadband clicks: percussive
    return y.astype(np.float32)


def test_stft_shapes_and_istft_round_trip(audio):
    y = _clicks()
    D = audio.stft(y)
    assert D.shape == (1025, 1 + len(y) // 512) and D.dtype == np.complex64
    # cross-check one frame against a direct DFT of the windowed, centred segment
    k = 37
    seg = np.concatenate([np.zeros(1024, np.float32), y])[k * 512:k * 512 + 2048]
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(2048) / 2048)
    assert np.allclose(D[:, k], np.fft.rfft(seg * w), atol=1e-3)
    yr = audio.istft(D, length=len(y))
    assert yr.shape == y.shape and np.abs(yr - y).max() < 1e-4   # Hann at hop n_fft/4 is a perfect-reconstruction pair


def test_mel_filterbank_slaney(audio):
    fb = audio.mel_filterbank()
    assert fb.shape == (128, 1025) and (fb >= 0).all()
    assert np.allclose(audio.mel_to_hz(audio.hz_to_mel([0.0, 440.0, 1000.0, 4000.0, 11025.0])), [0, 440, 1000, 4000, 11025])
    assert abs(float(audio.hz_to_mel(1000.0)) - 15.0) < 1e-9        # the Slaney scale's linear / log knee
    peak = fb.argmax(axis=1)
    assert (np.diff(peak) >= 0).all() and peak[0] <= 3 and peak[-1] >= 900   # bands ordered, spanning 0 .. sr/2
    # equal-area (Slaney) normalisation: every triangle integrates to ~1 over frequency (bin width sr / n_fft)
    area = fb.sum(axis=1) * (22050 / 2048)
    assert np.allclose(area[5:-1], 1.0, rtol=0.15)


def test_hpss_separates_tone_from_clicks(audio):
    y = _clicks()
    D = audio.stft(y)
    H, P = audio.hpss(D)
    assert H.shape == D.shape == P.shape
    # margin 1: the soft masks sum to one, so harmonic + percussive reconstructs the input
    assert np.abs((H + P) - D).max() < 1e-3 * np.abs(D).max()
    tone_bin = int(round(220.0 * 2048 / 22050))
    quiet = slice(150, 210)                                           # frames between clicks (t ~ 1.7 .. 2.4 s)
    assert np.abs(H[tone_bin, quiet]).mean() > 20 * np.abs(P[tone_bin, quiet]).mean()   # the tone is harmonic
    click_frame = int(0.5 * 22050 / 512)
    hi = slice(200, 1000)
    assert np.abs(P[hi, click_frame]).mean() > 3 * np.abs(H[hi, click_frame]).mean()      # the click is percussive
    with pytest.raises(ValueError):
        audio.hpss(D, margin=0.5)


def test_schedule_is_monotone_and_follows_the_percussion(audio, tmp_path):
    from scipy.io import wavfile

    y = _clicks(seconds=4.0)
    path = tmp_path / "clicks.wav"
    wavfile.write(path, 22050, (y * 32767).astype(np.int16))
    fps, duration = 30, 4.0
    T = audio.get_timesteps_arr(path, offset=0.0, duration=duration, fps=fps)
    assert T.shape == (int(duration * fps),)
    assert T[0] >= 0.0 and abs(T[-1] - 1.0) < 1e-6 and (np.diff(T) >= -1e-12).all()
    # four of six clicks sit in 3.0 .. 3.6 s: the schedule must spend clearly more of its range there than in the silent 1.5 .. 2.5 s
    f = lambda s: int(s * fps)
    assert (T[f(3.8)] - T[f(2.9)]) > 3.0 * (T[f(2.5)] - T[f(1.5)])
    # smooth = 1 is a straight line; offsets / durations select the excerpt
    assert np.allclose(audio.get_timesteps_arr(path, 0.0, duration, fps=fps, smooth=1.0), np.linspace(0, 1, int(duration * fps)))
    T2 = audio.get_timesteps_arr(path, offset=2.5, duration=1.5, fps=fps)
    assert T2.shape == (45,) and (np.diff(T2) >= -1e-12).all()


def test_loader_formats_and_resampling(audio, tmp_path):
    from scipy.io import wavfile

    sr = 44100
    t = np.arange(sr) / sr
    stereo = np.stack([np.sin(2 * np.pi * 440 * t), np.sin(2 * np.pi * 440 * t)], axis=1).astype(np.float32)
    p = tmp_path / "stereo44k.wav"
    wavfile.write(p, sr, stereo)
    y, got_sr = audio.load(p, offset=0.25, duration=0.5)
    assert got_sr == 22050 and abs(len(y) - 11025) <= 2 and y.dtype == np.float32
    k = np.abs(np.fft.rfft(y * np.hanning(len(y)))).argmax() * 22050 / len(y)
    assert abs(k - 440.0) < 5.0                                       # the tone survives the down-mix + resampling


def test_package_entry_point_uses_the_restatement_without_librosa(tmp_path):
    pytest.importorskip("torch")
    from scipy.io import wavfile

    from stable_diffusion_videos_b200.utils import get_timesteps_arr

    path = tmp_path / "c.wav"
    wavfile.write(path, 22050, (_clicks(seconds=2.0) * 32767).astype(np.int16))
    T = get_timesteps_arr(path, offset=0, duration=2, fps=30, margin=1.0, smooth=0.2)
    assert T.shape == (60,) and abs(T[-1] - 1.0) < 1e-6 and (np.diff(T) > 0).all()


def test_cfg5_schedule_fixture(audio, tmp_path):
    """BASELINE configs[4]: T for the reference's own choice.wav with the example's arguments (fps 30, margin 1.0,
    smooth 0.2) is committed as tests/golden/cfg5_choice_T.npy, the clip's PCM samples as tests/golden/cfg5_choice_wav.npz;
    the restatement must reproduce T from that WAV, and T must be a valid schedule (300 frames, in [0, 1], non-decreasing,
    ends at 1)."""
    from scipy.io import wavfile

    T = np.load(os.path.join(ROOT, "tests", "golden", "cfg5_choice_T.npy"))
    assert T.shape == (300,) and T.dtype == np.float64
    assert T.min() >= 0.0 and abs(T[-1] - 1.0) < 1e-12 and np.all(np.diff(T) >= 0)
    clip = np.load(os.path.join(ROOT, "tests", "golden", "cfg5_choice_wav.npz"))
    wav = tmp_path / "choice.wav"
    wavfile.write(wav, int(clip["sr"]), clip["samples"])
    again = audio.get_timesteps_arr(wav, offset=0, duration=10, fps=30, margin=1.0, smooth=0.2)
    assert np.allclose(again, T, atol=1e-9)
