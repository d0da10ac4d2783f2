"""stable-diffusion-videos_b200 — Blackwell-native latent-walk hot path.

Drop-in surface for the hot path of `stable_diffusion_videos` (reference __init__.py:99-119): import this package
as `stable_diffusion_videos_b200` and use `StableDiffusionWalkPipeline` / `make_video_pyav` / `get_timesteps_arr`
exactly as the reference's.  Heavy modules load lazily so `import` works on a CPU-only box (the CUDA library is
needed — and required — only when the pipeline runs).
"""
__version__ = "0.1.0"

_LAZY = {
    "StableDiffusionWalkPipeline": ("pipeline", "StableDiffusionWalkPipeline"),
    "NativeUNet": ("pipeline", "NativeUNet"),
    "NativeVAE": ("pipeline", "NativeVAE"),
    "make_video_pyav": ("utils", "make_video_pyav"),
    "get_timesteps_arr": ("utils", "get_timesteps_arr"),
    "slerp": ("utils", "slerp"),
    "Engine": ("engine", "Engine"),
    "UNetConfig": ("configs", "UNetConfig"),
    "VAEConfig": ("configs", "VAEConfig"),
    "RealESRGANModel": ("upsampling", "RealESRGANModel"),
}


def __getattr__(name):
    if name in _LAZY:
        import importlib

        mod, attr = _LAZY[name]
        return getattr(importlib.import_module(f"{__name__}.{mod}"), attr)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
