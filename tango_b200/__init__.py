"""tango_b200 — B200-native (sm_100a) implementation of the Tango text-to-audio inference hot path.

Public surface (mirrors the reference's): Tango, AudioDiffusion, UNet2DConditionModel, DDPMScheduler,
DDIMScheduler, DPMSolverMultistepScheduler, AutoencoderKL. Importing the package does not touch CUDA; the kernels live in
tango_b200/lib/libtango_b200.so (built by tango_b200.build) and are bound through ctypes in tango_b200.lib.
"""
__all__ = ["Tango", "AudioDiffusion", "UNet2DConditionModel", "DDPMScheduler", "DDIMScheduler", "DPMSolverMultistepScheduler",
           "AutoencoderKL"]


def __getattr__(name):
    if name in ("Tango", "AudioDiffusion"):
        from . import pipeline
        return getattr(pipeline, name)
    if name == "UNet2DConditionModel":
        from .unet import UNet2DConditionModel
        return UNet2DConditionModel
    if name in ("DDPMScheduler", "DDIMScheduler", "DPMSolverMultistepScheduler"):
        from . import schedulers
        return getattr(schedulers, name)
    if name == "AutoencoderKL":
        from .vae import AutoencoderKL
        return AutoencoderKL
    raise AttributeError(name)
