"""vgen_b200 -- B200-native (sm_100a) implementation of the VGen sampling hot path:
DiffusionDDIM.ddim_sample_loop -> UNetSD_T2VBase / UNetSD_I2VGen (and the VideoLCM / TFT2V / SR600 / HiGen
variants, with the VideoComposer condition adapters) forward -> AutoencoderKL.decode,
exposed under the reference's MODEL / DIFFUSION / AUTO_ENCODER registry names (`register()`).

Every op of the path is a hand-written CUDA kernel in libvgen_b200.so (include/vgen_b200.h); this
package holds only the host-side mirror of the reference interface.  There is no CPU / PyTorch
fallback: without the built library or a CUDA device the forward raises.
"""
from .registry import register  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require torch.cuda
    if name in ("UNetSD_T2VBase", "UNetSD_I2VGen", "UNetSD_VideoLCM", "UNetSD_TFT2V", "UNetSD_SR600", "UNetSD_HiGen"):
        from . import unet
        return getattr(unet, name)
    if name == "AutoencoderKL":
        from .autoencoder import AutoencoderKL
        return AutoencoderKL
    if name == "DiffusionDDIM":
        from .diffusion import DiffusionDDIM
        return DiffusionDDIM
    if name in ("GaussianDiffusion", "DiffusionDDIMSR"):
        from . import diffusion_gauss
        return getattr(diffusion_gauss, name)
    if name in ("FrozenOpenCLIPEmbedder", "FrozenOpenCLIPVisualEmbedder", "FrozenOpenCLIPTextVisualEmbedder"):
        from . import clip
        return getattr(clip, name)
    if name == "LCMScheduler":
        from .lcm import LCMScheduler
        return LCMScheduler
    raise AttributeError(name)
