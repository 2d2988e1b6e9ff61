"""medical_image_generation_b200 -- B200-native (sm_100a) drop-in for the 3D latent-diffusion hot path of
VKostoulas/Medical_Image_Generation (`medimgen`): strided DiffusionModelUNet / AutoencoderKL blocks and the
DDPMScheduler add_noise / step loop, as hand-written CUDA kernels behind a C ABI (include/medimgen_b200.h).

There is no CPU or library fallback: importing works anywhere (module construction, state_dict handling and the
scheduler's integer logic are host code), but every forward / scheduler call needs the built shared library and
a CUDA device, and raises otherwise.
"""
from .autoencoderkl import AutoencoderKL
from .inferers import DiffusionInferer, LatentDiffusionInferer
from .metrics import MultiScaleSSIMMetric, SSIMMetric, pairwise_ms_ssim
from .schedulers import DDIMScheduler, DDPMScheduler
from .unet import DiffusionModelUNet

__all__ = ["AutoencoderKL", "DiffusionModelUNet", "DDPMScheduler", "DDIMScheduler", "DiffusionInferer",
           "LatentDiffusionInferer", "SSIMMetric", "MultiScaleSSIMMetric", "pairwise_ms_ssim"]
