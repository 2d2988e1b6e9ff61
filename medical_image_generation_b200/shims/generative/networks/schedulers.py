"""generative.networks.schedulers (train_ldm.py:29, train_ddpm.py:19): the B200 DDPMScheduler and DDIMScheduler."""
from medical_image_generation_b200.schedulers import DDIMScheduler, DDPMScheduler  # noqa: F401

__all__ = ["DDPMScheduler", "DDIMScheduler"]
