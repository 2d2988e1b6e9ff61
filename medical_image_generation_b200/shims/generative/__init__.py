"""Minimal `generative` (monai-generative) package for the medimgen trainers on a box where the real package is not
installed. It provides exactly what `train_ldm.py:28-32`, `train_ddpm.py:17-19` and `train_autoencoder.py:26-27`
import: the scheduler and the two inferers ARE the B200 implementations (medical_image_generation_b200.schedulers /
.inferers); the AE trainer's discriminator, adversarial loss and (LPIPS-VGG, fake-3D) perceptual loss are torch.nn
restatements of the published definitions (the perceptual weights come from a local file); the SSIM and MS-SSIM
validation metrics are the B200 implementations (medical_image_generation_b200.metrics); what the training / sampling
step never executes (VQ-VAE, the FID and MMD metrics) is a placeholder class that raises when somebody tries to
construct it. Put on sys.path by `compat.install()` only when the real package cannot be imported."""
