"""CPU restatement of monai-generative's `DiffusionInferer.get_likelihood` and `LatentDiffusionInferer.get_likelihood`
(the DDPM variational bound of an input, with per-timestep maps for likelihood-based anomaly detection).

TEST INFRASTRUCTURE (see oracle/__init__.py). PARITY UNPINNED: like ddpm_oracle.py and ddim_oracle.py, the arithmetic
lives in the third-party package `monai-generative` (import name `generative`), unpinned and absent from this
repository and its test machines. This file restates its published algorithm on top of OracleDDPMScheduler (Ho et al.
2020, eq. 5 and the L_0 decoder of section 3.3, with the tanh approximation of the normal CDF, in monai-generative's
conventions). Places where the restatement chooses something that memory of the upstream source cannot settle are
marked [upstream-memory]. Because parity is unpinned, tests/test_likelihood.py anchors it with identities: the KL term
equals torch.distributions.kl_divergence of the two Normals, a model that predicts the true noise or the true sample
gives a closed-form bound, and the tanh CDF is within its known error of the exact one.
Plain torch CPU fp32 (inputs are taken to fp32 first); no device code.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from oracle.ddpm_oracle import OracleDDPMScheduler


def normal_kl(mean1, logvar1, mean2, logvar2):
    """KL(N(mean1, exp(logvar1)) || N(mean2, exp(logvar2))) per element, in upstream's operation order."""
    return 0.5 * (-1.0 + logvar2 - logvar1 + torch.exp(logvar1 - logvar2)
                  + ((mean1 - mean2) ** 2) * torch.exp(-logvar2))


def approx_standard_normal_cdf(x):
    k = torch.sqrt(torch.Tensor([2.0 / math.pi]).to(x.device))
    return 0.5 * (1.0 + torch.tanh(k * (x + 0.044715 * torch.pow(x, 3))))


def decoder_log_likelihood(inputs, means, log_scales, original_input_range=(0, 255), scaled_input_range=(0, 1)):
    """log p(inputs) under a Gaussian of mean `means` and log standard deviation `log_scales`, discretised into the bins
    of `original_input_range` mapped onto `scaled_input_range`; the end bins at +-1 extend to infinity."""
    assert inputs.shape == means.shape
    bin_width = (scaled_input_range[1] - scaled_input_range[0]) / (original_input_range[1] - original_input_range[0])
    centered_x = inputs - means
    inv_stdv = torch.exp(-log_scales)
    plus_in = inv_stdv * (centered_x + bin_width / 2)
    cdf_plus = approx_standard_normal_cdf(plus_in)
    min_in = inv_stdv * (centered_x - bin_width / 2)
    cdf_min = approx_standard_normal_cdf(min_in)
    log_cdf_plus = torch.log(cdf_plus.clamp(min=1e-12))
    log_one_minus_cdf_min = torch.log((1.0 - cdf_min).clamp(min=1e-12))
    cdf_delta = cdf_plus - cdf_min
    return torch.where(inputs < -0.999, log_cdf_plus,
                       torch.where(inputs > 0.999, log_one_minus_cdf_min, torch.log(cdf_delta.clamp(min=1e-12))))


def posterior_mean(scheduler: OracleDDPMScheduler, t: int, x_0, x_t):
    """Upstream DDPMScheduler._get_mean: the mean of q(x_{t-1} | x_t, x_0)."""
    alpha_t = scheduler.alphas[t]
    alpha_prod_t = scheduler.alphas_cumprod[t]
    alpha_prod_t_prev = scheduler.alphas_cumprod[t - 1] if t > 0 else scheduler.one
    x_0_coefficient = alpha_prod_t_prev.sqrt() * scheduler.betas[t] / (1 - alpha_prod_t)
    x_t_coefficient = alpha_t.sqrt() * (1 - alpha_prod_t_prev) / (1 - alpha_prod_t)
    return x_0_coefficient * x_0 + x_t_coefficient * x_t


def vlb_term(scheduler: OracleDDPMScheduler, model_output, t: int, noisy, inputs, original_input_range=(0, 255),
             scaled_input_range=(0, 1)):
    """The per-element bound term of timestep t (the loop body of upstream get_likelihood), fp32."""
    t = int(t)
    model_output, noisy, inputs = (v.float() for v in (model_output, noisy, inputs))
    alpha_prod_t = scheduler.alphas_cumprod[t]
    alpha_prod_t_prev = scheduler.alphas_cumprod[t - 1] if t > 0 else scheduler.one
    beta_prod_t = 1 - alpha_prod_t
    beta_prod_t_prev = 1 - alpha_prod_t_prev
    if scheduler.prediction_type == "epsilon":
        pred_original_sample = (noisy - beta_prod_t ** 0.5 * model_output) / alpha_prod_t ** 0.5
    elif scheduler.prediction_type == "sample":
        pred_original_sample = model_output
    else:
        pred_original_sample = (alpha_prod_t ** 0.5) * noisy - (beta_prod_t ** 0.5) * model_output
    if scheduler.clip_sample:
        pred_original_sample = torch.clamp(pred_original_sample, -1, 1)
    pred_original_sample_coeff = (alpha_prod_t_prev ** 0.5 * scheduler.betas[t]) / beta_prod_t
    current_sample_coeff = scheduler.alphas[t] ** 0.5 * beta_prod_t_prev / beta_prod_t
    predicted_mean = pred_original_sample_coeff * pred_original_sample + current_sample_coeff * noisy
    mean_q = posterior_mean(scheduler, t, inputs, noisy)
    # learned variances are out of scope: the predicted variance is the posterior's
    log_posterior_variance = torch.log(scheduler._variance(t))
    log_predicted_variance = log_posterior_variance
    if t == 0:
        return -decoder_log_likelihood(inputs, predicted_mean, 0.5 * log_predicted_variance, original_input_range,
                                       scaled_input_range)
    return normal_kl(mean_q, log_posterior_variance, predicted_mean, log_predicted_variance)


def get_likelihood(inferer_scheduler: OracleDDPMScheduler, inputs, diffusion_model, scheduler=None,
                   save_intermediates=False, conditioning=None, mode="crossattn", original_input_range=(0, 255),
                   scaled_input_range=(0, 1), noise=None):
    """Upstream DiffusionInferer.get_likelihood with the inferer's scheduler `inferer_scheduler`. `noise` replaces the
    single randn_like draw."""
    scheduler = scheduler or inferer_scheduler
    if not isinstance(scheduler, OracleDDPMScheduler):
        raise NotImplementedError("Likelihood computation is only compatible with DDPMScheduler")
    if mode not in ("crossattn", "concat"):
        raise NotImplementedError(f"{mode} condition is not supported")
    inputs = inputs.float()
    noise = torch.randn_like(inputs) if noise is None else noise.float()
    intermediates = []
    total_kl = torch.zeros(inputs.shape[0])
    for t in scheduler.timesteps:
        timesteps = torch.full(inputs.shape[:1], int(t)).long()
        # [upstream-memory] x_t comes from the inferer's own scheduler, the coefficients from the `scheduler` argument
        noisy = inferer_scheduler.add_noise(original_samples=inputs, noise=noise, timesteps=timesteps)
        if mode == "concat":
            model_output = diffusion_model(torch.cat([noisy, conditioning], dim=1), timesteps=timesteps, context=None)
        else:
            model_output = diffusion_model(noisy, timesteps=timesteps, context=conditioning)
        kl = vlb_term(scheduler, model_output, int(t), noisy, inputs, original_input_range, scaled_input_range)
        total_kl += kl.view(kl.shape[0], -1).mean(dim=1)
        if save_intermediates:
            intermediates.append(kl.cpu())
    return (total_kl, intermediates) if save_intermediates else total_kl


def latent_get_likelihood(inferer_scheduler, scale_factor, inputs, autoencoder_model, diffusion_model, scheduler=None,
                          save_intermediates=False, conditioning=None, mode="crossattn", original_input_range=(0, 255),
                          scaled_input_range=(0, 1), resample_latent_likelihoods=False,
                          resample_interpolation_mode="nearest", noise=None):
    """Upstream LatentDiffusionInferer.get_likelihood: the bound of the scaled latents, maps optionally resized to the
    inputs' spatial shape."""
    if resample_latent_likelihoods and not save_intermediates:
        raise ValueError("If `resample_latent_likelihoods` is True, `save_intermediates` must also be True")
    # [upstream-memory] the set of accepted interpolation modes and that a bad one raises ValueError
    if resample_latent_likelihoods and resample_interpolation_mode not in ("nearest", "bilinear", "trilinear"):
        raise ValueError("resample_interpolation_mode should be either nearest, bilinear, or trilinear")
    latents = autoencoder_model.encode_stage_2_inputs(inputs) * scale_factor
    out = get_likelihood(inferer_scheduler, latents, diffusion_model, scheduler, save_intermediates, conditioning, mode,
                         original_input_range, scaled_input_range, noise)
    if save_intermediates and resample_latent_likelihoods:
        resizer = nn.Upsample(size=tuple(inputs.shape[2:]), mode=resample_interpolation_mode)
        out = (out[0], [resizer(x) for x in out[1]])
    return out
