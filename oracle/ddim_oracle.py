"""CPU restatement of monai-generative's DDIMScheduler (`generative.networks.schedulers.DDIMScheduler`).

TEST INFRASTRUCTURE (see oracle/__init__.py). PARITY UNPINNED: like ddpm_oracle.py, the arithmetic lives in the
third-party package `monai-generative` (import name `generative`), listed unpinned by the reference and absent from
this repository and its test machines. This file restates its published algorithm (Song et al., "Denoising Diffusion
Implicit Models", eq. 12 with eta, in monai-generative's conventions: epsilon recomputed from the UNCLIPPED x0
prediction, `final_alpha_cumprod` for the step past timestep 0, `steps_offset` added to the timesteps). Places where
the restatement chooses something that memory of the upstream source cannot settle are marked [upstream-memory].
Because parity is unpinned, tests/test_ddim.py anchors it with closed-form identities: an exact eta = 0 step from
add_noise(x0, eps, t) lands on add_noise(x0, eps, t_prev), the inversion step lands on add_noise(x0, eps, t_next),
and with n = T, eta = 1 the step is OracleDDPMScheduler.step (fixed_small).
Plain torch CPU fp32 + numpy integer arithmetic; no device code.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.ddpm_oracle import make_betas


class OracleDDIMScheduler:
    def __init__(self, num_train_timesteps: int = 1000, schedule: str = "linear_beta", clip_sample: bool = True,
                 set_alpha_to_one: bool = True, steps_offset: int = 0, prediction_type: str = "epsilon",
                 **schedule_args):
        if prediction_type not in ("epsilon", "sample", "v_prediction"):
            raise ValueError("Argument `prediction_type` must be a member of `DDIMPredictionType`")
        self.betas = make_betas(schedule, num_train_timesteps, **schedule_args)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.init_noise_sigma = 1.0
        self.clip_sample = clip_sample
        self.steps_offset = steps_offset
        self.prediction_type = prediction_type
        # [upstream-memory] upstream may end its constructor with `self.set_timesteps(self.num_train_timesteps)`,
        # which with the offset check below would make any steps_offset >= 1 raise at construction. This restatement
        # (and the package) set the num_train_timesteps-step schedule directly, so steps_offset stays usable.
        self.num_inference_steps = num_train_timesteps
        self.timesteps = torch.from_numpy(np.arange(0, num_train_timesteps)[::-1].astype(np.int64).copy())

    def set_timesteps(self, num_inference_steps: int, device=None):
        if num_inference_steps > self.num_train_timesteps:
            raise ValueError("num_inference_steps cannot exceed num_train_timesteps")
        step_ratio = self.num_train_timesteps // num_inference_steps
        # [upstream-memory] the offset check; without it an offset >= ratio indexes past the last timestep
        if self.steps_offset >= step_ratio:
            raise ValueError("steps_offset must be smaller than num_train_timesteps // num_inference_steps")
        self.num_inference_steps = num_inference_steps
        ts = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(ts) + self.steps_offset

    def _get_variance(self, timestep: int, prev_timestep: int):
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        beta_prod_t_prev = 1 - alpha_prod_t_prev
        return (beta_prod_t_prev / beta_prod_t) * (1 - alpha_prod_t / alpha_prod_t_prev)

    def _predict(self, model_output, sample, alpha_prod_t):
        beta_prod_t = 1 - alpha_prod_t
        if self.prediction_type == "epsilon":
            x0 = (sample - beta_prod_t ** 0.5 * model_output) / alpha_prod_t ** 0.5
            eps = model_output
        elif self.prediction_type == "sample":
            x0 = model_output
            eps = (sample - alpha_prod_t ** 0.5 * x0) / beta_prod_t ** 0.5
        else:
            x0 = (alpha_prod_t ** 0.5) * sample - (beta_prod_t ** 0.5) * model_output
            eps = (alpha_prod_t ** 0.5) * model_output + (beta_prod_t ** 0.5) * sample
        if self.clip_sample:       # after eps: eps comes from the unclipped prediction
            x0 = torch.clamp(x0, -1, 1)
        return x0, eps

    def step(self, model_output, timestep, sample, eta: float = 0.0, generator=None, noise=None):
        """Returns (x_{t_prev}, x0_hat). `noise` injects z for parity; otherwise it is drawn on the CPU."""
        t = int(timestep)
        prev_timestep = t - self.num_train_timesteps // self.num_inference_steps
        alpha_prod_t = self.alphas_cumprod[t]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        x0, eps = self._predict(model_output, sample, alpha_prod_t)
        variance = self._get_variance(t, prev_timestep)
        std_dev_t = eta * variance ** 0.5
        pred_sample_direction = (1 - alpha_prod_t_prev - std_dev_t ** 2) ** 0.5 * eps
        prev = alpha_prod_t_prev ** 0.5 * x0 + pred_sample_direction
        if eta > 0:
            if noise is None:
                noise = torch.randn(model_output.shape, dtype=model_output.dtype, generator=generator)
            # [upstream-memory] upstream recomputes the variance here and scales as var ** 0.5 * eta * noise
            prev = prev + self._get_variance(t, prev_timestep) ** 0.5 * eta * noise
        return prev, x0

    def reversed_step(self, model_output, timestep, sample):
        """Returns (x_{t_next}, x0_hat): the deterministic step from t to t + T // n. Indexing the table past its
        end raises IndexError, as upstream's lookup does."""
        t = int(timestep)
        next_timestep = t + self.num_train_timesteps // self.num_inference_steps
        alpha_prod_t = self.alphas_cumprod[t]
        alpha_prod_t_next = self.alphas_cumprod[next_timestep]
        x0, eps = self._predict(model_output, sample, alpha_prod_t)
        pred_sample_direction = (1 - alpha_prod_t_next) ** 0.5 * eps
        return alpha_prod_t_next ** 0.5 * x0 + pred_sample_direction, x0
