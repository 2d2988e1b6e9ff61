"""DDPMScheduler and DDIMScheduler with the interface of monai-generative's `generative.networks.schedulers`
(the external dependency the reference drives at train_ldm.py:74,145,160,163-167,351 and
train_ddpm.py:380-382), backed by fused sm_100a kernels:

  add_noise / get_velocity      : one 128-bit vectorised kernel, per-sample coefficient gather (K14)
  DDPMScheduler.step            : ONE kernel per reverse step instead of ~12 elementwise launches (K15)
  DDIMScheduler.step / reversed_step : ONE kernel per step (ddim_step), for few-step sampling and DDIM inversion
  DDPMScheduler._vlb_term       : ONE kernel per timestep of the likelihood bound (ddpm_vlb_term), scalars from a device
                                  table (`vlb_coefficients`) so the whole timestep can be graph-captured

Index arithmetic (timesteps, alpha_bar[t], alpha_bar[t-1]) is done exactly as upstream: fp32 tables built
with torch on the host, `set_timesteps` in numpy int64, per-step coefficients evaluated in fp32 on the
host from those tables and passed to the kernel as scalars.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import ops
from ._lib import call, load


def _betas(schedule: str, num_train_timesteps: int, beta_start: float = 1e-4, beta_end: float = 2e-2,
           sig_range: float = 6.0, **unused) -> torch.Tensor:
    if schedule == "linear_beta":
        return torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    if schedule == "scaled_linear_beta":
        return torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    if schedule == "sigmoid_beta":
        return torch.sigmoid(torch.linspace(-sig_range, sig_range, num_train_timesteps)) * (beta_end - beta_start) \
            + beta_start
    raise ValueError(f"unknown noise schedule '{schedule}' (linear_beta, scaled_linear_beta, sigmoid_beta)")


_PREDICTION = {"epsilon": 0, "sample": 1, "v_prediction": 2}


class _NoiseSchedule:
    """What DDPMScheduler and DDIMScheduler share: the fp32 beta / alpha tables, their device copy, the fused
    add_noise / get_velocity kernel, the operand layout rules of a step and the draw of the step noise z."""

    def __init__(self, num_train_timesteps: int, schedule: str, clip_sample: bool, prediction_type: str,
                 **schedule_args) -> None:
        self.betas = _betas(schedule, num_train_timesteps, **schedule_args)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_train_timesteps = num_train_timesteps
        self.one = torch.tensor(1.0)
        self.clip_sample = clip_sample
        self.prediction_type = prediction_type
        self.num_inference_steps = None
        self.noise_mode = "host"  # "host": z drawn on the CPU like upstream (seed-compatible); "device": on the GPU
        self._dev_tables: dict = {}

    # -- tables on the device (fp32, read by the gather in the add_noise kernel) -----------------------
    def _acp_on(self, device) -> torch.Tensor:
        t = self._dev_tables.get(device)
        if t is None:
            t = self.alphas_cumprod.to(device=device, dtype=torch.float32).contiguous()
            self._dev_tables[device] = t
        return t

    def _noise_op(self, a, b, timesteps, velocity: int):
        if not a.is_cuda:
            raise RuntimeError(f"{type(self).__name__}: tensors must live on a CUDA device (no CPU path)")
        if a.dtype not in (torch.float32, torch.bfloat16):
            a = a.float()
        b = b.to(a.dtype)
        if a.stride() != b.stride() or not (a.is_contiguous() or ops._is_cl(a)):
            a, b = a.contiguous(), b.contiguous()
        B = a.shape[0]
        ts = timesteps.to(device=a.device, dtype=torch.int64).contiguous()
        if ts.numel() != B:
            raise RuntimeError(f"timesteps has {ts.numel()} entries for a batch of {B}")
        out = torch.empty_like(a)
        call("mig_ddpm_add_noise", ops._dt(a), ops._ptr(a), ops._ptr(b), ops._ptr(ts), ops._ptr(self._acp_on(a.device)),
             ops._ptr(out), B, a.numel() // B, self.num_train_timesteps, velocity, ops._stream())
        return out

    def add_noise(self, original_samples, noise, timesteps):
        """sqrt(acp[t]) * x0 + sqrt(1 - acp[t]) * noise, t per sample."""
        return self._noise_op(original_samples, noise, timesteps, 0)

    def get_velocity(self, sample, noise, timesteps):
        """sqrt(acp[t]) * noise - sqrt(1 - acp[t]) * sample."""
        return self._noise_op(sample, noise, timesteps, 1)

    # -- shared by the step kernels --------------------------------------------------------------------
    def _step_operands(self, model_output, sample):
        """(x, m): the sample in float32 / bfloat16 and the model output in the same dtype and strides (contiguous
        or channels-last; anything else is made contiguous)."""
        if not sample.is_cuda:
            raise RuntimeError(f"{type(self).__name__}.step: tensors must live on a CUDA device (no CPU path)")
        x = sample if sample.dtype in (torch.float32, torch.bfloat16) else sample.float()
        m = model_output.to(x.dtype)
        if m.stride() != x.stride() or not (x.is_contiguous() or ops._is_cl(x)):
            x, m = x.contiguous(), m.contiguous()
        return x, m

    def _step_noise(self, model_output, x, generator, noise):
        """z ~ N(0, 1) in x's dtype and strides: the injected `noise` if given, else drawn per `noise_mode` ("host":
        on the CPU in the model output's dtype, as upstream draws it; "device": on x's device)."""
        if noise is not None:
            z = noise.to(device=x.device, dtype=x.dtype)
        elif self.noise_mode == "host":
            z = torch.randn(model_output.size(), dtype=model_output.dtype, layout=model_output.layout,
                            generator=generator).to(device=x.device, dtype=x.dtype)
        else:
            z = torch.randn(x.shape, dtype=x.dtype, device=x.device, generator=generator)
        if z.stride() != x.stride():
            z = z.contiguous() if x.is_contiguous() else ops.as_cl(z)
        return z


class DDPMScheduler(_NoiseSchedule):
    def __init__(self, num_train_timesteps: int = 1000, schedule: str = "linear_beta",
                 variance_type: str = "fixed_small", clip_sample: bool = True, prediction_type: str = "epsilon",
                 **schedule_args) -> None:
        if variance_type not in ("fixed_small", "fixed_large", "learned", "learned_range"):
            raise ValueError("Argument `variance_type` must be a member of `DDPMVarianceType`")
        if prediction_type not in ("epsilon", "sample", "v_prediction"):
            raise ValueError("Argument `prediction_type` must be a member of `DDPMPredictionType`")
        if variance_type in ("learned", "learned_range"):
            raise NotImplementedError("learned variance types are not on the medimgen hot path")
        super().__init__(num_train_timesteps, schedule, clip_sample, prediction_type, **schedule_args)
        self.variance_type = variance_type
        self.timesteps = torch.arange(num_train_timesteps - 1, -1, -1)

    # -- sampling ------------------------------------------------------------------------------------
    def set_timesteps(self, num_inference_steps: int, device=None) -> None:
        if num_inference_steps > self.num_train_timesteps:
            raise ValueError(f"`num_inference_steps`: {num_inference_steps} cannot be larger than "
                             f"`self.num_train_timesteps`: {self.num_train_timesteps}")
        self.num_inference_steps = num_inference_steps
        step_ratio = self.num_train_timesteps // self.num_inference_steps
        ts = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].astype(np.int64)
        self.timesteps = torch.from_numpy(ts.copy()).to(device)

    def step_coefficients(self, timestep: int) -> dict:
        """fp32 host evaluation of the per-step scalars, same operation order as upstream `step`."""
        t = int(timestep)
        acp_t = self.alphas_cumprod[t]
        acp_prev = self.alphas_cumprod[t - 1] if t > 0 else self.one
        beta_prod_t = 1 - acp_t
        beta_prod_prev = 1 - acp_prev
        c0 = (acp_prev ** 0.5 * self.betas[t]) / beta_prod_t
        ct = self.alphas[t] ** 0.5 * beta_prod_prev / beta_prod_t
        sigma = self._get_variance(t) ** 0.5 if t > 0 else torch.tensor(0.0)
        return dict(sqrt_acp=float(acp_t ** 0.5), sqrt_one_minus_acp=float(beta_prod_t ** 0.5), c0=float(c0),
                    ct=float(ct), sigma=float(sigma), t=t, t_prev=t - 1)

    def _get_variance(self, timestep: int) -> torch.Tensor:
        """The fp32 variance of the posterior step at `timestep` (upstream `_get_variance`, fixed variance types)."""
        t = int(timestep)
        acp_t = self.alphas_cumprod[t]
        acp_prev = self.alphas_cumprod[t - 1] if t > 0 else self.one
        var = (1 - acp_prev) / (1 - acp_t) * self.betas[t]
        if self.variance_type == "fixed_small":
            var = torch.clamp(var, min=1e-20)
        elif self.variance_type == "fixed_large":
            var = self.betas[t]
        return var

    # -- likelihood ------------------------------------------------------------------------------------
    VLB_COEFS = ("sqrt_acp", "sqrt_one_minus_acp", "c0", "ct", "kl_const", "inv_var", "inv_std")

    def vlb_coefficients(self) -> torch.Tensor:
        """(T, 7) fp32 CPU table of the per-timestep scalars of the variational bound, evaluated like upstream
        `get_likelihood` evaluates them: the coefficients of `step`, and with lv = log(variance) the constant part of
        the KL of two Normals of equal variance (-1 + lv - lv + exp(lv - lv)), exp(-lv) and exp(-0.5 lv)."""
        rows = []
        for t in range(self.num_train_timesteps):
            k = self.step_coefficients(t)
            lv = torch.log(self._get_variance(t))
            kl_const = -1.0 + lv - lv + torch.exp(lv - lv)
            rows.append([k["sqrt_acp"], k["sqrt_one_minus_acp"], k["c0"], k["ct"], float(kl_const),
                         float(torch.exp(-lv)), float(torch.exp(-(0.5 * lv)))])
        return torch.tensor(rows, dtype=torch.float32)

    def _vlb_table_on(self, device) -> torch.Tensor:
        key = ("vlb", self.variance_type, device)
        t = self._dev_tables.get(key)
        if t is None:
            t = self.vlb_coefficients().to(device).contiguous()
            self._dev_tables[key] = t
        return t

    def _vlb_workspace(self, sample) -> torch.Tensor:
        """A scratch buffer large enough for `_vlb_term` on samples shaped like `sample`."""
        B = sample.shape[0]
        nbytes = load().mig_ddpm_vlb_workspace_bytes(B, sample.numel() // max(B, 1))
        if nbytes < 0:
            raise RuntimeError(f"_vlb_term: no workspace for a batch of shape {tuple(sample.shape)}")
        return torch.empty(nbytes, dtype=torch.uint8, device=sample.device)

    def _vlb_term(self, model_output, timesteps, sample, original_samples, total, workspace, kl_map=None,
                 half_bin: float = 0.5 / 255):
        """One timestep of upstream `get_likelihood` in one launch: the KL term (t > 0) or the decoder negative
        log-likelihood (t == 0) of every element, from the model output at the noisy `sample` x_t and the clean
        `original_samples` x_0, t per sample from the device tensor `timesteps`. Adds each sample's mean into `total`
        (fp64 (B,), on the device) and writes the fp32 map into `kl_map` when given (shaped and strided like the
        operands as returned by `_vlb_operands`). `half_bin` is half the decoder's bin width."""
        B = sample.shape[0]
        if timesteps.dtype != torch.int64 or timesteps.numel() != B or not timesteps.is_contiguous():
            raise RuntimeError(f"vlb_term: timesteps must be {B} contiguous int64 values")
        if total.dtype != torch.float64 or total.numel() != B:
            raise RuntimeError(f"vlb_term: total must hold {B} float64 values")
        if kl_map is not None and (kl_map.dtype != torch.float32 or kl_map.stride() != sample.stride()
                                   or kl_map.shape != sample.shape):
            raise RuntimeError("vlb_term: kl_map must be float32, shaped and strided like the sample")
        table = self._vlb_table_on(sample.device)
        call("mig_ddpm_vlb_term", ops._dt(sample), ops._ptr(model_output), ops._ptr(sample), ops._ptr(original_samples),
             ops._ptr(timesteps), ops._ptr(table), table.numel(), self.num_train_timesteps, B, sample.numel() // B,
             _PREDICTION[self.prediction_type], int(self.clip_sample), float(half_bin), ops._ptr(kl_map),
             ops._ptr(total), ops._ptr(workspace), workspace.numel(), ops._stream())

    def _vlb_operands(self, model_output, sample, original_samples):
        """(m, x_t, x_0) in one dtype (float32 or bfloat16, the sample's) and one layout (contiguous or channels-last,
        the sample's when both others can take it; otherwise all contiguous)."""
        x, m = self._step_operands(model_output, sample)
        x0 = original_samples.to(x.dtype)
        if x0.stride() != x.stride():
            x, m, x0 = x.contiguous(), m.contiguous(), x0.contiguous()
        return m, x, x0

    def step(self, model_output, timestep, sample, generator=None, noise=None):
        """One reverse-diffusion step. Returns (pred_prev_sample, pred_original_sample).
        `noise` (optional) injects z for parity tests; otherwise z ~ N(0,1) is drawn per `noise_mode`."""
        x, eps = self._step_operands(model_output, sample)
        k = self.step_coefficients(int(timestep))
        z = self._step_noise(model_output, x, generator, noise) if k["t"] > 0 else None
        prev = torch.empty_like(x)
        x0 = torch.empty_like(x)
        pred = _PREDICTION[self.prediction_type]
        call("mig_ddpm_step", ops._dt(x), ops._ptr(eps), ops._ptr(x), ops._ptr(z), ops._ptr(prev), ops._ptr(x0),
             x.numel(), k["sqrt_acp"], k["sqrt_one_minus_acp"], k["c0"], k["ct"], k["sigma"] if z is not None else 0.0,
             pred, int(self.clip_sample), ops._stream())
        return prev, x0


class DDIMScheduler(_NoiseSchedule):
    """Denoising diffusion implicit models (Song et al. 2020) with monai-generative's interface. Samples with few steps
    (`set_timesteps(50)`) from any epsilon-, sample- or v-trained model, and inverts a sample back to its noise
    (`reversed_step`). eta = 0 is the deterministic DDIM sampler; eta = 1 with `set_timesteps(num_train_timesteps)`
    is DDPM's fixed_small posterior."""

    def __init__(self, num_train_timesteps: int = 1000, schedule: str = "linear_beta", clip_sample: bool = True,
                 set_alpha_to_one: bool = True, steps_offset: int = 0, prediction_type: str = "epsilon",
                 **schedule_args) -> None:
        if prediction_type not in ("epsilon", "sample", "v_prediction"):
            raise ValueError("Argument `prediction_type` must be a member of `DDIMPredictionType`")
        super().__init__(num_train_timesteps, schedule, clip_sample, prediction_type, **schedule_args)
        # alpha_bar of the step after the last one (timestep -1): 1 (the clean sample) or alpha_bar[0]
        self.final_alpha_cumprod = self.one if set_alpha_to_one else self.alphas_cumprod[0]
        self.steps_offset = steps_offset
        self.init_noise_sigma = 1.0
        # the num_train_timesteps-step schedule, without the offset check of set_timesteps: steps_offset >= 1 is only
        # valid once set_timesteps chooses fewer steps
        self.num_inference_steps = num_train_timesteps
        self.timesteps = torch.arange(num_train_timesteps - 1, -1, -1)

    def set_timesteps(self, num_inference_steps: int, device=None) -> None:
        if num_inference_steps > self.num_train_timesteps:
            raise ValueError(f"`num_inference_steps`: {num_inference_steps} cannot be larger than "
                             f"`self.num_train_timesteps`: {self.num_train_timesteps}")
        step_ratio = self.num_train_timesteps // num_inference_steps
        if self.steps_offset >= step_ratio:
            raise ValueError(f"`steps_offset`: {self.steps_offset} cannot be greater than or equal to "
                             f"`num_train_timesteps // num_inference_steps`: {step_ratio}, as the timesteps would "
                             f"exceed the last training timestep")
        self.num_inference_steps = num_inference_steps
        ts = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].astype(np.int64) + self.steps_offset
        self.timesteps = torch.from_numpy(ts.copy()).to(device)

    def _acp_or_final(self, t: int) -> torch.Tensor:
        return self.alphas_cumprod[t] if t >= 0 else self.final_alpha_cumprod

    def step_coefficients(self, timestep: int, eta: float = 0.0) -> dict:
        """fp32 host evaluation of the per-step scalars, same operation order as upstream `step`."""
        t = int(timestep)
        t_prev = t - self.num_train_timesteps // self.num_inference_steps
        acp_t = self.alphas_cumprod[t]
        acp_prev = self._acp_or_final(t_prev)
        beta_prod_t = 1 - acp_t
        var = (1 - acp_prev) / beta_prod_t * (1 - acp_t / acp_prev)
        sigma = eta * var ** 0.5
        dir_coef = (1 - acp_prev - sigma ** 2) ** 0.5
        return dict(sqrt_acp=float(acp_t ** 0.5), sqrt_one_minus_acp=float(beta_prod_t ** 0.5),
                    sqrt_acp_prev=float(acp_prev ** 0.5), dir_coef=float(dir_coef), sigma=float(sigma), t=t,
                    t_prev=t_prev)

    def reversed_step_coefficients(self, timestep: int) -> dict:
        """The scalars of `reversed_step`: the step from t to t + T // n, with no noise term."""
        t = int(timestep)
        t_next = t + self.num_train_timesteps // self.num_inference_steps
        if t_next >= self.num_train_timesteps:
            raise IndexError(f"reversed_step from timestep {t} reaches timestep {t_next}, past the last training "
                             f"timestep {self.num_train_timesteps - 1}")
        acp_t = self.alphas_cumprod[t]
        acp_next = self.alphas_cumprod[t_next]
        beta_prod_t = 1 - acp_t
        return dict(sqrt_acp=float(acp_t ** 0.5), sqrt_one_minus_acp=float(beta_prod_t ** 0.5),
                    sqrt_acp_prev=float(acp_next ** 0.5), dir_coef=float((1 - acp_next) ** 0.5), sigma=0.0, t=t,
                    t_next=t_next)

    def _launch(self, x, m, z, k):
        prev = torch.empty_like(x)
        x0 = torch.empty_like(x)
        call("mig_ddim_step", ops._dt(x), ops._ptr(m), ops._ptr(x), ops._ptr(z), ops._ptr(prev), ops._ptr(x0),
             x.numel(), k["sqrt_acp"], k["sqrt_one_minus_acp"], k["sqrt_acp_prev"], k["dir_coef"],
             k["sigma"] if z is not None else 0.0, _PREDICTION[self.prediction_type], int(self.clip_sample),
             ops._stream())
        return prev, x0

    def step(self, model_output, timestep, sample, eta: float = 0.0, generator=None, noise=None):
        """One reverse step from `timestep` to the previous timestep of the schedule. Returns (pred_prev_sample,
        pred_original_sample). With eta > 0, z is `noise` when given (parity tests), otherwise drawn per
        `noise_mode`; with eta == 0 the step is deterministic and `noise` is ignored."""
        x, m = self._step_operands(model_output, sample)
        k = self.step_coefficients(int(timestep), eta)
        z = self._step_noise(model_output, x, generator, noise) if eta > 0 else None
        return self._launch(x, m, z, k)

    def reversed_step(self, model_output, timestep, sample):
        """One DDIM inversion step from `timestep` to the next timestep of the schedule (t + T // n), i.e. towards
        noise. Returns (pred_post_sample, pred_original_sample)."""
        x, m = self._step_operands(model_output, sample)
        return self._launch(x, m, None, self.reversed_step_coefficients(int(timestep)))
