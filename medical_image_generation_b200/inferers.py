"""DiffusionInferer / LatentDiffusionInferer with monai-generative's interface (the external dependency used at
train_ddpm.py:191,243 and train_ldm.py:112,157,362), driving the B200 modules and the fused scheduler kernels."""
from __future__ import annotations

import torch

from . import ops
from .schedulers import DDPMScheduler


class DiffusionInferer:
    def __init__(self, scheduler) -> None:
        self.scheduler = scheduler

    def __call__(self, inputs, diffusion_model, noise, timesteps, condition=None, mode: str = "crossattn"):
        if mode not in ("crossattn", "concat"):
            raise NotImplementedError(f"{mode} condition is not supported")
        noisy = self.scheduler.add_noise(original_samples=inputs, noise=noise, timesteps=timesteps)
        if mode == "concat":
            noisy = ops.cat_channels(noisy, condition)
            condition = None
        return diffusion_model(x=noisy, timesteps=timesteps, context=condition)

    @torch.no_grad()
    def sample(self, input_noise, diffusion_model, scheduler=None, save_intermediates: bool = False,
               intermediate_steps: int = 100, conditioning=None, mode: str = "crossattn", verbose: bool = True,
               step_noises=None, cuda_graph: bool = False):
        """Reverse process over `scheduler.timesteps`; the model is called with `torch.Tensor((t,))` like upstream.
        `step_noises` (optional list) injects the per-step z for parity tests. `cuda_graph=True` (extra, optional)
        captures the model forward once and replays it every step: the ~300 kernel launches of a reverse step stop
        costing host time (the fused scheduler step stays eager: its coefficients change every step)."""
        if mode not in ("crossattn", "concat"):
            raise NotImplementedError(f"{mode} condition is not supported")
        scheduler = scheduler or self.scheduler
        image = input_noise
        intermediates = []

        def forward(img, tt):
            if mode == "concat":
                return diffusion_model(ops.cat_channels(img, conditioning), timesteps=tt, context=None)
            return diffusion_model(img, timesteps=tt, context=conditioning)

        graph = None
        if cuda_graph and input_noise.is_cuda and len(scheduler.timesteps) > 2:
            static_img = input_noise.clone()
            static_t = torch.zeros(1, dtype=torch.float32, device=input_noise.device)
            forward(static_img, static_t)                      # warm-up: workspaces, filter shadows, tensor maps
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = forward(static_img, static_t)
        for i, t in enumerate(scheduler.timesteps):
            if graph is not None:
                static_img.copy_(image)
                static_t.fill_(float(t))
                graph.replay()
                out = static_out
            else:
                out = forward(image, torch.Tensor((t,)).to(input_noise.device))
            z = None if step_noises is None else step_noises[i]
            image, _ = scheduler.step(out, t, image, noise=z)
            if save_intermediates and t % intermediate_steps == 0:
                intermediates.append(image)
        return (image, intermediates) if save_intermediates else image

    @torch.no_grad()
    def get_likelihood(self, inputs, diffusion_model, scheduler=None, save_intermediates: bool = False,
                       conditioning=None, mode: str = "crossattn", original_input_range=(0, 255),
                       scaled_input_range=(0, 1), verbose: bool = True, *, noise=None, cuda_graph: bool = False):
        """The DDPM variational bound of each input, in nats per element: over `scheduler.timesteps`, the mean KL
        between the posterior q(x_{t-1} | x_t, x_0) and the model's p(x_{t-1} | x_t), and at t = 0 the mean negative
        log-likelihood of the input under the discretised Gaussian decoder whose bins are those of
        `original_input_range` scaled to `scaled_input_range`. Returns the fp32 (B,) total on the inputs' device (summed
        in fp64 on the device) and, with `save_intermediates`, the fp32 CPU map of every timestep.

        As upstream, one noise tensor is drawn for all timesteps and x_t comes from `self.scheduler.add_noise`. Each
        timestep's bound term is one fused kernel that reads its scalars from a device table, so `cuda_graph=True`
        (extra, optional) captures add_noise, the model forward and the bound term once and replays the whole step.
        `noise` (extra, optional) injects the noise for parity tests. `verbose` is accepted and ignored."""
        scheduler = scheduler or self.scheduler
        if not isinstance(scheduler, DDPMScheduler):
            raise NotImplementedError(f"Likelihood computation is only compatible with DDPMScheduler, you are using "
                                      f"{type(scheduler).__name__}")
        if mode not in ("crossattn", "concat"):
            raise NotImplementedError(f"{mode} condition is not supported")
        ops._require_cuda(inputs, "get_likelihood")
        B = inputs.shape[0]
        noise = torch.randn_like(inputs) if noise is None else noise.to(device=inputs.device, dtype=inputs.dtype)
        bin_width = (scaled_input_range[1] - scaled_input_range[0]) / (original_input_range[1] - original_input_range[0])
        half_bin = bin_width / 2
        total = torch.zeros(B, dtype=torch.float64, device=inputs.device)
        workspace = scheduler._vlb_workspace(inputs)
        intermediates = []

        def step(tt, acc, kl_map=None):
            """add_noise, the forward and the bound term of timestep tensor `tt`; adds into `acc`, returns the map."""
            noisy = self.scheduler.add_noise(original_samples=inputs, noise=noise, timesteps=tt)
            if mode == "concat":
                out = diffusion_model(ops.cat_channels(noisy, conditioning), timesteps=tt, context=None)
            else:
                out = diffusion_model(x=noisy, timesteps=tt, context=conditioning)
            m, x, x0 = scheduler._vlb_operands(out, noisy, inputs)
            if save_intermediates and kl_map is None:
                kl_map = torch.empty_like(x, dtype=torch.float32)
            scheduler._vlb_term(m, tt, x, x0, acc, workspace, kl_map, half_bin)
            return kl_map

        graph = None
        if cuda_graph and len(scheduler.timesteps) > 2:
            static_t = torch.full((B,), int(scheduler.timesteps[0]), dtype=torch.int64, device=inputs.device)
            static_map = step(static_t, torch.zeros_like(total))   # warm-up: workspaces, filter shadows, tensor maps
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step(static_t, total, static_map)
        for t in scheduler.timesteps:
            if graph is not None:
                static_t.fill_(int(t))
                graph.replay()
                kl_map = static_map
            else:
                kl_map = step(torch.full((B,), int(t), dtype=torch.int64, device=inputs.device), total)
            if save_intermediates:
                intermediates.append(kl_map.cpu())
        total = total.float()
        return (total, intermediates) if save_intermediates else total


class LatentDiffusionInferer(DiffusionInferer):
    def __init__(self, scheduler, scale_factor: float = 1.0) -> None:
        super().__init__(scheduler=scheduler)
        self.scale_factor = scale_factor

    def __call__(self, inputs, autoencoder_model, diffusion_model, noise, timesteps, condition=None,
                 mode: str = "crossattn"):
        with torch.no_grad():
            latent = ops.scale(autoencoder_model.encode_stage_2_inputs(inputs), float(self.scale_factor))
        return super().__call__(inputs=latent, diffusion_model=diffusion_model, noise=noise, timesteps=timesteps,
                                condition=condition, mode=mode)

    @torch.no_grad()
    def sample(self, input_noise, autoencoder_model, diffusion_model, scheduler=None, save_intermediates: bool = False,
               intermediate_steps: int = 100, conditioning=None, mode: str = "crossattn", verbose: bool = True,
               step_noises=None, cuda_graph: bool = False):
        out = super().sample(input_noise, diffusion_model, scheduler, save_intermediates, intermediate_steps,
                             conditioning, mode, verbose, step_noises, cuda_graph)
        latent, inter = out if save_intermediates else (out, None)
        image = autoencoder_model.decode_stage_2_outputs(ops.scale(latent, 1.0 / float(self.scale_factor)))
        if save_intermediates:
            return image, [autoencoder_model.decode_stage_2_outputs(ops.scale(l, 1.0 / float(self.scale_factor)))
                           for l in inter]
        return image

    @torch.no_grad()
    def get_likelihood(self, inputs, autoencoder_model, diffusion_model, scheduler=None,
                       save_intermediates: bool = False, conditioning=None, mode: str = "crossattn",
                       original_input_range=(0, 255), scaled_input_range=(0, 1), verbose: bool = True,
                       resample_latent_likelihoods: bool = False, resample_interpolation_mode: str = "nearest", *,
                       noise=None, cuda_graph: bool = False):
        """`DiffusionInferer.get_likelihood` of the latents `encode_stage_2_inputs(inputs) * scale_factor`. With
        `resample_latent_likelihoods` (which needs `save_intermediates`), every latent map is resized to the inputs'
        spatial shape with `nn.Upsample(mode=resample_interpolation_mode)`, as upstream does on its CPU maps."""
        if resample_latent_likelihoods and not save_intermediates:
            raise ValueError(f"If `resample_latent_likelihoods` is True, `save_intermediates` must also be True, got "
                             f"{save_intermediates}")
        if resample_latent_likelihoods and resample_interpolation_mode not in ("nearest", "bilinear", "trilinear"):
            raise ValueError(f"resample_interpolation_mode should be either nearest, bilinear, or trilinear, got "
                             f"{resample_interpolation_mode}")
        latents = ops.scale(autoencoder_model.encode_stage_2_inputs(inputs), float(self.scale_factor))
        out = super().get_likelihood(latents, diffusion_model, scheduler, save_intermediates, conditioning, mode,
                                     original_input_range, scaled_input_range, verbose, noise=noise,
                                     cuda_graph=cuda_graph)
        if save_intermediates and resample_latent_likelihoods:
            resizer = torch.nn.Upsample(size=tuple(inputs.shape[2:]), mode=resample_interpolation_mode)
            out = (out[0], [resizer(m) for m in out[1]])
        return out
