"""GPU: DDIMScheduler's fused step kernel (ddim_step) against the CPU oracle, the custom op, the noise draw, and DDIM
sampling / inversion end to end through the public inferers with a model whose exact answer is known."""
import pytest
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import _lib, ops, planner
from oracle.ddim_oracle import OracleDDIMScheduler
from util import assert_close_local, bf16_round, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
LDM = planner.LDM_SCHEDULER_KWARGS
TOL = {torch.float32: 2e-6, torch.bfloat16: 8e-3}   # the bars of test_scheduler_kernels_vs_oracle


def _operands(shape, dtype, cl, g):
    """(m, x, z): CPU fp32 values exactly representable in `dtype`, and their device copies in `dtype` / layout."""
    host = [torch.randn(shape, generator=g) * s for s in (1.0, 1.5, 1.0)]
    if dtype == torch.bfloat16:
        host = [bf16_round(h) for h in host]
    dev = [h.to(DEV, dtype) for h in host]
    if cl:
        dev = [d.contiguous(memory_format=torch.channels_last_3d) for d in dev]
    return host, dev


# 750 elements: not a multiple of the 4 (fp32) or 8 (bf16) lanes of a 16-byte vector -> scalar tail;
# channels-last 2x8x4x4x4: the vector path with strided operands
LAYOUTS = [((2, 3, 5, 5, 5), False), ((2, 8, 4, 4, 4), True)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_ddim_step_kernel_vs_oracle(dtype, pred):
    g = torch.Generator().manual_seed(5)
    tol = TOL[dtype]
    for clip, one in ((True, True), (False, True), (True, False)):     # one: set_alpha_to_one
        s = mig.DDIMScheduler(clip_sample=clip, set_alpha_to_one=one, **dict(LDM, prediction_type=pred))
        o = OracleDDIMScheduler(clip_sample=clip, set_alpha_to_one=one, **dict(LDM, prediction_type=pred))
        for n in (1000, 50):                      # at n = 50, t = 1 and t = 0 step past timestep 0 (final alpha)
            s.set_timesteps(n)
            o.set_timesteps(n)
            for shape, cl in LAYOUTS:
                for t in (999, 500, 1, 0):
                    (m, x, z), (md, xd, zd) = _operands(shape, dtype, cl, g)
                    for eta in (0.0, 1.0):
                        prev, x0 = s.step(md, t, xd, eta=eta, noise=zd)
                        assert prev.dtype == dtype and prev.stride() == xd.stride() and x0.stride() == xd.stride()
                        wprev, wx0 = o.step(m, t, x, eta=eta, noise=z)
                        e = (rel_err(prev, wprev), rel_err(x0, wx0))
                        assert max(e) < tol, (clip, one, n, shape, t, eta, e)
                    if t + 1000 // n < 1000:
                        nxt, x0 = s.reversed_step(md, t, xd)
                        wnxt, wx0 = o.reversed_step(m, t, x)
                        e = (rel_err(nxt, wnxt), rel_err(x0, wx0))
                        assert max(e) < tol, ("reversed", clip, n, shape, t, e)
                    else:
                        with pytest.raises(IndexError):
                            s.reversed_step(md, t, xd)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ddim_step_abi_without_x0_and_rejections(dtype):
    """x0_hat may be NULL (prev is unchanged); z is required when sigma != 0; n <= 0 is a no-op."""
    g = torch.Generator().manual_seed(6)
    s = mig.DDIMScheduler(**LDM)
    s.set_timesteps(50)
    (m, x, z), (md, xd, zd) = _operands((3, 1, 7, 9, 11), dtype, False, g)
    want, _ = s.step(md, 500, xd, eta=1.0, noise=zd)
    k = s.step_coefficients(500, 1.0)
    prev = torch.empty_like(xd)
    dt = ops._dt(xd)
    _lib.call("mig_ddim_step", dt, ops._ptr(md), ops._ptr(xd), ops._ptr(zd), ops._ptr(prev), None, xd.numel(),
              k["sqrt_acp"], k["sqrt_one_minus_acp"], k["sqrt_acp_prev"], k["dir_coef"], k["sigma"], 0, 1, ops._stream())
    assert torch.equal(prev, want)
    with pytest.raises(RuntimeError, match="noise buffer required"):
        _lib.call("mig_ddim_step", dt, ops._ptr(md), ops._ptr(xd), None, ops._ptr(prev), None, xd.numel(),
                  k["sqrt_acp"], k["sqrt_one_minus_acp"], k["sqrt_acp_prev"], k["dir_coef"], 0.5, 0, 1, ops._stream())
    _lib.call("mig_ddim_step", dt, None, None, None, None, None, 0, 1.0, 0.0, 1.0, 0.0, 0.0, 0, 1, ops._stream())
    torch.cuda.synchronize()


def test_full_schedule_eta_one_matches_the_ddpm_kernel():
    """n = T, eta = 1, clipping off: DDIMScheduler.step is DDPMScheduler.step (fixed_small) given the same z."""
    g = torch.Generator().manual_seed(7)
    worst = 0.0
    for pred in ("epsilon", "sample", "v_prediction"):
        kw = dict(LDM, prediction_type=pred)
        d, p = mig.DDIMScheduler(clip_sample=False, **kw), mig.DDPMScheduler(clip_sample=False, **kw)
        d.set_timesteps(1000)
        p.set_timesteps(1000)
        for t in (999, 700, 500, 100, 10, 2, 1, 0):
            m, x, z = (torch.randn(2, 1, 16, 16, 8, generator=g).to(DEV) for _ in range(3))
            got, gx0 = d.step(m, t, x, eta=1.0, noise=z)
            want, wx0 = p.step(m, t, x, noise=z)
            worst = max(worst, rel_err(got, want))
            assert rel_err(gx0, wx0) < 1e-6, (pred, t)
    assert worst < 1e-5, worst


def test_step_noise_host_and_device_modes():
    g = torch.Generator().manual_seed(8)
    s, o = mig.DDIMScheduler(**LDM), OracleDDIMScheduler(**LDM)
    s.set_timesteps(50)
    o.set_timesteps(50)
    (m, x, _), (md, xd, _) = _operands((2, 1, 8, 8, 8), torch.float32, False, g)
    # host mode: z drawn on the CPU exactly as upstream draws it, so a seeded generator reproduces the oracle
    got, _ = s.step(md, 500, xd, eta=0.7, generator=torch.Generator().manual_seed(11))
    want, _ = o.step(m, 500, x, eta=0.7, generator=torch.Generator().manual_seed(11))
    assert rel_err(got, want) < 2e-6
    det, _ = s.step(md, 500, xd)                         # eta = 0 draws nothing and is deterministic
    assert rel_err(got, det) > 1e-3
    # device mode: finite, and a fresh z every step
    s.noise_mode = "device"
    a, _ = s.step(md, 500, xd, eta=1.0)
    b, _ = s.step(md, 500, xd, eta=1.0)
    assert torch.isfinite(a).all() and torch.isfinite(b).all()
    base, _ = s.step(md, 500, xd, eta=1.0, noise=torch.zeros_like(xd))
    sigma = s.step_coefficients(500, 1.0)["sigma"]
    za, zb = (a - base) / sigma, (b - base) / sigma               # the z each step drew
    assert rel_err(za, zb) > 0.5 and 0.8 < float(za.std()) < 1.2


def test_ddim_step_custom_op_and_opcheck():
    import medical_image_generation_b200.custom_ops  # noqa: F401
    g = torch.Generator().manual_seed(9)
    s = mig.DDIMScheduler(**dict(LDM, prediction_type="v_prediction"))
    s.set_timesteps(50)
    (m, x, z), (md, xd, zd) = _operands((2, 3, 6, 6, 6), torch.float32, False, g)
    k = s.step_coefficients(640, 0.5)
    args = (md, xd, zd, k["sqrt_acp"], k["sqrt_one_minus_acp"], k["sqrt_acp_prev"], k["dir_coef"], k["sigma"], 2, True)
    prev, x0 = torch.ops.medimgen_b200.ddim_step(*args)
    want, wx0 = s.step(md, 640, xd, eta=0.5, noise=zd)
    assert torch.equal(prev, want) and torch.equal(x0, wx0)
    assert "Tensor" in str(torch.ops.medimgen_b200.ddim_step.default._schema)
    torch.library.opcheck(torch.ops.medimgen_b200.ddim_step.default, args,
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    torch.library.opcheck(torch.ops.medimgen_b200.ddim_step.default, (md, xd, None, *args[3:7], 0.0, 2, False),
                          test_utils=("test_schema", "test_faketensor"))
    with pytest.raises(RuntimeError, match="one shape"):
        torch.ops.medimgen_b200.ddim_step(md[:1], *args[1:])


# ---- end to end with an analytic model ----------------------------------------------------------------------------------
class PointMassEps(torch.nn.Module):
    """The exact epsilon of a data distribution concentrated on x*: eps(x, t) = (x - sqrt(a_t) x*) / sqrt(1 - a_t).
    The alpha_bar table is indexed with the timestep tensor on the device, so the forward can be graph-captured."""

    def __init__(self, x_star, alphas_cumprod):
        super().__init__()
        self.x_star = torch.nn.Parameter(x_star.clone(), requires_grad=False)
        self.register_buffer("acp", alphas_cumprod.clone())

    def forward(self, x, timesteps, context=None):
        a = self.acp[timesteps.long()].reshape(-1, *([1] * (x.ndim - 1)))
        return (x - a.sqrt() * self.x_star) / (1 - a).sqrt()


def _point_mass(shape, seed=12):
    g = torch.Generator().manual_seed(seed)
    x_star = (torch.rand(shape, generator=g) * 1.8 - 0.9).to(DEV)      # inside [-1, 1]: the default clipping is a no-op
    s = mig.DDIMScheduler(**LDM)
    return s, x_star, PointMassEps(x_star, s.alphas_cumprod).to(DEV)


def test_ddim_sampling_recovers_the_point_mass_through_the_inferers():
    shape = (1, 1, 16, 16, 12)
    s, x_star, model = _point_mass(shape)
    s.set_timesteps(50)
    noise = torch.randn(shape, generator=torch.Generator().manual_seed(1)).to(DEV)
    inf = mig.DiffusionInferer(s)
    errs = {}
    for graph in (False, True):
        out = inf.sample(noise, model, s, verbose=False, cuda_graph=graph)
        errs[f"graph={graph}"] = rel_err(out, x_star)
    from medical_image_generation_b200.engine import sample_volumes
    vols = sample_volumes(model, s, shape[1:], 2, num_inference_steps=50)
    assert len(s.timesteps) == 50 and s.noise_mode == "device"
    for v, vol in vols.items():
        errs[f"sample_volumes[{v}]"] = rel_err(vol, x_star)
    assert max(errs.values()) < 1e-7, errs             # measured 1.9e-9 on a B200
    # eta = 1 through the same inferer: on a point mass x0_hat is x* from any state, and the last step has sigma = 0
    zs = [torch.randn(shape, generator=torch.Generator().manual_seed(20 + i)).to(DEV) for i in range(50)]
    s_eta = mig.DDIMScheduler(**LDM)
    s_eta.set_timesteps(50)
    s_eta.step = lambda out, t, img, noise=None: mig.DDIMScheduler.step(s_eta, out, t, img, eta=1.0, noise=noise)
    out = inf.sample(noise, model, s_eta, verbose=False, step_noises=zs)
    errs["eta=1"] = rel_err(out, x_star)
    print(f"point mass, DDIM-50: {errs}")
    assert errs["eta=1"] < 1e-7, errs                 # measured 1.8e-9


def test_ddim_latent_sampling_decodes_the_point_mass():
    ae = mig.AutoencoderKL(spatial_dims=3, in_channels=1, out_channels=1, num_res_blocks=1, num_channels=(16, 32),
                           attention_levels=(False, False), latent_channels=3, norm_num_groups=8,
                           with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False,
                           downsample_parameters=[[[1, 1, 1], [3, 3, 3], [1, 1, 1]], [[2, 2, 2], [3, 3, 3], [1, 1, 1]]],
                           upsample_parameters=[[[2, 2, 2], [3, 3, 3], [1, 1, 1]]],
                           compute_dtype=torch.float32).to(DEV).eval()
    shape = (1, 3, 8, 16, 16)
    s, x_star, model = _point_mass(shape, seed=13)
    s.set_timesteps(50)
    scale = 0.7
    noise = torch.randn(shape, generator=torch.Generator().manual_seed(2)).to(DEV)
    inf = mig.LatentDiffusionInferer(s, scale_factor=scale)
    with torch.no_grad():
        want = ae.decode_stage_2_outputs(x_star / scale)
        for graph in (False, True):
            img = inf.sample(noise, autoencoder_model=ae, diffusion_model=model, scheduler=s, verbose=False,
                             cuda_graph=graph)
            assert img.shape == (1, 1, 16, 32, 32)
            err = rel_err(img, want)
            print(f"latent point mass, DDIM-50, cuda_graph={graph}: {err:.2e}")
            assert err < 1e-5, graph                       # measured 0.9-1.1e-6 (fp32 decoder)


def test_ddim_inversion_walks_the_forward_marginals_and_back():
    shape = (2, 1, 12, 12, 8)
    s, x_star, model = _point_mass(shape, seed=14)
    s.set_timesteps(50)
    ratio = 1000 // 50
    up = [int(t) for t in s.timesteps.flip(0)]                           # 0, 20, ..., 980
    with torch.no_grad():
        eps_c = model(x_star, torch.zeros(2, device=DEV))
        x = x_star.clone()
        worst = 0.0
        for t in up[:-1]:
            x, _ = s.reversed_step(model(x, torch.full((2,), float(t), device=DEV)), t, x)
            want = s.add_noise(x_star, eps_c, torch.full((2,), t + ratio, device=DEV, dtype=torch.int64))
            worst = max(worst, rel_err(x, want))
        print(f"inversion: worst state vs add_noise(x*, eps_c, t) {worst:.2e}")
        assert worst < 3e-5, worst     # measured 8.7e-6: near t = 980 the state is ~0.03 x*, so its norm is small
        with pytest.raises(IndexError):
            s.reversed_step(model(x, torch.full((2,), float(up[-1]), device=DEV)), up[-1], x)
        for t in s.timesteps:
            x, _ = s.step(model(x, torch.full((2,), float(t), device=DEV)), t, x)
        print(f"inversion and back: {rel_err(x, x_star):.2e}")
        assert rel_err(x, x_star) < 1e-7                # measured 2.5e-9


# ---- the benchmark's sampling model ---------------------------------------------------------------------------------------
# The sampled state is fp32 (the U-Net computes in bf16 and its output is cast): worst over the 50 steps on an NVIDIA B200
# at its 1000 W limit, prev / x0: global 4.3e-8 / 3.1e-8, per voxel 2.1e-7 / 1.1e-7, per channel as global (one channel).
STEP_BARS = dict(glob=5e-7, row=2e-6, col=5e-7)


def test_config4_ddim_50_steps_every_step_vs_fp64_oracle():
    import bench
    torch.manual_seed(7)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.SAMPLING_CFG, compute_dtype=torch.bfloat16))
    model = model.to(DEV).eval()
    s, o = mig.DDIMScheduler(**LDM), OracleDDIMScheduler(**LDM)
    s.set_timesteps(50)
    o.set_timesteps(50)
    s.noise_mode = "device"
    worst = {"prev": {"glob": 0.0, "row": 0.0, "col": 0.0}, "x0": {"glob": 0.0, "row": 0.0, "col": 0.0}}
    seen = []

    def checked_step(out, t, img, noise=None):
        prev, x0 = mig.DDIMScheduler.step(s, out, t, img, noise=noise)
        wprev, wx0 = o.step(out.double().cpu(), int(t), img.double().cpu())
        for name, got, want in (("prev", prev, wprev), ("x0", x0, wx0)):
            e = assert_close_local(got, want, **STEP_BARS, what=f"{name} at t={int(t)}")
            for k in worst[name]:
                worst[name][k] = max(worst[name][k], e[k])
        seen.append(int(t))
        return prev, x0

    s.step = checked_step
    noise = torch.randn((1, *bench.VOLUME), generator=torch.Generator().manual_seed(42)).to(DEV)
    vol = mig.DiffusionInferer(s).sample(noise, model, s, verbose=False, cuda_graph=True)
    assert seen == [int(t) for t in s.timesteps] and len(seen) == 50
    assert torch.isfinite(vol).all()
    print(f"config-4 DDIM-50 worst per-step errors vs fp64 ({vol.dtype} state): {worst}")
