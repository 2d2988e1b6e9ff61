"""GPU: the fused variational-bound kernel (mig_ddpm_vlb_term) against the CPU oracle, and get_likelihood end to end
through the public inferers (eager and CUDA-graph), the latent inferer with resampling, and the generative shim."""
import pytest
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import _lib, compat, ops, planner
from oracle import likelihood_oracle as L
from oracle.ddpm_oracle import OracleDDPMScheduler
from util import bf16_round, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
LDM = planner.LDM_SCHEDULER_KWARGS
HALF_BIN = 0.5 / 255
# Arithmetic is fp32 for both storages (bf16 only rounds the operands, which the oracle sees rounded too), so one set of
# bars serves both. The kernel forms x0_hat with ddpm_step's expression, whose x_t - sqrt(1 - acp) * m the compiler
# contracts into one FMA where the oracle rounds twice; where that difference cancels against x0 the map differs by
# more than 2e-6: worst 6.3e-6 (fixed_large, clip off) on an NVIDIA B200 at its 1000 W limit. Means: worst 1.5e-6.
MAP_TOL, MEAN_TOL = 1e-5, 1e-5


def _run(s, m, xt, x0, t, with_map=True):
    """One kernel call through the scheduler's launch helper: (total (B,) fp64, map or None)."""
    m, x, z = s._vlb_operands(m, xt, x0)
    B = x.shape[0]
    ts = torch.full((B,), t, dtype=torch.int64, device=DEV)
    total = torch.zeros(B, dtype=torch.float64, device=DEV)
    kl = torch.empty_like(x, dtype=torch.float32) if with_map else None
    s._vlb_term(m, ts, x, z, total, s._vlb_workspace(x), kl, HALF_BIN)
    return total, kl


def _operands(shape, dtype, pred, g):
    """Host fp32 (m, x_t, x_0) exactly representable in `dtype`; x_0 in [-1, 1] with some voxels at +-1."""
    m = torch.randn(shape, generator=g) * (0.7 if pred == "sample" else 1.0)
    xt = torch.randn(shape, generator=g) * 1.2
    x0 = torch.rand(shape, generator=g) * 2 - 1
    x0.view(-1)[::7] = 1.0
    x0.view(-1)[3::11] = -1.0
    host = [m, xt, x0]
    if dtype == torch.bfloat16:
        host = [bf16_round(h) for h in host]
    return host


# 375 / 153 elements per sample: not a multiple of the 16-byte vector (scalar path); channels-last 8 x 4^3: vector path
# with strided operands; 2 x 3 x 8^3 contiguous: vector path
LAYOUTS = [((2, 3, 5, 5, 5), False), ((3, 1, 17, 9, 1), False), ((2, 8, 4, 4, 4), True), ((2, 3, 8, 8, 8), False)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_vlb_kernel_vs_oracle(dtype, pred):
    g = torch.Generator().manual_seed(1)
    worst = {"map": 0.0, "mean": 0.0}
    edge_voxels = 0
    for vt in ("fixed_small", "fixed_large"):
        for clip in (True, False):
            kw = dict(LDM, prediction_type=pred, variance_type=vt, clip_sample=clip)
            s, o = mig.DDPMScheduler(**kw), OracleDDPMScheduler(**kw)
            for shape, cl in LAYOUTS:
                B = shape[0]
                for t in (999, 500, 1, 0):
                    host = _operands(shape, dtype, pred, g)
                    dev = [h.to(DEV, dtype) for h in host]
                    if cl:
                        dev = [d.contiguous(memory_format=torch.channels_last_3d) for d in dev]
                    total, kl = _run(s, *dev, t)
                    total_nomap, _ = _run(s, *dev, t, with_map=False)
                    assert torch.equal(total, total_nomap), "the map changed the reduction"
                    assert kl.stride() == dev[1].stride()
                    want = L.vlb_term(o, host[0], t, host[1], host[2])
                    got = kl.cpu()
                    want_mean = want.view(B, -1).double().mean(1)
                    what = (vt, clip, shape, cl, t)
                    if t == 0 and vt == "fixed_small":
                        # a scale of 1e-10: the decoder term is a step function of |x0 - mu| at half the bin width, so
                        # kernel and oracle may differ only where |x0 - mu| is within rounding of that edge
                        m, xt, x0 = (h.double() for h in host)
                        bad = (got - want).abs() > MAP_TOL * (want.abs() + 1)
                        if bad.any():
                            k = s.vlb_coefficients()[0].double()
                            if pred == "epsilon":
                                x0h = (xt - k[1] * m) / k[0]
                            elif pred == "sample":
                                x0h = m
                            else:
                                x0h = k[0] * xt - k[1] * m
                            if clip:
                                x0h = x0h.clamp(-1, 1)
                            dist = ((x0 - k[2] * x0h).abs() - HALF_BIN).abs()
                            assert bool((dist[bad] < 1e-6).all()), (what, dist[bad])
                            edge_voxels += int(bad.sum())
                        good = ~bad
                        assert rel_err(got[good], want[good]) < MAP_TOL, what
                        continue
                    e_map = rel_err(got, want)
                    e_mean = float(((total.cpu() - want_mean).abs() / want_mean.abs().clamp_min(1e-30)).max())
                    worst["map"], worst["mean"] = max(worst["map"], e_map), max(worst["mean"], e_mean)
                    assert e_map < MAP_TOL and e_mean < MEAN_TOL, (what, e_map, e_mean)
    print(f"vlb kernel {dtype} {pred}: worst map {worst['map']:.2e}, worst mean {worst['mean']:.2e}, "
          f"decoder voxels on the bin edge {edge_voxels}")


def test_vlb_kernel_is_deterministic_and_accumulates():
    g = torch.Generator().manual_seed(2)
    s = mig.DDPMScheduler(**LDM)
    dev = [h.to(DEV) for h in _operands((2, 4, 32, 32, 16), torch.float32, "epsilon", g)]
    m, x, z = s._vlb_operands(*dev)
    ts = torch.full((2,), 300, dtype=torch.int64, device=DEV)
    ws = s._vlb_workspace(x)
    runs = []
    for _ in range(2):
        total = torch.zeros(2, dtype=torch.float64, device=DEV)
        kl = torch.empty_like(x)
        s._vlb_term(m, ts, x, z, total, ws, kl, HALF_BIN)
        one = total.clone()
        s._vlb_term(m, ts, x, z, total, ws, kl, HALF_BIN)      # adds, never overwrites
        runs.append((one, total, kl))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][2], runs[1][2])
    assert torch.equal(runs[0][1], 2 * runs[0][0])


def test_vlb_abi_rejections():
    s = mig.DDPMScheduler(**LDM)
    x = torch.randn(2, 1, 4, 4, 4, device=DEV)
    ts = torch.full((2,), 5, dtype=torch.int64, device=DEV)
    total = torch.zeros(2, dtype=torch.float64, device=DEV)
    table = s._vlb_table_on(x.device)
    ws = s._vlb_workspace(x)
    p = ops._ptr
    lib = _lib.load()
    assert lib.mig_ddpm_vlb_workspace_bytes(0, 64) == -1 and lib.mig_ddpm_vlb_workspace_bytes(2, 0) == -1
    assert lib.mig_ddpm_vlb_workspace_bytes(2, 64) == ws.numel()

    def call(dtype=0, ptrs=None, table_len=None, T=1000, B=2, per=64, pred=0, half=HALF_BIN, ws_bytes=None):
        args = ptrs or (p(x), p(x), p(x), p(ts), p(table))
        _lib.call("mig_ddpm_vlb_term", dtype, *args, table.numel() if table_len is None else table_len, T, B, per, pred,
                  1, half, None, p(total), p(ws), ws.numel() if ws_bytes is None else ws_bytes, ops._stream())

    call()                                                   # the valid call
    for kw, msg in ((dict(table_len=7 * 999), "coefficient table"), (dict(T=999), "coefficient table"),
                    (dict(ws_bytes=8), "workspace too small"), (dict(pred=3), "prediction"), (dict(B=0), "batch"),
                    (dict(per=0), "at least one element"), (dict(half=-1.0), "half bin"),
                    (dict(ptrs=(p(x), p(x), None, p(ts), p(table))), "must not be NULL"), (dict(dtype=7), "dtype")):
        with pytest.raises(RuntimeError, match=msg):
            call(**kw)
    with pytest.raises(RuntimeError, match="timesteps"):
        s._vlb_term(x, ts.float(), x, x, total, ws)
    torch.cuda.synchronize()


# ---- end to end through the inferers --------------------------------------------------------------------------------
class PointMassEps(torch.nn.Module):
    """The exact epsilon of data concentrated on x*: eps(x, t) = (x - sqrt(a_t) x*) / sqrt(1 - a_t), so x0_hat = x*
    and every KL term is 0.5 (c + c0^2 (x0 - x*)^2 / var). Indexes alpha_bar with the device timesteps, so it can be
    graph-captured."""

    def __init__(self, x_star, alphas_cumprod):
        super().__init__()
        self.register_buffer("x_star", x_star.clone())
        self.register_buffer("acp", alphas_cumprod.clone())

    def forward(self, x, timesteps, context=None):
        a = self.acp[timesteps.long()].reshape(-1, *([1] * (x.ndim - 1)))
        return (x[:, :self.x_star.shape[1]] - a.sqrt() * self.x_star) / (1 - a).sqrt()


def _point_mass_problem(shape, seed):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(shape, generator=g) * 2 - 1
    x0.view(-1)[::13] = 1.0
    x_star = (x0 + 0.05 * torch.randn(shape, generator=g)).clamp(-0.95, 0.95)
    noise = torch.randn(shape, generator=g)
    return x0, x_star, noise


@pytest.mark.parametrize("variance_type", ["fixed_small", "fixed_large"])
def test_point_mass_likelihood_graph_equals_eager_and_oracle(variance_type):
    shape = (2, 1, 16, 16, 12)
    x0, x_star, noise = _point_mass_problem(shape, 3)
    s = mig.DDPMScheduler(variance_type=variance_type, **LDM)
    o = OracleDDPMScheduler(variance_type=variance_type, **LDM)
    model = PointMassEps(x_star, s.alphas_cumprod).to(DEV)
    inf = mig.DiffusionInferer(s)
    got = {}
    for graph in (False, True):
        got[graph] = inf.get_likelihood(x0.to(DEV), model, save_intermediates=True, verbose=False, noise=noise.to(DEV),
                                        cuda_graph=graph)
    assert got[False][0].dtype == torch.float32 and got[False][0].shape == (2,) and got[False][0].is_cuda
    assert torch.equal(got[False][0], got[True][0]), "graph and eager totals differ"
    assert len(got[True][1]) == 1000 and all(torch.equal(a, b) for a, b in zip(got[False][1], got[True][1]))
    assert all(k.device.type == "cpu" and k.dtype == torch.float32 and k.shape == shape for k in got[True][1])
    want, want_inter = L.get_likelihood(o, x0, PointMassEps(x_star, o.alphas_cumprod), save_intermediates=True,
                                        noise=noise)
    err = float(((got[True][0].cpu().double() - want.double()).abs() / want.double().abs()).max())
    sums = torch.stack([k.view(2, -1).double().mean(1) for k in got[True][1]]).sum(0)
    print(f"point mass {variance_type}: total {got[True][0].tolist()}, oracle {want.tolist()}, rel err {err:.2e}")
    assert err < MEAN_TOL, err
    assert torch.allclose(sums, got[True][0].cpu().double(), rtol=1e-6, atol=0)
    # t = 1 (the largest KL weight) map against the oracle's
    assert rel_err(got[True][1][-2], want_inter[-2]) < 1e-5


def test_concat_mode_and_scheduler_argument():
    """concat: the conditioning is concatenated on the channel axis and the model gets context=None. The `scheduler`
    argument (a short schedule) drives the loop and the coefficients; x_t comes from the inferer's scheduler."""
    shape = (2, 2, 12, 12, 8)
    x0, x_star, noise = _point_mass_problem(shape, 4)
    cond = torch.randn(2, 1, 12, 12, 8, generator=torch.Generator().manual_seed(5))
    s = mig.DDPMScheduler(**LDM)
    short = mig.DDPMScheduler(**dict(LDM, prediction_type="epsilon"), clip_sample=False)
    short.set_timesteps(50)
    o, o_short = OracleDDPMScheduler(**LDM), OracleDDPMScheduler(**LDM, clip_sample=False)
    o_short.set_timesteps(50)

    class ConcatModel(torch.nn.Module):
        def __init__(self, pm):
            super().__init__()
            self.pm = pm

        def forward(self, x, timesteps, context=None):
            assert context is None and x.shape[1] == 3
            return self.pm(x, timesteps) + 0.1 * x[:, 2:3]

    model = ConcatModel(PointMassEps(x_star, s.alphas_cumprod)).to(DEV)
    inf = mig.DiffusionInferer(s)
    got = [inf.get_likelihood(x0.to(DEV), model, scheduler=short, conditioning=cond.to(DEV), mode="concat",
                              noise=noise.to(DEV), cuda_graph=g) for g in (False, True)]
    assert torch.equal(got[0], got[1])
    want = L.get_likelihood(o, x0, ConcatModel(PointMassEps(x_star, o.alphas_cumprod)), scheduler=o_short,
                            conditioning=cond, mode="concat", noise=noise)
    err = float(((got[1].cpu().double() - want.double()).abs() / want.double().abs()).max())
    print(f"concat, 50 steps: rel err {err:.2e}")
    assert err < MEAN_TOL, err


def _small_unet(dtype):
    import bench
    torch.manual_seed(11)
    model = mig.DiffusionModelUNet(spatial_dims=3, in_channels=1, out_channels=1, num_res_blocks=1,
                                   num_channels=[16, 32], attention_levels=[False, True], num_head_channels=[0, 32],
                                   norm_num_groups=8, strides=[[1, 1, 1], [2, 2, 2]], kernel_sizes=[[3, 3, 3]] * 2,
                                   paddings=[[1, 1, 1]] * 2, compute_dtype=dtype)
    return bench.rerandomize_zero_init(model).to(DEV).eval()     # else the zero-initialised output conv gives eps = 0


def test_small_unet_likelihood_vs_oracle_on_recorded_outputs():
    shape = (2, 1, 16, 16, 16)
    x0, _, noise = _point_mass_problem(shape, 6)
    model = _small_unet(torch.float32)
    s, o = mig.DDPMScheduler(**LDM), OracleDDPMScheduler(**LDM)
    s.set_timesteps(25)
    o.set_timesteps(25)
    recorded = []

    def recording(x, timesteps, context=None):
        out = model(x, timesteps, context)
        recorded.append(out.detach().float().cpu())
        return out

    inf = mig.DiffusionInferer(s)
    total, inter = inf.get_likelihood(x0.to(DEV), recording, save_intermediates=True, noise=noise.to(DEV))
    replay = iter(recorded)
    want, want_inter = L.get_likelihood(o, x0, lambda x, timesteps, context: next(replay), save_intermediates=True,
                                        noise=noise)
    err = float(((total.cpu().double() - want.double()).abs() / want.double().abs()).max())
    e_maps = max(rel_err(a, b) for a, b in zip(inter[:-1], want_inter[:-1]))
    graph = inf.get_likelihood(x0.to(DEV), model, noise=noise.to(DEV), cuda_graph=True)
    e_graph = float(((graph - total).abs() / total.abs()).max())
    print(f"small U-Net, 25 steps: total {total.tolist()} vs oracle rel {err:.2e}, t > 0 maps {e_maps:.2e}, "
          f"graph vs eager {e_graph:.2e}")
    assert err < MEAN_TOL and e_maps < 1e-5, (err, e_maps)
    assert e_graph < 1e-5, e_graph     # GroupNorm statistics are summed with atomics: not bit-reproducible


def test_latent_likelihood_with_resampling_matches_the_pixel_path():
    ae = mig.AutoencoderKL(spatial_dims=3, in_channels=1, out_channels=1, num_res_blocks=1, num_channels=(16, 32),
                           attention_levels=(False, False), latent_channels=3, norm_num_groups=8,
                           with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False,
                           downsample_parameters=[[[1, 1, 1], [3, 3, 3], [1, 1, 1]], [[2, 2, 2], [3, 3, 3], [1, 1, 1]]],
                           upsample_parameters=[[[2, 2, 2], [3, 3, 3], [1, 1, 1]]],
                           compute_dtype=torch.float32).to(DEV).eval()
    images = torch.rand(2, 1, 16, 16, 16, generator=torch.Generator().manual_seed(7)).to(DEV)
    scale = 0.7
    s = mig.DDPMScheduler(**LDM)
    s.set_timesteps(20)
    # encode_stage_2_inputs draws the latent sample: the same seed before each encoding gives the same latents
    torch.manual_seed(123)
    with torch.no_grad():
        latents = ops.scale(ae.encode_stage_2_inputs(images), scale)
    g = torch.Generator().manual_seed(8)
    x_star = (latents.cpu() + 0.05 * torch.randn(latents.shape, generator=g)).clamp(-0.95, 0.95)
    noise = torch.randn(latents.shape, generator=g).to(DEV)
    model = PointMassEps(x_star, s.alphas_cumprod).to(DEV)
    lat = mig.LatentDiffusionInferer(s, scale_factor=scale)
    torch.manual_seed(123)
    total, maps = lat.get_likelihood(images, ae, model, save_intermediates=True, resample_latent_likelihoods=True,
                                     resample_interpolation_mode="trilinear", noise=noise, cuda_graph=True)
    want, want_maps = mig.DiffusionInferer(s).get_likelihood(latents, model, save_intermediates=True, noise=noise)
    assert len(maps) == 20 and all(m.shape == (2, 3, 16, 16, 16) and m.device.type == "cpu" for m in maps)
    up = torch.nn.Upsample(size=(16, 16, 16), mode="trilinear")
    e_total = float(((total - want).abs() / want.abs()).max())
    e_maps = max(rel_err(a, up(b)) for a, b in zip(maps, want_maps))
    print(f"latent vs pixel path: total {e_total:.2e}, resampled maps {e_maps:.2e}")
    # the encoder's GroupNorm statistics are summed with atomics, so the two encodings may differ in the last bits;
    # x0_hat amplifies that by 1 / sqrt(acp_t) at large t: measured total 0, maps 1.0e-5
    assert e_total < 1e-5 and e_maps < 1e-4, (e_total, e_maps)
    plain = lat.get_likelihood(images, ae, model, save_intermediates=True, noise=noise)
    assert plain[1][0].shape == (2, 3, 8, 8, 8)


def test_generative_shim_get_likelihood():
    import importlib.util
    if importlib.util.find_spec("generative") is not None and "shims" not in importlib.util.find_spec(
            "generative").origin:
        pytest.skip("a real monai-generative is installed")
    compat.install()
    try:
        from generative.inferers import DiffusionInferer, LatentDiffusionInferer
        from generative.networks.schedulers import DDPMScheduler
        assert DiffusionInferer is mig.DiffusionInferer and LatentDiffusionInferer is mig.LatentDiffusionInferer
        shape = (1, 1, 8, 8, 8)
        x0, x_star, noise = _point_mass_problem(shape, 9)
        s = DDPMScheduler(**LDM)
        model = PointMassEps(x_star, s.alphas_cumprod).to(DEV)
        inf = DiffusionInferer(s)
        a = inf.get_likelihood(x0.to(DEV), model, noise=noise.to(DEV))
        b = inf.get_likelihood(x0.to(DEV), model, noise=noise.to(DEV))
        assert torch.equal(a, b) and torch.isfinite(a).all()
    finally:
        compat.uninstall()
