"""GPU: whole-model and per-block parity of the B200 modules against (a) the committed golden vectors produced
by the UNMODIFIED reference and (b) the CPU oracle run live on the same seeded inputs.
fp32 path: 1e-4 relative; bf16 path: 2e-2 relative (BASELINE.json north_star)."""
import pytest
import torch
import torch.nn.functional as F

from util import BF16_TOL, FP32_TOL, graph_vs_eager, rel_err, tol_for

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _build(g, dtype):
    import medical_image_generation_b200 as mig
    from oracle.golden_util import golden_params
    cls = mig.DiffusionModelUNet if g["kind"] == "unet" else mig.AutoencoderKL
    m = cls(**g["cfg"], compute_dtype=dtype)
    params = golden_params(g["shapes"], g["seed"])
    m.load_state_dict(params)
    return m.to(DEV).train(), params


# unet3d_ldm_width: BASELINE config 3 at FULL width (256/512/768, 441 M parameters, single 512-/768-channel heads) on 2x3x8^3
UNETS = ["unet3d_small", "unet3d_aniso", "unet2d_small", "unet3d_cond", "unet3d_updown", "unet3d_ldm_width"]
AES = ["ae3d_small", "ae3d_attn_aniso", "ae2d_small", "ae3d_convtranspose"]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", UNETS)
def test_unet_matches_reference_golden(golden, name, dtype):
    from oracle.golden_util import sketch
    g = golden(name)
    m, _ = _build(g, dtype)
    inp = g["inputs"]
    x = inp["x"].to(DEV).requires_grad_(True)
    kw = {}
    if "context" in inp:
        kw = dict(context=inp["context"].to(DEV), class_labels=inp["class_labels"].to(DEV))
    taps = {}
    hooks = [m.conv_in.register_forward_hook(lambda _m, _i, o: taps.__setitem__("conv_in", o)),
             m.middle_block.register_forward_hook(lambda _m, _i, o: taps.__setitem__("mid", o)),
             m.down_blocks[0].resnets[0].register_forward_hook(lambda _m, _i, o: taps.__setitem__("down0_res0", o)),
             m.up_blocks[0].register_forward_hook(lambda _m, _i, o: taps.__setitem__("up0", o))]
    y = m(x, inp["timesteps"].to(DEV), **kw)
    for h in hooks:
        h.remove()
    tol = tol_for(dtype)
    assert y.shape == g["out"].shape and y.dtype == torch.float32
    for k in ("conv_in", "down0_res0", "mid", "up0"):                    # per-block outputs
        assert rel_err(taps[k], g["taps"][k]) < tol, k
    assert rel_err(y, g["out"]) < tol
    (y * inp["probe"].to(DEV)).sum().backward()
    gtol = tol * (1 if dtype == torch.float32 else 2.5)   # bf16 activation grads pass through ~40 rounding layers
    assert rel_err(x.grad, g["grad_x"]) < gtol
    named = dict(m.named_parameters())
    for k in g["no_grad_params"]:
        assert named[k].grad is None, k
    worst, worst_key = 0.0, None
    for k, sk in g["grad_sketch"].items():
        assert named[k].grad is not None, k
        if k.endswith("to_k.bias"):
            # softmax is invariant to a shift of all keys, so d loss / d to_k.bias is EXACTLY zero mathematically;
            # both sides hold rounding noise only. Check it is negligible next to the matching to_q.bias gradient.
            qn = float(named[k.replace("to_k", "to_q")].grad.norm())
            assert float(named[k].grad.norm()) < 0.05 * qn + 1e-4, k
            continue
        if float(sk[2]) ** 0.5 < 1e-4:
            # also exactly zero mathematically: with one channel per group (G == C) GroupNorm removes any per-(n,c)
            # constant, so the time-embedding projection of that block gets no gradient. Noise only, both sides.
            assert float(named[k].grad.norm()) < (1e-3 if dtype == torch.float32 else 0.1), k
            continue
        e = rel_err(sketch(named[k].grad), sk, floor=0.1)
        if e > worst:
            worst, worst_key = e, k
    assert worst < (1e-3 if dtype == torch.float32 else 8e-2), (worst, worst_key)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", AES)
def test_autoencoder_matches_reference_golden(golden, name, dtype):
    from medical_image_generation_b200 import ops
    from oracle.golden_util import sketch
    g = golden(name)
    m, _ = _build(g, dtype)
    inp = g["inputs"]
    x = inp["x"].to(DEV).requires_grad_(True)
    z_mu, z_sigma = m.encode(x)
    z = ops.vae_reparam(z_mu, z_sigma, inp["eps"].to(DEV))   # sampling() with the golden's noise injected (ae:786)
    recon = m.decode(z)
    tol = tol_for(dtype)
    assert rel_err(z_mu, g["z_mu"]) < tol and rel_err(z_sigma, g["z_sigma"]) < tol
    assert rel_err(recon, g["out"]) < tol
    kl = ops.kl_loss(z_mu, z_sigma)
    loss = ops.l1_loss(recon, x.detach()) + 1e-7 * kl          # train_autoencoder.py:412-414
    assert rel_err(kl, g["kl"]) < tol and rel_err(loss, g["loss"]) < tol
    loss.backward()
    gtol = 1e-3 if dtype == torch.float32 else 0.25           # L1's sign() gradient flips on rounding noise
    assert rel_err(x.grad, g["grad_x"]) < gtol
    named = dict(m.named_parameters())
    worst = max(rel_err(sketch(named[k].grad), sk, floor=0.1) for k, sk in g["grad_sketch"].items())
    assert worst < (2e-3 if dtype == torch.float32 else 0.25), worst


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_per_block_parity_vs_oracle(dtype):
    """ResnetBlock / AttentionBlock / Downsample / Upsample called directly with NCDHW tensors, like a user of the
    reference would, against the oracle's block functions."""
    from medical_image_generation_b200 import unet as U, layers
    from oracle import torch_oracle as O
    g = torch.Generator().manual_seed(21)
    tol = tol_for(dtype)

    def randomise(mod):
        with torch.no_grad():
            for p in mod.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * (0.2 if p.ndim > 1 else 0.3) + (1.0 if p.ndim == 1 and p.shape[0] > 0 and False else 0.0))
        return mod

    x = torch.randn(2, 32, 6, 6, 6, generator=g)
    emb = torch.randn(2, 64, generator=g)
    rb = randomise(U.ResnetBlock(3, 32, 64, 48, norm_num_groups=16)).to(DEV)
    sd = {"blk." + k: v.detach().cpu().contiguous() for k, v in rb.state_dict().items()}
    want = O.unet_resnet_block(sd, "blk", x, emb, 16, 1e-6)
    got = rb(x.to(DEV).to(dtype), emb.to(DEV))
    assert got.shape == want.shape and rel_err(got, want) < tol

    ab = randomise(layers.SelfAttentionBlock(3, 32, 16, norm_num_groups=16)).to(DEV)
    sd = {"blk." + k: v.detach().cpu().contiguous() for k, v in ab.state_dict().items()}
    want = O.self_attention_block(sd, "blk", x, 16, 1e-6, 16)
    assert rel_err(ab(x.to(DEV).to(dtype)), want) < tol

    ds = randomise(U.Downsample(3, 32, True, 32, stride=[2, 2, 1], kernel_size=[3, 3, 3], padding=[1, 1, 1])).to(DEV)
    sd = {"blk." + k: v.detach().cpu().contiguous() for k, v in ds.state_dict().items()}
    want = O._conv(sd, "blk.op", x, [2, 2, 1], [1, 1, 1])
    assert rel_err(ds(x.to(DEV).to(dtype)), want) < tol

    up = randomise(U.Upsample(3, 32, True, 32, stride=[2, 2, 1], padding=[1, 1, 1])).to(DEV)
    sd = {"blk." + k: v.detach().cpu().contiguous() for k, v in up.state_dict().items()}
    want = O._conv(sd, "blk.conv", O._nearest_up(x, [2, 2, 1]), 1, [1, 1, 1])
    got = up(x.to(DEV).to(dtype))
    assert got.shape == want.shape and rel_err(got, want) < tol


def test_upsample_defect_raises_like_reference():
    """Planner output for a thin axis (kernel 1 / pad 0) breaks the reference U-Net's skip concat with a RuntimeError
    (SURVEY.md section 0.6); the drop-in must fail the same way, not silently 'fix' it."""
    import medical_image_generation_b200 as mig
    from oracle import torch_oracle as O
    p = O.compute_downsample_parameters([32, 32, 16], 3)
    m = mig.DiffusionModelUNet(spatial_dims=3, in_channels=2, out_channels=2, num_res_blocks=1,
                               num_channels=[16, 32, 32], attention_levels=[False, False, True],
                               num_head_channels=[0, 0, 32], norm_num_groups=16, strides=[q[0] for q in p],
                               kernel_sizes=[q[1] for q in p], paddings=[q[2] for q in p]).to(DEV)
    with pytest.raises(RuntimeError, match="[Ss]izes of tensors must match"):
        m(torch.randn(1, 2, 32, 32, 16, device=DEV), torch.tensor([5], device=DEV))


def test_inferer_sampling_loop_matches_oracle(golden):
    """DiffusionInferer.sample over 8 steps with injected per-step noise == oracle loop over the oracle U-Net."""
    import medical_image_generation_b200 as mig
    from oracle import torch_oracle as O
    from oracle.ddpm_oracle import OracleDDPMScheduler, OracleDiffusionInferer
    g = golden("unet3d_aniso")
    m, params = _build(g, torch.float32)
    m.eval()
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    s, o = mig.DDPMScheduler(**kw), OracleDDPMScheduler(**kw)
    s.set_timesteps(8); o.set_timesteps(8)
    assert torch.equal(s.timesteps.cpu(), o.timesteps)
    gen = torch.Generator().manual_seed(77)
    x = torch.randn(1, 1, 12, 12, 6, generator=gen)
    zs = [torch.randn(x.shape, generator=gen) for _ in range(8)]
    want = OracleDiffusionInferer(o).sample(
        x, lambda img, timesteps, context=None: O.unet_forward(params, g["cfg"], img, timesteps), o, step_noises=zs)
    got = mig.DiffusionInferer(s).sample(x.to(DEV), m, s, verbose=False, step_noises=[z.to(DEV) for z in zs])
    assert rel_err(got, want) < 5e-4


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_single_timestep_broadcasts_over_the_batch(golden, dtype):
    """The inferers call the model with ONE timestep for the whole batch (`torch.Tensor((t,))`, train_ldm.py:356-362): the
    reference broadcasts temb[:, :, None, None, None] (unet:691-695). Batch 2 with a (1,) timestep must equal the oracle
    and the same samples run one by one (the fused epilogue indexes the time-embedding bias per sample)."""
    from oracle import torch_oracle as O
    g = golden("unet3d_aniso")
    m, params = _build(g, dtype)
    m.eval()
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2, 1, 12, 12, 6, generator=gen)
    t = torch.Tensor((417,))
    want = O.unet_forward(params, g["cfg"], x, t)
    with torch.no_grad():
        got = m(x.to(DEV), timesteps=t.to(DEV))
        one = torch.cat([m(x[i:i + 1].to(DEV), timesteps=t.to(DEV)) for i in range(2)])
    tol = 1e-4 if dtype == torch.float32 else BF16_TOL
    assert rel_err(got, want) < tol
    assert rel_err(got[1:], one[1:]) < (1e-5 if dtype == torch.float32 else BF16_TOL)   # batch-dependent reduction order
    # and through the sampler: two volumes in one batch == the oracle loop
    from oracle.ddpm_oracle import OracleDDPMScheduler, OracleDiffusionInferer
    import medical_image_generation_b200 as mig
    if dtype == torch.float32:
        kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
        s, o = mig.DDPMScheduler(**kw), OracleDDPMScheduler(**kw)
        s.set_timesteps(4); o.set_timesteps(4)
        zs = [torch.randn(x.shape, generator=gen) for _ in range(4)]
        want_s = OracleDiffusionInferer(o).sample(
            x, lambda img, timesteps, context=None: O.unet_forward(params, g["cfg"], img, timesteps), o, step_noises=zs)
        got_s = mig.DiffusionInferer(s).sample(x.to(DEV), m, s, verbose=False, step_noises=[z.to(DEV) for z in zs])
        assert rel_err(got_s, want_s) < 5e-4


def test_inferer_sampling_with_cuda_graph(golden):
    """sample(cuda_graph=True) replays one captured model forward per step and must reproduce the eager loop."""
    import medical_image_generation_b200 as mig
    g = golden("unet3d_aniso")
    m, _ = _build(g, torch.bfloat16)
    m.eval()
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    s = mig.DDPMScheduler(**kw)
    s.set_timesteps(6)
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(1, 1, 12, 12, 6, generator=gen).to(DEV)
    zs = [torch.randn(x.shape, generator=gen).to(DEV) for _ in range(6)]
    inf = mig.DiffusionInferer(s)
    eager = inf.sample(x, m, s, verbose=False, step_noises=zs)
    graphed = inf.sample(x, m, s, verbose=False, step_noises=zs, cuda_graph=True)
    assert torch.isfinite(graphed).all() and rel_err(graphed, eager) < 1e-3


def test_inferer_concat_conditioning(golden):
    """mode='concat' (upstream DiffusionInferer): the condition is concatenated to the noisy input along channels and
    no cross-attention context is passed; __call__ and sample() against the oracle U-Net on the same tensors."""
    import medical_image_generation_b200 as mig
    from oracle import torch_oracle as O
    from oracle.ddpm_oracle import OracleDDPMScheduler
    g = golden("unet3d_updown")          # in_channels = 2: one image channel + one condition channel
    m, params = _build(g, torch.float32)
    m.eval()
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    s, o = mig.DDPMScheduler(**kw), OracleDDPMScheduler(**kw)
    gen = torch.Generator().manual_seed(123)
    x0, noise, cond = (torch.randn(2, 1, 8, 8, 4, generator=gen) for _ in range(3))
    t = torch.randint(0, 1000, (2,), generator=gen)
    with torch.no_grad():
        got = mig.DiffusionInferer(s)(x0.to(DEV), m, noise.to(DEV), t.to(DEV), condition=cond.to(DEV), mode="concat")
        want = O.unet_forward(params, g["cfg"], torch.cat([o.add_noise(x0, noise, t), cond], dim=1), t)
    assert got.shape == want.shape and rel_err(got, want) < 5e-4
    with pytest.raises(NotImplementedError):
        mig.DiffusionInferer(s)(x0.to(DEV), m, noise.to(DEV), t.to(DEV), condition=cond.to(DEV), mode="film")


_CURVE_CACHE = {}


def _oracle_loss_curve(g, steps, lr):
    """`steps` AdamW steps of epsilon-prediction training (train_ldm.py:143-183 semantics) of the oracle U-Net driven
    by torch.optim.AdamW + clip_grad_norm_ on CPU fp32. Returns (losses, batches) so the CUDA path sees the same data."""
    from oracle import torch_oracle as O
    from oracle.ddpm_oracle import OracleDDPMScheduler
    from oracle.golden_util import golden_params
    key = (g["name"], steps, lr)
    if key in _CURVE_CACHE:
        return _CURVE_CACHE[key]
    ref_params = {k: v.clone().requires_grad_(True) for k, v in golden_params(g["shapes"], g["seed"]).items()}
    used = [ref_params[k] for k in ref_params if "proj_attn" not in k]
    opt_ref = torch.optim.AdamW(used, lr=lr)
    o = OracleDDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    gen = torch.Generator().manual_seed(5)
    B = g["batch"]
    shape = tuple(g["inputs"]["x"].shape[1:])
    curve, batches = [], []
    for _ in range(steps):
        x0 = torch.randn((B, *shape), generator=gen)
        noise = torch.randn(x0.shape, generator=gen)
        t = torch.randint(0, 1000, (B,), generator=gen)
        loss = torch.nn.functional.mse_loss(O.unet_forward(ref_params, g["cfg"], o.add_noise(x0, noise, t), t), noise)
        opt_ref.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(used, 1.0)
        opt_ref.step()
        curve.append(float(loss))
        batches.append((x0, noise, t))
    _CURVE_CACHE[key] = (curve, batches)
    return curve, batches


CURVE_STEPS = 200          # north_star: "200-step loss curves tracking"
CURVE_TOL_FP32 = 1e-2      # every one of the 200 losses within 1 % of the oracle's (fp32 CUDA-core path, torch AdamW)
CURVE_TOL_BF16_STEP = 0.10  # bf16 production path (flat fused AdamW, bf16 shadow weights): every loss within 10 % ...
CURVE_TOL_BF16_MEAN = 0.02  # ... and the mean |relative deviation| over the 200 steps within 2 %


def test_train_step_loss_curve_tracks_oracle_fp32(golden):
    """200 AdamW steps on the small anisotropic 3-D U-Net: fp32 CUDA path + torch.optim.AdamW vs the oracle on CPU, same
    data / noise / timesteps every step."""
    import medical_image_generation_b200 as mig
    g = golden("unet3d_aniso")
    curve_ref, batches = _oracle_loss_curve(g, CURVE_STEPS, 1e-4)
    m, _ = _build(g, torch.float32)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4)
    s = mig.DDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    curve = []
    for x0, noise, t in batches:
        pred = m(s.add_noise(x0.to(DEV), noise.to(DEV), t.to(DEV)), t.to(DEV))
        loss = mig.ops.mse_loss(pred, noise.to(DEV))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        opt.step()
        curve.append(float(loss))
    dev = [abs(a - b) / abs(b) for a, b in zip(curve, curve_ref)]
    print(f"fp32 loss curve: max rel dev {max(dev):.3e} (first 20: {max(dev[:20]):.3e}), loss {curve_ref[0]:.4f} -> {curve_ref[-1]:.4f}")
    assert max(dev[:20]) < 2e-3, dev[:20]
    assert max(dev) < CURVE_TOL_FP32, max(dev)
    assert sum(curve[-20:]) < sum(curve[:20])


def test_train_step_loss_curve_tracks_oracle_bf16(golden):
    """The PRODUCTION path over the same 200 steps: bf16 tensor-core kernels, engine.LDMTrainer (flat fused clip + AdamW,
    bf16 shadow weights) against the fp32 oracle + torch.optim.AdamW. bf16 rounding makes single losses wobble, so the
    bar is per-step <= 10 % and mean |deviation| <= 2 % (stated tolerances; fp32 bar is 1 %)."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_aniso")
    curve_ref, batches = _oracle_loss_curve(g, CURVE_STEPS, 1e-4)
    m, _ = _build(g, torch.bfloat16)
    s = mig.DDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    tr = LDMTrainer(m, s, lr=1e-4, grad_clip_max_norm=1.0)
    curve = [float(tr.step(x0.to(DEV), noise=noise.to(DEV), timesteps=t.to(DEV))) for x0, noise, t in batches]
    tr.opt.close()
    dev = [abs(a - b) / abs(b) for a, b in zip(curve, curve_ref)]
    print(f"bf16 loss curve: max rel dev {max(dev):.3e}, mean {sum(dev) / len(dev):.3e}")
    assert max(dev) < CURVE_TOL_BF16_STEP, max(dev)
    assert sum(dev) / len(dev) < CURVE_TOL_BF16_MEAN
    assert sum(curve[-20:]) < sum(curve[:20])


def test_shadow_follows_in_place_parameter_changes(golden):
    """Reference resume order (train_ldm.py:522-525): the optimiser exists BEFORE load_model() copies the checkpoint into
    the parameters. The bf16 shadow the tensor-core kernels read must follow such in-place changes of the fp32 master."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    from oracle.golden_util import golden_params
    g = golden("unet3d_small")
    s = mig.DDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    m = mig.DiffusionModelUNet(**g["cfg"], compute_dtype=torch.bfloat16).to(DEV)     # random init ...
    tr = LDMTrainer(m, s)                                                               # ... shadow = random init
    m.load_state_dict(golden_params(g["shapes"], g["seed"]))                            # checkpoint arrives afterwards
    fresh, _ = _build(g, torch.bfloat16)
    x = g["inputs"]["x"].to(DEV)
    t = g["inputs"]["timesteps"].to(DEV)
    with torch.no_grad():
        got, want = m.eval()(x, t), fresh.eval()(x, t)
    # (GroupNorm statistics are reduced with atomics: two bf16 runs of the SAME weights agree to <1e-2, stale weights not at all)
    assert rel_err(got, want) < BF16_TOL and rel_err(got, g["out"]) < BF16_TOL
    with torch.no_grad():   # a later manual edit of one filter is picked up as well
        m.conv_in.conv.weight.mul_(0.5)
        fresh.conv_in.conv.weight.mul_(0.5)
        assert rel_err(m(x, t), fresh(x, t)) < BF16_TOL
    tr.opt.close()


def test_graph_capture_failure_leaves_clean_state(golden, monkeypatch):
    """A failed CUDA-graph capture falls back to eager steps without leaving the host step counter ahead of the
    device counter (the captured-but-never-executed step must not count)."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_small")
    m, _ = _build(g, torch.bfloat16)
    s = mig.DDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    tr = LDMTrainer(m, s, cuda_graph=True, graph_warmup_steps=1)
    x = torch.randn(2, 3, 8, 8, 8, device=DEV)
    tr.step(x)
    real = tr._eager_step
    calls = {"n": 0}

    def flaky(*a, **k):
        calls["n"] += 1
        out = real(*a, **k)
        if calls["n"] == 1:     # inside the capture: the step body ran on the host, then capture "fails"
            raise RuntimeError("injected capture failure")
        return out

    monkeypatch.setattr(tr, "_eager_step", flaky)
    with pytest.warns(UserWarning, match="capture of the training step failed"):
        tr.step(x)
    tr.step(x)
    torch.cuda.synchronize()
    assert tr.cuda_graph is False
    assert tr.opt.step_count == int(tr.opt.step_dev) == 3
    tr.opt.close()


def test_flat_engine_matches_torch_optimizer(golden):
    """engine.LDMTrainer (flat buffers, wgrad accumulating into main_grad, fused clip+AdamW, bf16 shadow) must take
    the same optimisation trajectory as the plain autograd + torch.optim.AdamW + clip_grad_norm_ path (fp32)."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_small")
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    ma, _ = _build(g, torch.float32)
    mb, _ = _build(g, torch.float32)
    s = mig.DDPMScheduler(**kw)
    tr = LDMTrainer(ma, s, lr=1e-3, grad_clip_max_norm=1.0)
    opt = torch.optim.AdamW(mb.parameters(), lr=1e-3)
    gen = torch.Generator().manual_seed(3)
    for step in range(4):
        x0 = torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV)
        noise = torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV)
        t = torch.randint(0, 1000, (2,), generator=gen).to(DEV)
        la = tr.step(x0, noise=noise, timesteps=t)
        pred = mb(s.add_noise(x0, noise, t), t)
        lb = mig.ops.mse_loss(pred, noise)
        opt.zero_grad(set_to_none=True)
        lb.backward()
        gn = torch.nn.utils.clip_grad_norm_(mb.parameters(), 1.0)
        opt.step()
        assert abs(float(la) - float(lb)) < 1e-4 * abs(float(lb)) + 1e-6, (step, float(la), float(lb))
        assert rel_err(tr.opt.grad_norm(), gn) < 1e-3
    pa, pb = dict(ma.named_parameters()), dict(mb.named_parameters())
    worst = max(rel_err(pa[k], pb[k]) for k in pa)
    assert worst < 2e-4, worst
    for k in pa:   # never-used parameters are untouched, like torch skips grad=None
        if "proj_attn" in k:
            assert torch.equal(pa[k], pb[k])
    # the bf16 shadow is the round-to-nearest of the master copy, exactly
    k0 = "conv_in.conv.weight"
    assert torch.equal(pa[k0]._mig_shadow, pa[k0].detach().to(torch.bfloat16))
    assert torch.equal(tr.opt.shadow, tr.opt.master.to(torch.bfloat16))
    tr.opt.close()


def test_gradient_accumulation_matches_torch(golden):
    """config['grad_accumulate_step'] = 2 (train_ldm.py:173): two backward passes sum their gradients, clip + AdamW run
    on the sum; a trailing partial group is stepped by flush()."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_small")
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    ma, _ = _build(g, torch.float32)
    mb, _ = _build(g, torch.float32)
    s = mig.DDPMScheduler(**kw)
    tr = LDMTrainer(ma, s, lr=1e-3, grad_clip_max_norm=1.0, grad_accumulate_step=2)
    opt = torch.optim.AdamW(mb.parameters(), lr=1e-3)
    gen = torch.Generator().manual_seed(5)
    opt.zero_grad(set_to_none=True)
    for step in range(5):   # 2 full groups + 1 trailing micro-step
        x0 = torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV)
        noise = torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV)
        t = torch.randint(0, 1000, (2,), generator=gen).to(DEV)
        tr.step(x0, noise=noise, timesteps=t)
        mig.ops.mse_loss(mb(s.add_noise(x0, noise, t), t), noise).backward()
        if (step + 1) % 2 == 0 or step == 4:
            if step == 4:
                tr.flush()
            torch.nn.utils.clip_grad_norm_(mb.parameters(), 1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
    pa, pb = dict(ma.named_parameters()), dict(mb.named_parameters())
    worst = max(rel_err(pa[k], pb[k]) for k in pa)
    assert worst < 2e-4, worst
    tr.opt.close()


def test_optimizer_state_interchange_with_torch(golden):
    """ckpt['optimizer_state_dict'] interchange (train_ldm.py:472-477): the flat optimiser exports torch.optim.AdamW's
    state_dict layout; loading it into a real torch AdamW (and back into a fresh flat optimiser) continues the same
    trajectory."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_small")
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    s = mig.DDPMScheduler(**kw)
    ma, _ = _build(g, torch.float32)
    tr = LDMTrainer(ma, s, lr=1e-3, grad_clip_max_norm=1.0)
    gen = torch.Generator().manual_seed(11)

    def batch():
        return (torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV), torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV),
                torch.randint(0, 1000, (2,), generator=gen).to(DEV))

    for _ in range(2):
        tr.step(*batch())
    sd = tr.opt.torch_state_dict()
    # (1) resume in torch
    mb, _ = _build(g, torch.float32)
    mb.load_state_dict(ma.state_dict())
    opt = torch.optim.AdamW(mb.parameters(), lr=1e-3)
    opt.load_state_dict(sd)
    # (2) resume in a fresh flat optimiser
    mc, _ = _build(g, torch.float32)
    mc.load_state_dict(ma.state_dict())
    tr.opt.close()
    tr2 = LDMTrainer(mc, s, lr=5e-4, grad_clip_max_norm=1.0)
    tr2.opt.load_torch_state_dict(opt.state_dict())
    assert tr2.opt.step_count == 2 and abs(tr2.opt.lr - 1e-3) < 1e-12
    x0, noise, t = batch()
    tr2.step(x0, noise=noise, timesteps=t)
    opt.zero_grad(set_to_none=True)
    mig.ops.mse_loss(mb(s.add_noise(x0, noise, t), t), noise).backward()
    torch.nn.utils.clip_grad_norm_(mb.parameters(), 1.0)
    opt.step()
    pb, pc = dict(mb.named_parameters()), dict(mc.named_parameters())
    worst = max(rel_err(pc[k], pb[k]) for k in pb)
    assert worst < 2e-4, worst
    tr2.opt.close()


# graphed vs eager step on the same inputs (GroupNorm / split-K atomics reorder fp32 sums); worst on a B200:
GRAPH_LOSS_TOL = 2e-3    # 5.0e-4
GRAPH_NORM_TOL = 5e-3    # 1.8e-3
GRAPH_DRIFT_TOL = 0.2    # 4.2e-2; a replay reading a stale input, noise or shadow gives about 1


def test_cuda_graph_step_replays_correctly(golden):
    """The whole training step captured in a CUDA graph: step counter lives on the device, and every replay is the step
    an eager trainer takes from the same state with the same batch, noise and timesteps (per-step loss and gradient
    norm, and where the masters end up: a replay reading a stale input, noise or shadow drifts by a ratio near 1)."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import LDMTrainer
    g = golden("unet3d_small")
    m, _ = _build(g, torch.bfloat16)
    m_eager, _ = _build(g, torch.bfloat16)
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    tr = LDMTrainer(m, mig.DDPMScheduler(**kw), lr=1e-4, cuda_graph=True, graph_warmup_steps=2)
    tr_eager = LDMTrainer(m_eager, mig.DDPMScheduler(**kw), lr=1e-4)
    gen = torch.Generator().manual_seed(4)
    xs = [torch.randn(2, 3, 8, 8, 8, generator=gen).to(DEV) for _ in range(7)]
    p0 = tr.opt.master.clone()
    rows, noises, drift = graph_vs_eager(tr, tr_eager, xs)
    tr_eager.opt.close()
    assert tr._graph is not None, "capture did not happen"
    assert int(tr.opt.step_dev) == 7 and tr.opt.step_count == 7
    assert not any(torch.equal(noises[i], noises[i + 1]) for i in range(2, 6)), "replays drew the same noise"
    for la, lb, ga, gb in rows:
        assert abs(la - lb) < GRAPH_LOSS_TOL * abs(lb) and abs(ga - gb) < GRAPH_NORM_TOL * gb, rows
    assert drift < GRAPH_DRIFT_TOL, drift
    x = xs[-1]
    snap = tr.opt.master.clone()
    tr.step(x)
    assert not torch.equal(snap, tr.opt.master) and not torch.equal(p0, snap)
    # a new input shape re-captures instead of replaying a stale graph
    x2 = torch.randn(1, 3, 8, 8, 8, device=DEV)
    for _ in range(4):
        l2 = float(tr.step(x2))
    assert l2 == l2 and tr._graph_key[0] == (1, 3, 8, 8, 8)
    tr.opt.close()


def test_ae_trainer_and_sampling_sharder(golden):
    """AETrainer (L1 + kl_weight*KL generator step) lowers the loss, and its first fp32 step gives the oracle's loss and
    gradient norm; sample_volumes is seed-deterministic per volume
    (what the N-rank sharder relies on: volume v always uses seed base+v wherever it runs)."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import AETrainer, sample_volumes
    g = golden("ae3d_small")
    m, _ = _build(g, torch.bfloat16)
    tr = AETrainer(m, lr=1e-3, kl_weight=1e-7)
    x = g["inputs"]["x"].to(DEV)
    losses = [float(tr.step(x)) for _ in range(12)]
    assert losses[-1] < losses[0], losses
    tr.opt.close()
    # the first step in fp32 against the oracle on the CPU: same weights, images and sampling noise
    from oracle import torch_oracle as O
    m32, params = _build(g, torch.float32)
    tr32 = AETrainer(m32, lr=1e-3, kl_weight=1e-7)
    eps = g["inputs"]["eps"]
    loss = float(tr32.step(x, eps=eps.to(DEV)))
    ref = {k: v.float().clone().requires_grad_(True) for k, v in params.items()}
    recon, z_mu, z_sigma = O.ae_forward(ref, g["cfg"], g["inputs"]["x"].float(), eps)
    ref_loss = F.l1_loss(recon, g["inputs"]["x"].float()) + 1e-7 * O.kl_loss(z_mu, z_sigma)
    ref_loss.backward()
    ref_norm = sum(float(p.grad.double().pow(2).sum()) for p in ref.values() if p.grad is not None) ** 0.5
    assert abs(loss - float(ref_loss)) <= FP32_TOL * float(ref_loss), (loss, float(ref_loss))
    assert abs(float(tr32.opt.grad_norm()) - ref_norm) <= FP32_TOL * ref_norm, (float(tr32.opt.grad_norm()), ref_norm)
    tr32.opt.close()
    gu = golden("unet3d_aniso")
    u, _ = _build(gu, torch.float32)
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    a = sample_volumes(u, mig.DDPMScheduler(**kw), (1, 12, 12, 6), 3, base_seed=42, num_inference_steps=4, noise_mode="host")
    b = sample_volumes(u, mig.DDPMScheduler(**kw), (1, 12, 12, 6), 3, base_seed=42, num_inference_steps=4, noise_mode="host")
    # same seeds -> same volumes (up to the rounding of atomic reduction order inside GroupNorm)
    assert sorted(a) == [0, 1, 2] and all(rel_err(a[k], b[k]) < 1e-4 for k in a)
    assert not torch.equal(a[0], a[1]) and all(torch.isfinite(v).all() for v in a.values())


def test_ldm_width_unet_with_folded_upsample_convs_matches_reference_golden(golden):
    """BASELINE config 3 at full width with BOTH Upsample convolutions folded (ops.set_upconv('always'); in 'auto' mode
    the 8^3 golden is too small for the fold to pay): same bf16 bar as the unfolded model."""
    from medical_image_generation_b200 import ops, _lib
    from oracle.golden_util import sketch
    g = golden("unet3d_ldm_width")
    m, _ = _build(g, torch.bfloat16)
    inp = g["inputs"]
    x = inp["x"].to(DEV).requires_grad_(True)
    ops.set_upconv("always")
    try:
        before = _lib.launch_count
        y = m(x, inp["timesteps"].to(DEV))
        (y * inp["probe"].to(DEV)).sum().backward()
        launches = _lib.launch_count - before
    finally:
        ops.set_upconv("auto")
    assert rel_err(y, g["out"]) < BF16_TOL
    assert rel_err(x.grad, g["grad_x"]) < 2.5 * BF16_TOL
    named = dict(m.named_parameters())
    for k in ("up_blocks.0.upsampler.conv.conv.weight", "up_blocks.1.upsampler.conv.conv.weight",
              "up_blocks.0.upsampler.conv.conv.bias", "up_blocks.1.upsampler.conv.conv.bias"):
        assert rel_err(sketch(named[k].grad), g["grad_sketch"][k], floor=0.1) < 8e-2, k
    # and the fold really ran: the unfolded model needs fewer ABI calls (2 x (8 class convs + 8 class wgrads + glue))
    before = _lib.launch_count
    m.zero_grad(set_to_none=True)
    y2 = m(x, inp["timesteps"].to(DEV))
    (y2 * inp["probe"].to(DEV)).sum().backward()
    assert launches > (_lib.launch_count - before) + 20
