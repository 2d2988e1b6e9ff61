"""The autoencoder training step (BASELINE config 2) and the end-to-end LDM step (config 5), kernel call by kernel call.

Config 2 trains the AutoencoderKL (32/64/128 channels, GroupNorm 16, latent 3) on 2 x 1 x 96^3 with L1 + 1e-7 KL
(tools/ae_bench.py). Config 5 encodes 2 x 2 x 160 x 160 x 128 volumes with a frozen AutoencoderKL and trains the
LDM-default U-Net on the 2 x 3 x 40 x 40 x 32 latents (tools/ldm_e2e_bench.py). These run kernels and branches the
benchmarked configs 3 and 4 never reach: the 32-channel halo kernels at 2 x 32 x 96^3 and 2 x 32 x 160 x 160 x 128, the
strided 32-channel Downsample (dgrad as stride-residue classes), the thin CUDA-core conv_in / out conv and their
fp32-atomic wgrad over 1.77 M voxels, GroupNorm with 2 channels per group over millions of elements, the upsample fold at
64 / 128 channels, unfused attention at L = 6400 (three-pass softmax) and at L = 800, d = 768 on a non-cubic pyramid,
and the VAE tail (sigma, reparameterisation, L1, KL). Every distinct ops call of one real step is recorded
and checked against a full-precision reference with the harness of tests/callcheck.py, and the whole step is compared
with the fp32 oracle.
"""
import pytest
import torch
import torch.nn.functional as F

from callcheck import _check_backward, _check_forward, _kl_ref, _peak, _Recorder, _Report
from util import local_errors, rel_err

DEV = "cuda"
AE2_SIZE = (96, 96, 96)
VOL5 = (160, 160, 128)


@pytest.fixture
def no_tf32():
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def _conv_kinds(rec):
    """Which conv branches a recorded conv call exercises, from the shape rules of the dispatch in csrc/conv.cu,
    conv_halo.cu and conv_thin.cu (bf16, `auto` engine)."""
    x, w = rec["x"], rec["w"]
    cin, cout, k, s = x.shape[1], w.shape[0], tuple(w.shape[2:]), rec["stride"]
    out = rec["outs"][0]
    vox = out.shape[0] * out[0, 0].numel()
    kinds = set()
    if x.dtype != torch.bfloat16:
        return kinds
    if any(v == 2 for v in s):
        kinds.add("stride2")
    if cin == 32 and all(v == 1 for v in s) and max(k) <= 3 and cout <= 64 and vox >= 32768:
        kinds.add("halo")            # conv_halo_kernel forward; wgrad_halo_kernel when cout <= 32
    if cin <= 2 and cout == 32:
        kinds.add("thin_in")         # thin_conv_kernel forward, thin_wgrad_kernel (fp32 atomics)
    if cout <= 2 and cin == 32:
        kinds.add("thin_out")
    return kinds


def _launched(monkeypatch, ops, fn):
    """The C entry points `fn()` launches, in order."""
    seen = []
    real = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.append(name), real(name, *a))[1])
    try:
        fn()
    finally:
        monkeypatch.setattr(ops, "call", real)
    return seen


# ------------------------------------------------------------------------------------------------------------------
# BASELINE config 2: AutoencoderKL training step at 2 x 1 x 96^3
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ae_trainer():
    """Model and trainer as tools/ae_bench.py builds them, trained through AETrainer."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import AETrainer
    torch.manual_seed(0)
    kw = planner.autoencoder_kwargs(list(AE2_SIZE), in_channels=1, latent_channels=3, levels=2)
    ae = mig.AutoencoderKL(**kw, compute_dtype=torch.bfloat16).to(DEV).train()
    tr = AETrainer(ae, lr=5e-5, kl_weight=1e-7, grad_clip_max_norm=1.0)
    yield kw, ae, tr
    tr.opt.close()
    del ae, tr
    torch.cuda.empty_cache()


def _ae_batch(seed, batch=2):
    """Images in [0, 1) like the tool, and the sampling noise of the 4x smaller latent."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((batch, 1, *AE2_SIZE), generator=g)
    eps = torch.randn((batch, 3, *(s // 4 for s in AE2_SIZE)), generator=g)
    return x.to(DEV), eps.to(DEV)


# C entry points one eager AETrainer step launches through ops (config 2, defaults; recorded on a B200): the fold at both
# Upsample convs (mig_upconv_*, mig_class_interleave), the GroupNorm statistics in the conv epilogue, the VAE tail
# (mig_vae_sample_*, mig_addcmul, mig_mul), L1 (mig_mse_* in L1 mode) and KL, and the fp32 images cast to bf16 on entry
# (mig_cast). A routing change fails here: make sure the new path is among the calls checked, then update the list.
AE_STEP_CALLS = sorted([
    "mig_addcmul", "mig_cast", "mig_class_interleave", "mig_colsum", "mig_conv_dgrad", "mig_conv_fwd",
    "mig_conv_fwd_stats", "mig_conv_wgrad", "mig_groupnorm_apply", "mig_groupnorm_bwd", "mig_groupnorm_fwd",
    "mig_kl_bwd", "mig_kl_fwd", "mig_mse_bwd", "mig_mse_fwd", "mig_mul", "mig_nchw_to_nhwc", "mig_nhwc_to_nchw",
    "mig_upconv_fold_filter", "mig_upconv_fwd", "mig_upconv_unfold_wgrad", "mig_vae_sample_bwd", "mig_vae_sample_fwd",
])


@pytest.mark.gpu
def test_ae_training_step_calls_at_config2_shape(ae_trainer, monkeypatch, no_tf32):
    """Every distinct ops call of one eager AETrainer step at 2 x 1 x 96^3: forward in place, backward standalone on the
    recorded output gradient, the epilogue GroupNorm sums, the bf16 shadow and the C entry points the step used."""
    from medical_image_generation_b200 import ops
    _, _, tr = ae_trainer
    torch.cuda.reset_peak_memory_stats()
    rep = _Report("AE training step, BASELINE config 2")
    recorder = _Recorder(monkeypatch, ops)
    x, eps = _ae_batch(100)
    tr.step(x, eps=eps)
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(AE_STEP_CALLS), f"entry points: {sorted(recorder.names)} (expected "
                f"{AE_STEP_CALLS}; missing {sorted(set(AE_STEP_CALLS) - recorder.names)}, new "
                f"{sorted(recorder.names - set(AE_STEP_CALLS))})")
    rep.require(torch.equal(tr.opt.shadow, tr.opt.master.to(torch.bfloat16)), "bf16 shadow != bf16(master)")
    ops_seen, kinds = {}, set()
    for rec in recorder.calls.values():
        ops_seen[rec["op"]] = ops_seen.get(rec["op"], 0) + 1
        if rec["op"] == "conv":
            kinds |= _conv_kinds(rec)
        _check_forward(rep, rec)
        _check_backward(rep, recorder.real, rec)
    rep.require({"conv", "upconv", "gn", "sigma", "reparam", "l1", "kl"} <= set(ops_seen), f"ops recorded: {ops_seen}")
    rep.require({"halo", "thin_in", "thin_out", "stride2"} <= kinds, f"conv branches checked: {sorted(kinds)}")
    rep.require(any(r["op"] == "conv" and r["sums"] is not None for r in recorder.calls.values()),
                "no conv delivered epilogue GroupNorm statistics")
    # both Upsample convs fold: 128 channels at 24^3 -> 48^3 and 64 channels at 48^3 -> 96^3
    folds = {tuple(r["x"].shape[1:]): r["sig"][-1] for r in recorder.calls.values() if r["op"] == "upconv"}
    rep.require(folds == {(128, 24, 24, 24): True, (64, 48, 48, 48): True}, f"upsample fold per input: {folds}")
    print(f"distinct calls checked: {ops_seen}; conv branches {sorted(kinds)}; folds {folds}")
    _peak(rep, "AE training calls")
    rep.finish()


# whole AE step against the oracle: the config-3 bars where the worst value on a B200 stays under half of them, else
# about twice the worst. Every per-call check of the step sits at bf16 rounding (test above); the whole step compounds
# it through 21 convolutions into a one-channel output, and the L1 gradient is a sign that bf16 rounding flips wherever
# recon is close to the image, which reaches every encoder gradient through the decoder.
AE_OUT_BAR = 3e-2       # recon / z_mu / z_sigma rel_err; worst 1.56e-2 (recon)
AE_ROW_BAR = 0.25       # recon per voxel; worst 0.12
AE_GRAD_BAR = 0.15      # worst 8.3e-2 (encoder.blocks.2.norm1.bias)
AE_LOSS_BAR = 5e-3      # worst 4.9e-4
AE_NORM_BAR = 5e-3      # worst 1.4e-3


@pytest.mark.gpu
def test_ae_training_step_matches_oracle_at_config2_shape(ae_trainer, no_tf32):
    """One production AETrainer step and the fp32 oracle (ae_forward, L1 + 1e-7 KL) on the same weights, images and
    sampling noise: loss, recon, z_mu, z_sigma, every parameter's gradient and the gradient norm."""
    from oracle import torch_oracle as O
    kw, ae, tr = ae_trainer
    torch.cuda.reset_peak_memory_stats()
    params = {k: v.detach().float().contiguous().clone().requires_grad_(True) for k, v in ae.state_dict().items()}
    x, eps = _ae_batch(200)
    got = {}
    encode, decode = ae.encode, ae.decode

    def enc(images):
        z_mu, z_sigma = encode(images)
        got.update(z_mu=z_mu.detach().clone(), z_sigma=z_sigma.detach().clone())
        return z_mu, z_sigma

    def dec(z):
        recon = decode(z)
        got["recon"] = recon.detach().clone()
        return recon

    ae.encode, ae.decode = enc, dec
    try:
        loss = float(tr.step(x, eps=eps).detach())
    finally:
        del ae.encode, ae.decode
    recon, z_mu, z_sigma = O.ae_forward(params, kw, x, eps)
    ref_loss = F.l1_loss(recon, x) + 1e-7 * O.kl_loss(z_mu, z_sigma)
    ref_loss.backward()
    rep = _Report("AE training step vs oracle, BASELINE config 2")
    rep.value("loss", abs(loss - float(ref_loss)) / float(ref_loss), AE_LOSS_BAR, "loss")
    for name, ref in (("recon", recon), ("z_mu", z_mu), ("z_sigma", z_sigma)):
        rep.value("output", rel_err(got[name], ref), AE_OUT_BAR, f"{name} (rel_err)")
    e = local_errors(got["recon"], recon)
    rep.value("recon voxel", e["row"], AE_ROW_BAR, f"recon per voxel, worst at (n, *spatial) {e['row_at']}")
    sq = 0.0
    for k, p in ae.named_parameters():
        ref = params[k].grad
        rep.require(ref is not None, f"oracle gives no gradient for {k}")
        if ref is None:
            continue
        sq += float(ref.double().pow(2).sum())
        rep.value("param grad", rel_err(p.main_grad, ref, floor=1e-12), AE_GRAD_BAR, k)
    rep.value("grad_norm", abs(float(tr.opt.grad_norm()) - sq ** 0.5) / sq ** 0.5, AE_NORM_BAR, "opt.grad_norm()")
    _peak(rep, "AE oracle step")
    rep.finish()


# ------------------------------------------------------------------------------------------------------------------
# BASELINE config 5: frozen AE encode at 2 x 2 x 160 x 160 x 128, U-Net step on 2 x 3 x 40 x 40 x 32 latents
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ae5():
    """The frozen autoencoder of tools/ldm_e2e_bench.py."""
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    torch.manual_seed(0)
    kw = planner.autoencoder_kwargs(VOL5, in_channels=2, latent_channels=3)
    ae = mig.AutoencoderKL(**kw, compute_dtype=torch.bfloat16).to(DEV).eval().requires_grad_(False)
    yield kw, ae
    del ae
    torch.cuda.empty_cache()


def _volumes(seed, batch=2):
    return torch.rand((batch, 2, *VOL5), generator=torch.Generator().manual_seed(seed)).to(DEV)


# ... of the config-5 encode under no_grad: the filters cast to bf16 once (mig_cast: the frozen AE has no optimiser
# shadow), the GroupNorm statistics in the conv epilogue, sigma only (no reparameterisation in encode).
ENCODE_CALLS = sorted([
    "mig_cast", "mig_conv_fwd", "mig_conv_fwd_stats", "mig_groupnorm_apply", "mig_groupnorm_fwd", "mig_nchw_to_nhwc",
    "mig_nhwc_to_nchw", "mig_vae_sample_fwd",
])
ENCODE_BAR = 2e-2        # z_mu / z_sigma against the fp32 oracle; worst 1.02e-2 (z_mu)


@pytest.mark.gpu
def test_ae_encode_calls_at_config5_shape(ae5, monkeypatch, no_tf32):
    """Every distinct ops call of the frozen AE's encode at 2 x 2 x 160 x 160 x 128 (halo kernels over 3.3 M voxels per
    sample, GroupNorm over 6.55 M elements per group), and z_mu / z_sigma against the fp32 oracle."""
    from medical_image_generation_b200 import ops
    from oracle import torch_oracle as O
    kw, ae = ae5
    torch.cuda.reset_peak_memory_stats()
    x = _volumes(300)
    rep = _Report("AE encode, BASELINE config 5")
    recorder = _Recorder(monkeypatch, ops)
    with torch.no_grad():
        z_mu, z_sigma = ae.encode(x)
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(ENCODE_CALLS), f"entry points: {sorted(recorder.names)} (expected {ENCODE_CALLS})")
    kinds = set()
    for rec in recorder.calls.values():
        if rec["op"] == "conv":
            kinds |= _conv_kinds(rec)
        _check_forward(rep, rec)
    rep.require({"halo", "thin_in", "stride2"} <= kinds, f"conv branches checked: {sorted(kinds)}")
    recorder.calls.clear()
    params = {k: v.detach().float() for k, v in ae.state_dict().items()}
    with torch.no_grad():
        mu_r, sigma_r = O.ae_encode(params, kw, x)
    rep.value("encode", rel_err(z_mu, mu_r), ENCODE_BAR, "z_mu (rel_err)")
    rep.value("encode", rel_err(z_sigma, sigma_r), ENCODE_BAR, "z_sigma (rel_err)")
    _peak(rep, "encode calls")
    rep.finish()


@pytest.fixture(scope="module")
def ldm5(ae5):
    """The U-Net and trainer of tools/ldm_e2e_bench.py, and one batch of latents the frozen AE encoded, scaled to unit
    standard deviation (train_ldm.py:110-112)."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import LDMTrainer
    kw, ae = ae5
    lat = planner.compute_output_size(VOL5, kw["downsample_parameters"])
    cfg = planner.ddpm_kwargs(lat, latent_channels=3)
    torch.manual_seed(1)
    unet = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**cfg, compute_dtype=torch.bfloat16)).to(DEV).train()
    tr = LDMTrainer(unet, mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS), lr=2e-5, grad_clip_max_norm=1.0)
    with torch.no_grad():
        z = ae.encode_stage_2_inputs(_volumes(400))
        z = z * (1.0 / float(z.float().std()))
    yield cfg, unet, tr, z
    tr.opt.close()
    del unet, tr, z
    torch.cuda.empty_cache()


def _ldm_batch(z, seed):
    g = torch.Generator().manual_seed(seed)
    noise = torch.randn(z.shape, generator=g)
    t = torch.randint(0, 1000, (z.shape[0],), generator=g)
    return noise.to(DEV), t.to(DEV)


# ... of one eager config-5 U-Net step: the fold at 20 x 20 x 16 -> 40 x 40 x 32 (512 channels), the unfolded nearest
# upsample + conv at 10 x 10 x 8 -> 20 x 20 x 16 (too few tiles to fold), and the unfused attention chain at both
# attention levels (no flash kernel: see UNFUSED below).
LDM5_STEP_CALLS = sorted([
    "mig_add", "mig_class_interleave", "mig_colsum", "mig_concat_channels", "mig_conv_dgrad", "mig_conv_fwd",
    "mig_conv_fwd_stats", "mig_conv_wgrad", "mig_gemm_strided", "mig_groupnorm_apply", "mig_groupnorm_bwd",
    "mig_groupnorm_fwd", "mig_mse_bwd", "mig_mse_fwd", "mig_nchw_to_nhwc", "mig_nhwc_to_nchw", "mig_silu_bwd",
    "mig_silu_fwd", "mig_softmax_bwd_narrow", "mig_softmax_fwd", "mig_split_channels", "mig_temb_proj_all_bwd",
    "mig_temb_proj_all_fwd", "mig_timestep_embedding", "mig_upconv_fold_filter", "mig_upconv_fwd",
    "mig_upconv_unfold_wgrad", "mig_upsample_nearest_bwd", "mig_upsample_nearest_fwd",
])
# Attention routing in training (ops.set_flash_attention, `auto`): single heads of d = 512 / 768 take the unfused GEMM +
# softmax chain for L > 256 while its L x L buffers stay under 2 GiB, because the fused kernels must slice the head's
# accumulators and recompute Q K^T per slice. So both levels of config 5 run unfused: L = 6400 (three-pass softmax,
# rows > 2048) and L = 800; the fused kernels only take the 6^3 block (L = 216) of config 3.
UNFUSED = {"mig_gemm_strided", "mig_softmax_fwd", "mig_softmax_bwd_narrow"}
FLASH = {"mig_flash_attention_fwd_ld", "mig_flash_attention_bwd"}


@pytest.mark.gpu
def test_ldm_step_calls_at_config5_shape(ldm5, monkeypatch, no_tf32):
    """Every distinct ops call of one eager LDMTrainer step on 2 x 3 x 40 x 40 x 32 latents (pyramid 40 x 40 x 32,
    20 x 20 x 16, 10 x 10 x 8): forward in place, backward standalone; the unfused attention chain at L = 6400, d = 512
    and at L = 800, d = 768."""
    from medical_image_generation_b200 import ops
    _, _, tr, z = ldm5
    torch.cuda.reset_peak_memory_stats()
    rep = _Report("LDM step, BASELINE config 5")
    recorder = _Recorder(monkeypatch, ops)
    noise, t = _ldm_batch(z, 500)
    tr._eager_step(z, noise, t)
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(LDM5_STEP_CALLS), f"entry points: {sorted(recorder.names)} (expected "
                f"{LDM5_STEP_CALLS}; missing {sorted(set(LDM5_STEP_CALLS) - recorder.names)}, new "
                f"{sorted(recorder.names - set(LDM5_STEP_CALLS))})")
    rep.require(torch.equal(tr.opt.shadow, tr.opt.master.to(torch.bfloat16)), "bf16 shadow != bf16(master)")
    ops_seen, routes = {}, {}
    for rec in recorder.calls.values():
        ops_seen[rec["op"]] = ops_seen.get(rec["op"], 0) + 1
        _check_forward(rep, rec)
        if rec["op"] == "sdpa_qkv":
            L, d = rec["qkv"].shape[1], rec["qkv"].shape[2] // 3
            routes[(L, d)] = set(_launched(monkeypatch, ops, lambda: _check_backward(rep, recorder.real, rec)))
        else:
            _check_backward(rep, recorder.real, rec)
    rep.require({"conv", "upconv", "gn", "linear", "temb", "sdpa_qkv"} <= set(ops_seen), f"ops recorded: {ops_seen}")
    rep.require(sorted(routes) == [(800, 768), (6400, 512)], f"attention shapes {sorted(routes)}")
    rep.require(UNFUSED <= routes.get((6400, 512), set()) and not FLASH & routes.get((6400, 512), set()),
                f"L = 6400 route {sorted(routes.get((6400, 512), ()))}")
    rep.require(UNFUSED <= routes.get((800, 768), set()) and not FLASH & routes.get((800, 768), set()),
                f"L = 800 route {sorted(routes.get((800, 768), ()))}")
    print(f"distinct calls checked: {ops_seen}")
    _peak(rep, "LDM step calls")
    rep.finish()


# whole U-Net step against the oracle (the config-3 bars; worst value on a B200 beside each)
LDM_OUT_BAR = 1e-2      # worst 4.0e-3
LDM_GRAD_BAR = 6e-2     # worst 3.6e-2 (up_blocks.0.attentions.2.to_k.weight)
LDM_LOSS_BAR = 5e-3     # worst 4.4e-4
LDM_NORM_BAR = 5e-3     # worst 1.5e-4


@pytest.mark.gpu
def test_ldm_step_matches_oracle_at_config5_shape(ldm5, monkeypatch, no_tf32):
    """One production U-Net step on the encoded latents and the fp32 oracle on the same weights, noisy input and
    timesteps: loss, U-Net output, every parameter's full gradient and the global gradient norm."""
    from oracle import torch_oracle as O
    cfg, unet, tr, z = ldm5
    torch.cuda.reset_peak_memory_stats()
    params = {k: v.detach().float().contiguous().clone().requires_grad_(True) for k, v in unet.state_dict().items()}
    noise, t = _ldm_batch(z, 600)
    got = {}
    hook = unet.register_forward_hook(lambda m, a, kw, out: got.update(x=kw["x"].detach().clone(), out=out.detach().clone()),
                                      with_kwargs=True)
    try:
        loss = float(tr._eager_step(z, noise, t).detach())
    finally:
        hook.remove()
    real_temb = O.timestep_embedding    # (builds its frequency table on the CPU)
    monkeypatch.setattr(O, "timestep_embedding", lambda ts, dim, max_period=10000: real_temb(ts.cpu(), dim, max_period).to(ts.device))
    pred = O.unet_forward(params, cfg, got["x"], t)
    ref_loss = F.mse_loss(pred, noise)
    ref_loss.backward()
    rep = _Report("LDM step vs oracle, BASELINE config 5")
    rep.value("loss", abs(loss - float(ref_loss)) / float(ref_loss), LDM_LOSS_BAR, "loss")
    rep.value("output", rel_err(got["out"], pred), LDM_OUT_BAR, "U-Net output (rel_err)")
    e = local_errors(got["out"], pred)
    print(f"U-Net output: per-voxel {e['row']:.3e} at {e['row_at']}, per-channel {e['col']:.3e}")
    sq = 0.0
    for k, p in unet.named_parameters():
        ref = params[k].grad
        if ref is None:
            rep.require("proj_attn" in k, f"oracle gives no gradient for {k}")
            continue
        sq += float(ref.double().pow(2).sum())
        if k.endswith("to_k.bias"):
            continue    # exactly zero mathematically (softmax is shift invariant): noise on both sides
        rep.value("param grad", rel_err(p.main_grad, ref, floor=1e-12), LDM_GRAD_BAR, k)
    rep.value("grad_norm", abs(float(tr.opt.grad_norm()) - sq ** 0.5) / sq ** 0.5, LDM_NORM_BAR, "opt.grad_norm()")
    _peak(rep, "LDM oracle step")
    rep.finish()


# ------------------------------------------------------------------------------------------------------------------
# edges of the VAE tail
# ------------------------------------------------------------------------------------------------------------------
# log-variances at the clamp bounds, just inside, just outside and far outside (all exact in bf16)
_LOGVARS = [-1e4, -30.25, -30.0, -29.75, -1.0, 0.0, 1.0, 19.875, 20.0, 20.125, 1e4]
_EDGE_TOL = {torch.float32: 1e-6, torch.bfloat16: 2 ** -8}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_vae_sigma_at_clamp_bounds(dtype):
    """sigma = exp(clamp(lv, -30, 20) / 2) and its gradient at and around the bounds. torch.clamp passes the gradient
    when lv equals a bound, and so does the kernel (`lv >= -30 && lv <= 20`); outside, both give exactly zero."""
    from medical_image_generation_b200 import ops
    lv = torch.tensor(_LOGVARS).to(dtype).reshape(1, 1, -1)
    probe = torch.linspace(0.5, 1.5, lv.numel()).to(dtype).reshape(lv.shape)
    ld = lv.to(DEV).requires_grad_(True)
    sigma = ops.vae_sigma(ld)
    sigma.backward(probe.to(DEV))
    lr = lv.float().requires_grad_(True)
    want = torch.exp(torch.clamp(lr, -30.0, 20.0) / 2)
    want.backward(probe.float())
    tol = _EDGE_TOL[dtype]
    assert sigma.dtype == dtype
    got, ref = sigma.float().cpu(), want.detach()
    assert ((got - ref).abs() <= tol * ref.abs()).all(), (got, ref)
    dg, dr = ld.grad.float().cpu(), lr.grad
    assert torch.equal(dg == 0, dr == 0), (dg, dr)          # the same elements pass the gradient
    assert ((dg - dr).abs() <= 2 * tol * dr.abs()).all(), (dg, dr)
    assert (dr.flatten()[[2, 8]] != 0).all() and (dr.flatten()[[0, 1, 9, 10]] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_l1_backward_where_prediction_equals_target(dtype):
    """d|a - b| / da is 0 where a == b exactly (torch's sign(0)); elsewhere +-1/n."""
    from medical_image_generation_b200 import ops
    g = torch.Generator().manual_seed(11)
    a = torch.randn(2, 1, 16, 16, 16, generator=g).to(dtype)
    b = torch.randn(a.shape, generator=g).to(dtype)
    b[:, :, :8] = a[:, :, :8]
    ad = a.to(DEV).requires_grad_(True)
    loss = ops.l1_loss(ad, b.to(DEV))
    loss.backward()
    ar = a.double().requires_grad_(True)
    want = F.l1_loss(ar, b.double())
    want.backward()
    assert abs(float(loss) - float(want)) <= 1e-6 * float(want)
    assert (ad.grad[:, :, :8] == 0).all()
    assert torch.equal(ad.grad.float().cpu(), ar.grad.to(dtype).float())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_kl_loss_at_tiny_sigma(dtype):
    """KL with sigma = exp(-15) (the lower clamp), where the backward's 1/sigma is 3.3e6: loss against fp64, gradients
    against fp32 autograd, element by element."""
    from medical_image_generation_b200 import ops
    g = torch.Generator().manual_seed(12)
    mu = torch.randn(2, 3, 6, 6, 6, generator=g).to(dtype)
    sigma = torch.exp(torch.randn(mu.shape, generator=g))
    sigma.view(-1)[::7] = torch.exp(torch.tensor(-15.0))
    sigma = sigma.to(dtype)
    md, sd = mu.to(DEV).requires_grad_(True), sigma.to(DEV).requires_grad_(True)
    kl = ops.kl_loss(md, sd)
    kl.backward(torch.tensor(0.5, device=DEV))
    want = _kl_ref(mu.double(), sigma.double())
    assert abs(float(kl) - float(want)) <= 1e-5 * abs(float(want))
    mr, sr = mu.float().requires_grad_(True), sigma.float().requires_grad_(True)
    (0.5 * _kl_ref(mr, sr)).backward()
    # d/dmu = mu g / B; d/dsigma = (sigma - 1/sigma) g / B, which cancels near sigma = 1: bound by its two terms
    tol, s = _EDGE_TOL[dtype], sr.detach()
    for name, got, ref, scale in (("dmu", md.grad, mr.grad, mr.grad.abs()),
                                  ("dsigma", sd.grad, sr.grad, (s + 1 / s) * 0.5 / mu.shape[0])):
        err = (got.float().cpu() - ref).abs()
        assert (err <= 2 * tol * scale).all(), (name, float((err / scale).max()))
    assert float(sr.grad.abs().max()) > 0.9 / 3.06e-7 * 0.5 / mu.shape[0]    # the 1/sigma term at sigma = exp(-15)
