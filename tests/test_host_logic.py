"""CPU-only: C-ABI library loads and exports every declared symbol; module constructors, state_dict layout and
error behaviour mirror the reference; scheduler integer logic is bit-exact against the oracle restatement."""
import ctypes
import os

import numpy as np
import pytest
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import _lib
from oracle import ddpm_oracle, torch_oracle as O
from oracle.golden_util import CASES, golden_params


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "build the extension first: python -m medical_image_generation_b200.build"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _lib.declared_symbols()
    assert len(declared) >= 40
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/medimgen_b200.h but not exported"
    assert set(declared) == set(_lib._SIGNATURES), "ctypes signature table out of sync with the header"
    assert _lib.load().mig_abi_version() == 4


def test_struct_layouts_match_header():
    assert ctypes.sizeof(_lib.ConvGeom) == 4 * (1 + 3 + 3 + 2 + 9)
    assert ctypes.sizeof(_lib.GemmDesc) == 4 * 5 + 4 + 8 * 12 + 8  # 5 ints (+pad), 12 int64, float+int


@pytest.mark.parametrize("name", list(CASES))
def test_state_dict_layout_matches_reference(golden, name):
    g = golden(name)
    cls = mig.DiffusionModelUNet if g["kind"] == "unet" else mig.AutoencoderKL
    m = cls(**g["cfg"])
    sd = m.state_dict()
    assert list(sd.keys()) == list(g["shapes"].keys())          # same keys, same order
    for k, shape in g["shapes"].items():
        assert tuple(sd[k].shape) == tuple(shape), k
    # parameter registration order == reference (optimizer_state_dict indices of reference checkpoints)
    assert [n for n, _ in m.named_parameters()] == list(g["shapes"].keys())
    # loading reference-layout tensors (plain contiguous) keeps values and the kernel-friendly filter layout
    params = golden_params(g["shapes"], g["seed"])
    m.load_state_dict(params)
    for k, v in m.state_dict().items():
        assert torch.equal(v, params[k]), k
    for p in m.parameters():
        if p.ndim in (4, 5):
            fmt = torch.channels_last if p.ndim == 4 else torch.channels_last_3d
            assert p.is_contiguous(memory_format=fmt)
    # save / load round trip through torch.save like train_ldm.py:472-477
    import io
    buf = io.BytesIO()
    torch.save({"network_state_dict": m.state_dict()}, buf)
    buf.seek(0)
    m2 = cls(**g["cfg"])
    m2.load_state_dict(torch.load(buf)["network_state_dict"])
    for k, v in m2.state_dict().items():
        assert torch.equal(v, params[k])


def test_zero_init_and_unused_proj_attn():
    m = mig.DiffusionModelUNet(**CASES["unet3d_small"]["cfg"])
    sd = m.state_dict()
    assert float(sd["out.2.conv.weight"].abs().max()) == 0.0
    assert float(sd["down_blocks.0.resnets.0.conv2.conv.weight"].abs().max()) == 0.0
    assert float(sd["down_blocks.0.resnets.0.conv1.conv.weight"].abs().max()) > 0.0
    assert "middle_block.attention.proj_attn.weight" in sd


def test_constructor_errors_mirror_reference():
    U, A = mig.DiffusionModelUNet, mig.AutoencoderKL
    ok = CASES["unet3d_small"]["cfg"]
    with pytest.raises(IndexError):   # 3 default strides for 4 default levels (unet:1745-1763 with :1867)
        U(spatial_dims=3, in_channels=1, out_channels=1)
    with pytest.raises(IndexError):   # ae:664-667 with ae:413
        A(spatial_dims=3)
    with pytest.raises(ValueError, match="cross_attention_dim"):
        U(**{**ok, "with_conditioning": True})
    with pytest.raises(ValueError, match="with_conditioning=True"):
        U(**{**ok, "cross_attention_dim": 8})
    with pytest.raises(ValueError, match="Dropout"):
        U(**{**ok, "dropout_cattn": 1.5})
    with pytest.raises(ValueError, match="multiple of norm_num_groups"):
        U(**{**ok, "num_channels": [30, 64, 96]})
    with pytest.raises(ValueError, match="same size of attention_levels"):
        U(**{**ok, "attention_levels": [False, True]})
    with pytest.raises(ValueError, match="num_head_channels"):
        U(**{**ok, "num_head_channels": [0, 64]})
    with pytest.raises(ValueError, match="num_res_blocks"):
        U(**{**ok, "num_res_blocks": [2, 2]})
    with pytest.raises(ZeroDivisionError):  # middle block always uses num_head_channels[-1] (unet:1875-1888)
        U(**{**ok, "attention_levels": [False, False, False], "num_head_channels": [0, 0, 0]})
    aok = CASES["ae3d_small"]["cfg"]
    with pytest.raises(ValueError, match="multiple of norm_num_groups"):
        A(**{**aok, "num_channels": [16, 30, 64]})
    with pytest.raises(ValueError, match="same size of attention_levels"):
        A(**{**aok, "attention_levels": [False]})


def test_no_cpu_fallback():
    m = mig.DiffusionModelUNet(**CASES["unet2d_small"]["cfg"])
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(1, 1, 16, 16), torch.tensor([3]))
    s = mig.DDPMScheduler()
    with pytest.raises(RuntimeError, match="CUDA"):
        s.add_noise(torch.zeros(1, 1, 4, 4), torch.zeros(1, 1, 4, 4), torch.tensor([1]))


SCHEDS = [dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205),
          dict(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0005, beta_end=0.0195),
          dict(num_train_timesteps=250, schedule="sigmoid_beta"),
          dict(num_train_timesteps=1000, schedule="linear_beta", variance_type="fixed_large",
               prediction_type="v_prediction")]


@pytest.mark.parametrize("kw", SCHEDS)
def test_scheduler_tables_and_timesteps_bit_exact_vs_oracle(kw):
    s, o = mig.DDPMScheduler(**kw), ddpm_oracle.OracleDDPMScheduler(**kw)
    assert torch.equal(s.betas, o.betas) and torch.equal(s.alphas_cumprod, o.alphas_cumprod)
    assert torch.equal(s.timesteps, o.timesteps)
    T = kw["num_train_timesteps"]
    for n in (T, T // 2, 50, 7, 3, 1):
        s.set_timesteps(n)
        o.set_timesteps(n)
        assert s.timesteps.dtype == torch.int64 and torch.equal(s.timesteps, o.timesteps)
        assert int(s.timesteps[-1]) == 0 and len(s.timesteps) == n
    with pytest.raises(ValueError):
        s.set_timesteps(T + 1)


@pytest.mark.parametrize("kw", SCHEDS[:2])
def test_step_coefficients_match_oracle_posterior(kw):
    """host-side fp32 scalars == what the oracle's step() uses (checked through a scalar 'tensor')."""
    s, o = mig.DDPMScheduler(**kw), ddpm_oracle.OracleDDPMScheduler(**kw)
    for t in (0, 1, 2, 499, 998, 999):
        k = s.step_coefficients(t)
        x, e, z = torch.tensor([0.3]), torch.tensor([-0.7]), torch.tensor([1.3])
        prev, x0 = o.step(e, t, x, noise=z)
        x0_mine = torch.clamp((x - k["sqrt_one_minus_acp"] * e) / k["sqrt_acp"], -1, 1)
        mine = k["c0"] * x0_mine + k["ct"] * x + k["sigma"] * z
        assert abs(float(mine - prev)) <= 2e-6 * max(1.0, abs(float(prev))), t
        assert k["t_prev"] == t - 1
        if t == 0:
            assert k["sigma"] == 0.0


def test_oracle_scheduler_closed_form_identities():
    """The oracle is unpinned by the reference (third-party, absent): check it against DDPM identities."""
    o = ddpm_oracle.OracleDDPMScheduler(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015,
                                        beta_end=0.0205, clip_sample=False)
    acp = o.alphas_cumprod
    assert torch.all(acp[1:] < acp[:-1]) and 0 < float(acp[-1]) < float(acp[0]) < 1
    g = torch.Generator().manual_seed(0)
    x0, eps = torch.rand(2, 3, 4, 4, 4, generator=g) * 2 - 1, torch.randn(2, 3, 4, 4, 4, generator=g)
    for t in (0, 10, 500, 999):
        ts = torch.tensor([t, t])
        xt = o.add_noise(x0, eps, ts)
        prev, x0_hat = o.step(eps, t, xt, noise=torch.zeros_like(xt))
        assert torch.allclose(x0_hat, x0, atol=2e-3 if t > 900 else 1e-4)       # true eps recovers x0
        v = o.get_velocity(x0, eps, ts)
        a, b = acp[t] ** 0.5, (1 - acp[t]) ** 0.5
        assert torch.allclose(a * xt - b * v, x0, atol=1e-5)                     # v-parameterisation identity
        if t == 0:
            assert torch.allclose(prev, x0, atol=1e-4)                            # posterior mean at t=0 is x0
        else:  # posterior mean of q(x_{t-1}|x_t,x_0) equals sqrt(acp_prev) x0 + sqrt(1-acp_prev-var) * eps direction
            want_mean = (acp[t - 1] ** 0.5 * o.betas[t] / (1 - acp[t])) * x0 + \
                        (o.alphas[t] ** 0.5 * (1 - acp[t - 1]) / (1 - acp[t])) * xt
            assert torch.allclose(prev, want_mean, atol=1e-5)


def test_planner_shapes_for_baseline_configs():
    """The benchmark shapes come from the reference's planner (configuration.py:751-902)."""
    p = O.compute_downsample_parameters([96, 96, 96], 3)
    assert [q[0] for q in p] == [[1, 1, 1], [2, 2, 2], [2, 2, 2]] and O.compute_output_size([96, 96, 96], p) == [24] * 3
    p = O.compute_downsample_parameters([160, 160, 128], 3)
    assert O.compute_output_size([160, 160, 128], p) == [40, 40, 32]
    p = O.compute_downsample_parameters([32, 32, 16], 3)   # thin axis: kernel 1 / pad 0 (the Upsample defect case)
    assert p[0][1] == [3, 3, 1] and p[0][2] == [1, 1, 0]


def test_package_planner_matches_reference_golden(golden):
    """The PACKAGE planner (medical_image_generation_b200/planner.py, what bench.py and users call) against the values the
    unmodified reference functions produced (tests/golden/planner.pt, configuration.py:751-818)."""
    from medical_image_generation_b200 import planner
    plan = golden("planner")
    assert len(plan["params"]) >= 27
    for (size, n), want in plan["params"].items():
        got = planner.compute_downsample_parameters(list(size), n)
        assert got == want, (size, n)
        assert planner.compute_output_size(list(size), got) == plan["out"][(size, n)]


def test_package_planner_kwargs_match_reference_dicts(golden):
    """create_autoencoder_dict / create_ddpm_dict (configuration.py:821-902): the constructor kwargs the package planner
    emits must equal the reference's `vae_params` / `ddpm_params`, stored in tests/golden/reference_checks.pt and, when
    the reference is present, also computed live from it."""
    from oracle import reference_loader as ref
    from oracle.gen_golden_checks import PLANNER_PATCHES, planner_ds_cfg
    from medical_image_generation_b200 import planner
    stored = golden("reference_checks")["planner_dicts"]
    pf = ref.planner_functions() if ref.available() else None
    for patch, in_ch in PLANNER_PATCHES:
        want = stored[(tuple(patch), in_ch)]
        if pf is not None:
            nd = len(patch)
            assert pf["create_autoencoder_dict"](planner_ds_cfg(patch), list(range(in_ch)), nd) == want["vae"], patch
            assert pf["create_ddpm_dict"](planner_ds_cfg(patch), nd) == want["ddpm"], patch
        mine = planner.autoencoder_kwargs(patch, in_channels=in_ch)
        latent = planner.compute_output_size(patch, mine["downsample_parameters"])
        for name, got in (("vae", mine), ("ddpm", planner.ddpm_kwargs(latent, latent_channels=8))):
            assert set(got) == set(want[name])
            for k, v in want[name].items():
                assert got[k] == v, (patch, name, k, got[k], v)


def test_autoencoder_initialize_covers_transposed_convs():
    """InitWeights_He (ae:41-49) re-initialises Conv AND ConvTranspose filters (kaiming normal, a=1e-2) and zeroes biases."""
    from medical_image_generation_b200.layers import ConvNd, ConvTransposeNd
    cfg = dict(CASES["ae3d_convtranspose"]["cfg"])
    m = mig.AutoencoderKL(**cfg)
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    torch.manual_seed(0)
    m.apply(m.initialize)
    seen_t = 0
    for name, mod in m.named_modules():
        if isinstance(mod, (ConvNd, ConvTransposeNd)):
            seen_t += isinstance(mod, ConvTransposeNd)
            assert float(mod.bias.abs().max()) == 0.0, name
            assert not torch.equal(mod.weight, before[name + ".weight"]), name
            fan_in = mod.weight.shape[1] * int(np.prod(mod.weight.shape[2:]))
            want_std = (2.0 / (1 + 1e-2 ** 2)) ** 0.5 / fan_in ** 0.5
            if mod.weight.numel() >= 2048:
                assert abs(float(mod.weight.std()) / want_std - 1) < 0.15, name
    assert seen_t >= 1


def test_compat_install_rebinds_trainer_imports():
    """compat.install() (SURVEY 8f-1): the names the medimgen trainers import resolve to the B200 classes, in the
    defining modules and in an already imported trainer module; uninstall() restores them. Dummy modules stand in for
    medimgen / generative, which are not installed here."""
    import sys
    import types
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import compat

    class Old:  # noqa: D401
        pass

    fakes = {}
    for name in ("medimgen", "generative", "generative.networks"):
        fakes[name] = types.ModuleType(name)
        fakes[name].__path__ = []
    for name, attrs in (("medimgen.diffusion_model_unet_with_strides", ["DiffusionModelUNet"]),
                        ("medimgen.autoencoderkl_with_strides", ["AutoencoderKL"]),
                        ("generative.networks.schedulers", ["DDPMScheduler"]),
                        ("generative.inferers", ["DiffusionInferer", "LatentDiffusionInferer"])):
        m = types.ModuleType(name)
        for a in attrs:
            setattr(m, a, Old)
        fakes[name] = m
    trainer = types.ModuleType("medimgen.train_ldm")
    trainer.DiffusionModelUNet = Old      # `from ... import DiffusionModelUNet` done before install()
    trainer.VQVAE = Old                   # untouched
    fakes["medimgen.train_ldm"] = trainer
    saved = {k: sys.modules.get(k) for k in fakes}
    sys.modules.update(fakes)
    try:
        patched = compat.install()
        assert "generative.inferers.LatentDiffusionInferer" in patched and "medimgen.train_ldm.DiffusionModelUNet" in patched
        assert fakes["medimgen.diffusion_model_unet_with_strides"].DiffusionModelUNet is mig.DiffusionModelUNet
        assert fakes["generative.networks.schedulers"].DDPMScheduler is mig.DDPMScheduler
        assert trainer.DiffusionModelUNet is mig.DiffusionModelUNet and trainer.VQVAE is Old
        compat.uninstall()
        assert fakes["generative.inferers"].DiffusionInferer is Old and trainer.DiffusionModelUNet is Old
    finally:
        compat.uninstall()
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_compat_registers_resident_data_module_when_reference_pipeline_is_not_importable(tmp_path, monkeypatch):
    """`from medimgen.data_processing import get_data_loaders` (train_ldm.py:34) resolves to the resident loaders when the
    reference's module cannot be imported (zarr / blosc2 / batchgenerators missing, as in this image)."""
    import sys
    import medical_image_generation_b200.compat as compat
    from medical_image_generation_b200 import data
    pkgdir = tmp_path / "medimgen"
    pkgdir.mkdir()
    (pkgdir / "__init__.py").write_text("")
    (pkgdir / "data_processing.py").write_text("import zarr_is_not_installed_here\n")
    monkeypatch.syspath_prepend(str(tmp_path))
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("medimgen", "generative")}
    for k in saved:
        del sys.modules[k]
    try:
        patched = compat.install()
        assert any("data_processing" in p for p in patched), patched
        from medimgen.data_processing import get_data_loaders, MedicalDataset
        assert get_data_loaders is data.get_data_loaders and MedicalDataset is data.MedicalDataset
    finally:
        compat.uninstall()
        for k in [k for k in sys.modules if k.split(".")[0] in ("medimgen", "generative")]:
            del sys.modules[k]
        sys.modules.update(saved)
    assert "medimgen.data_processing" not in sys.modules or "medimgen.data_processing" in saved


def test_perceptual_loss_lpips_vgg_fake_3d(tmp_path, monkeypatch):
    """generative.losses.PerceptualLoss as configuration.py:961-964 configures it (row f3): LPIPS-VGG, fake-3D slice
    sampling, weights from a local file only."""
    import sys
    shims = os.path.join(os.path.dirname(mig.__file__), "shims")
    monkeypatch.syspath_prepend(shims)
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "generative"}
    for k in saved:
        del sys.modules[k]
    try:
        from generative.losses import PerceptualLoss
        monkeypatch.delenv("MEDIMGEN_LPIPS_WEIGHTS", raising=False)
        with pytest.raises(RuntimeError, match="local file"):
            PerceptualLoss(spatial_dims=3, network_type="vgg", is_fake_3d=True, fake_3d_ratio=0.2)
        with pytest.raises(NotImplementedError):
            PerceptualLoss(spatial_dims=3, network_type="medicalnet_resnet10_23datasets", is_fake_3d=False, pretrained=False)
        torch.manual_seed(0)
        pl = PerceptualLoss(spatial_dims=3, network_type="vgg", is_fake_3d=True, fake_3d_ratio=0.25, pretrained=False)
        assert all(not p.requires_grad for p in pl.parameters()) and not pl.perceptual_function.training
        pl.train()
        assert not pl.perceptual_function.training          # frozen metric network
        a = torch.rand(2, 1, 16, 16, 16, requires_grad=True)
        b = torch.rand(2, 1, 16, 16, 16)
        seen = []
        orig = pl.perceptual_function.forward
        pl.perceptual_function.forward = lambda x, y, **k: (seen.append(tuple(x.shape)), orig(x, y, **k))[1]
        loss = pl(a, b)
        assert seen == [(8, 1, 16, 16)] * 3                  # int(2 * 16 * 0.25) slices along each of the three axes
        assert loss.ndim == 0 and float(loss) > 0
        loss.backward()
        assert float(a.grad.abs().sum()) > 0
        assert float(pl(b, b)) == 0.0
        with pytest.raises(ValueError):
            pl(a, b[:, :, :8])
        # symmetric in its arguments (same slice draw)
        torch.manual_seed(3); l1 = float(pl(a.detach(), b))
        torch.manual_seed(3); l2 = float(pl(b, a.detach()))
        assert abs(l1 - l2) < 1e-6
        # weights from a file: the lpips package's key layout, lin layers stored twice
        sd = dict(pl.perceptual_function.state_dict())
        assert "net.slice1.0.weight" in sd and "net.slice5.28.bias" in sd and "lin4.model.1.weight" in sd
        sd.update({f"lins.{k}.model.1.weight": sd[f"lin{k}.model.1.weight"] for k in range(5)})
        path = tmp_path / "lpips_vgg.pt"
        torch.save(sd, path)
        monkeypatch.setenv("MEDIMGEN_LPIPS_WEIGHTS", str(path))
        pl2 = PerceptualLoss(spatial_dims=3, network_type="vgg", is_fake_3d=True, fake_3d_ratio=0.25)
        torch.manual_seed(3)
        assert abs(float(pl2(a.detach(), b)) - l1) < 1e-7
        p2d = PerceptualLoss(spatial_dims=2, network_type="vgg", pretrained=False)
        assert float(p2d(torch.rand(2, 1, 32, 32), torch.rand(2, 1, 32, 32))) > 0
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] == "generative"]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_upconv_fold_algebra_fp64():
    """The sub-pixel decomposition behind ops.upsample_conv_nd (csrc/upconv.cu), in fp64 on the CPU with the package's own
    fold table (ops._axis_fold): per-class convolutions of the low-resolution tensor == conv(nearest_upsample(x)); the
    stride-f convolution of dy with the folded (f + k - 1)^n-tap filter == d/dx; class wgrads unfolded == d/dw."""
    import itertools
    import torch.nn.functional as F
    from medical_image_generation_b200 import ops
    torch.manual_seed(0)
    for f3, k3, p3, n3 in [((2, 2, 2), (3, 3, 3), (1, 1, 1), (3, 4, 5)), ((2, 2, 1), (3, 3, 3), (1, 1, 1), (4, 3, 5)),
                           ((1, 2, 2), (1, 3, 3), (0, 1, 1), (1, 5, 4))]:
        x = torch.randn(2, 3, *n3, dtype=torch.float64, requires_grad=True)
        w = torch.randn(4, 3, *k3, dtype=torch.float64, requires_grad=True)
        b = torch.randn(4, dtype=torch.float64)
        xu = x
        for i in range(3):
            xu = xu.repeat_interleave(f3[i], dim=2 + i)
        ref = F.conv3d(xu, w, b, padding=p3)
        dy = torch.randn_like(ref)
        gx, gw = torch.autograd.grad(ref, (x, w), dy)
        folds = [ops._axis_fold(k3[i], f3[i], p3[i]) for i in range(3)]
        y = torch.zeros_like(ref)
        dW = torch.zeros_like(w)
        xd, wd_ = x.detach(), w.detach()
        for r in itertools.product(*[range(v) for v in f3]):
            base = [folds[i][r[i]][0] for i in range(3)]
            nu = [folds[i][r[i]][1] for i in range(3)]
            umap = {t: tuple((r[i] + t[i] - p3[i]) // f3[i] - base[i] for i in range(3))
                    for t in itertools.product(*[range(v) for v in k3])}
            wc = torch.zeros(4, 3, *nu, dtype=torch.float64)
            for t, u in umap.items():
                wc[(slice(None), slice(None)) + u] += wd_[(slice(None), slice(None)) + t]
            pad = []
            for i in (2, 1, 0):     # pad_before = -base, pad_after = nu - 1 + base: out_dims = in_dims
                pad += [-base[i], nu[i] - 1 + base[i]]
            xp = F.pad(xd, pad)
            y[:, :, r[0]::f3[0], r[1]::f3[1], r[2]::f3[2]] = F.conv3d(xp, wc, b)
            dyc = dy[:, :, r[0]::f3[0], r[1]::f3[1], r[2]::f3[2]]
            dwc = torch.zeros_like(wc)
            for u in itertools.product(*[range(v) for v in nu]):
                xs = xp[:, :, u[0]:u[0] + n3[0], u[1]:u[1] + n3[1], u[2]:u[2] + n3[2]]
                dwc[(slice(None), slice(None)) + u] = torch.einsum("nodhw,nidhw->oi", dyc, xs)
            for t, u in umap.items():
                dW[(slice(None), slice(None)) + t] += dwc[(slice(None), slice(None)) + u]
        assert float((y - ref).abs().max()) < 1e-12
        assert float((dW - gw).abs().max()) < 1e-11
        K2 = [f3[i] + k3[i] - 1 for i in range(3)]
        pad2 = [k3[i] - 1 - p3[i] for i in range(3)]
        wd = torch.zeros(3, 4, *K2, dtype=torch.float64)
        for s in itertools.product(*[range(v) for v in K2]):
            for t in itertools.product(*[range(v) for v in k3]):
                if all(0 <= (s[i] - pad2[i]) + t[i] - p3[i] < f3[i] for i in range(3)):
                    wd[(slice(None), slice(None)) + s] += wd_[(slice(None), slice(None)) + t].t()
        dx = F.conv3d(dy, wd, None, stride=f3, padding=pad2)
        assert dx.shape == gx.shape and float((dx - gx).abs().max()) < 1e-11


def test_lpips_vgg_trunk_matches_torchvision_vgg16_layout(monkeypatch):
    """The perceptual loss's trunk (shims/generative/losses/perceptual.py) against torchvision's vgg16 definition -- the
    network the `lpips` package slices: same conv indices / shapes (so `net.slice*.N.*` keys of a real LPIPS state dict
    load) and, with the weights copied over, the same relu1_2 / 2_2 / 3_3 / 4_3 / 5_3 feature maps."""
    import sys
    torchvision = pytest.importorskip("torchvision")
    shims = os.path.join(os.path.dirname(mig.__file__), "shims")
    monkeypatch.syspath_prepend(shims)
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "generative"}
    for k in saved:
        del sys.modules[k]
    try:
        from generative.losses.perceptual import LPIPS
        torch.manual_seed(0)
        tv = torchvision.models.vgg16(weights=None).features.eval()
        lp = LPIPS(pretrained=False)
        sd = {}
        for k in range(1, 6):
            for name, mod in getattr(lp.net, f"slice{k}").named_children():
                ref_mod = tv[int(name)]
                assert type(mod) is type(ref_mod), (k, name)
                if isinstance(mod, torch.nn.Conv2d):
                    assert mod.weight.shape == ref_mod.weight.shape and mod.padding == ref_mod.padding
                    sd[f"slice{k}.{name}.weight"], sd[f"slice{k}.{name}.bias"] = ref_mod.weight, ref_mod.bias
        lp.net.load_state_dict(sd)
        x = torch.rand(2, 3, 32, 32)
        feats = lp.net(x)
        taps, h = [], x
        for i, layer in enumerate(tv):
            h = layer(h)
            if i in (3, 8, 15, 22, 29):
                taps.append(h)
        assert len(feats) == 5
        for a, b in zip(feats, taps):
            assert a.shape == b.shape and torch.allclose(a, b, atol=1e-6)
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] == "generative"]:
            del sys.modules[k]
        sys.modules.update(saved)
