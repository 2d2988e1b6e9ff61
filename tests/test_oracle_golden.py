"""CPU: pin oracle/ (the restatement) to the committed golden vectors produced by the UNMODIFIED
reference (oracle/gen_golden.py), and - when /root/reference is present - to the reference live."""
import numpy as np
import pytest
import torch

from oracle import torch_oracle as O
from oracle import reference_loader as ref
from oracle.golden_util import CASES, golden_params, sketch

UNET_CASES = [k for k, v in CASES.items() if v["kind"] == "unet"]
AE_CASES = [k for k, v in CASES.items() if v["kind"] == "ae"]


def rel_err(a, b, floor=1e-30):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / b.norm().clamp_min(floor))


def sketch_err(grad, want):
    """Gradients that are mathematically zero (e.g. to_k.bias: softmax is shift-invariant) are fp noise
    ~1e-7 on both sides, so the denominator is floored."""
    return rel_err(sketch(grad), want, floor=0.1)


def _leaf_params(g):
    return {k: v.clone().requires_grad_(True) for k, v in golden_params(g["shapes"], g["seed"]).items()}


@pytest.mark.parametrize("name", UNET_CASES)
def test_unet_oracle_matches_reference_golden(golden, name):
    g = golden(name)
    sd = _leaf_params(g)
    inp = g["inputs"]
    x = inp["x"].clone().requires_grad_(True)
    taps = {}
    y = O.unet_forward(sd, g["cfg"], x, inp["timesteps"], context=inp.get("context"),
                       class_labels=inp.get("class_labels"), taps=taps)
    assert rel_err(y, g["out"]) < 1e-5
    assert rel_err(taps["conv_in"], g["taps"]["conv_in"]) < 1e-5
    assert rel_err(taps["mid"], g["taps"]["mid"]) < 1e-5
    (y * inp["probe"]).sum().backward()
    assert rel_err(x.grad, g["grad_x"]) < 1e-4
    for k, sk in g["grad_sketch"].items():
        assert sd[k].grad is not None, k
        assert sketch_err(sd[k].grad, sk) < 1e-3, k
    for k in g["no_grad_params"]:  # proj_attn is created but never applied (unet:383 vs 418-458)
        assert sd[k].grad is None and "proj_attn" in k


@pytest.mark.parametrize("name", AE_CASES)
def test_ae_oracle_matches_reference_golden(golden, name):
    g = golden(name)
    sd = _leaf_params(g)
    inp = g["inputs"]
    x = inp["x"].clone().requires_grad_(True)
    recon, z_mu, z_sigma = O.ae_forward(sd, g["cfg"], x, inp["eps"])
    assert rel_err(recon, g["out"]) < 1e-5
    assert rel_err(z_mu, g["z_mu"]) < 1e-5 and rel_err(z_sigma, g["z_sigma"]) < 1e-5
    kl = O.kl_loss(z_mu, z_sigma)
    assert rel_err(kl, g["kl"]) < 1e-5
    loss = torch.nn.functional.l1_loss(recon, inp["x"]) + 1e-7 * kl
    assert rel_err(loss, g["loss"]) < 1e-5
    loss.backward()
    assert rel_err(x.grad, g["grad_x"]) < 1e-4
    for k, sk in g["grad_sketch"].items():
        assert sketch_err(sd[k].grad, sk) < 1e-3, k


def test_planner_restatement_matches_reference_golden(golden):
    plan = golden("planner")
    for (size, n), want in plan["params"].items():
        got = O.compute_downsample_parameters(list(size), n)
        assert got == want, (size, n)
        assert O.compute_output_size(list(size), got) == plan["out"][(size, n)]


def test_timestep_embedding_cos_first_and_odd_pad():
    t = torch.tensor([0, 1, 999])
    e = O.timestep_embedding(t, 7)
    assert e.shape == (3, 7)
    assert torch.all(e[0, :3] == 1) and torch.all(e[0, 3:6] == 0) and torch.all(e[:, 6] == 0)
    with pytest.raises(ValueError):
        O.timestep_embedding(t[None], 8)


@pytest.mark.skipif(not ref.available(), reason="/root/reference not present (GPU box)")
def test_oracle_matches_live_reference_default_widths():
    """LDM-default widths at a tiny latent: oracle == unmodified reference, live."""
    cfg = dict(spatial_dims=3, in_channels=3, out_channels=3, num_res_blocks=2, num_channels=[64, 128, 192],
               attention_levels=[False, True, True], num_head_channels=[0, 128, 192],
               strides=[[1, 1, 1], [2, 2, 2], [2, 2, 2]], kernel_sizes=[[3, 3, 3]] * 3, paddings=[[1, 1, 1]] * 3)
    torch.manual_seed(0)
    m = ref.unet_module().DiffusionModelUNet(**cfg)
    ref.rerandomize_zero_init(m)
    x, t = torch.randn(1, 3, 8, 8, 8), torch.tensor([417])
    with torch.no_grad():
        want = m(x, t)
        got = O.unet_forward(m.state_dict(), cfg, x, t)
    assert float(want.abs().max()) > 1e-3
    assert rel_err(got, want) < 1e-5


def test_reference_quirks_hold(golden):
    """SURVEY section 0.6: fresh U-Net output is exactly 0; default constructors raise IndexError. The reference's
    outcomes are stored in tests/golden/reference_checks.pt; the package (through the oracle for the forward) must
    reproduce them, and the reference itself is checked against them when present."""
    import medical_image_generation_b200 as mig
    want = golden("reference_checks")["quirks"]
    cfg = CASES["unet3d_small"]["cfg"]
    x, t = torch.randn(1, 3, 8, 8, 8), torch.tensor([3])
    impls = [(mig.DiffusionModelUNet, mig.AutoencoderKL, lambda m: O.unet_forward(m.state_dict(), cfg, x, t))]
    if ref.available():
        impls.append((ref.unet_module().DiffusionModelUNet, ref.ae_module().AutoencoderKL, lambda m: m(x, t)))
    for U, AE, forward in impls:
        with pytest.raises(Exception) as e:
            U(spatial_dims=3, in_channels=1, out_channels=1)
        assert type(e.value).__name__ == want["DiffusionModelUNet(spatial_dims=3, in_channels=1, out_channels=1)"]
        with pytest.raises(Exception) as e:
            AE(spatial_dims=3)
        assert type(e.value).__name__ == want["AutoencoderKL(spatial_dims=3)"]
        with torch.no_grad():
            y = forward(U(**cfg))
        assert float(y.abs().max()) == want["fresh U-Net output max |y|"]
