"""CPU: anchors the unpinned likelihood oracle (oracle/likelihood_oracle.py) with identities, checks the host table the
vlb kernel reads against it, and the argument errors of the public get_likelihood methods (raised before any device
work)."""
import math

import pytest
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import planner
from oracle import likelihood_oracle as L
from oracle.ddim_oracle import OracleDDIMScheduler
from oracle.ddpm_oracle import OracleDDPMScheduler

LDM = planner.LDM_SCHEDULER_KWARGS


def _inputs(shape, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g) * 2 - 1
    x.view(-1)[:4] = torch.tensor([-1.0, 1.0, -0.9995, 0.9995])     # all three decoder branches
    return x, torch.randn(shape, generator=g)


def test_kl_term_is_the_kl_divergence_of_two_normals():
    g = torch.Generator().manual_seed(0)
    m1, m2 = (torch.randn(1000, generator=g, dtype=torch.float64) for _ in range(2))
    lv1, lv2 = (torch.randn(1000, generator=g, dtype=torch.float64) * 3 for _ in range(2))
    want = torch.distributions.kl_divergence(torch.distributions.Normal(m1, (0.5 * lv1).exp()),
                                             torch.distributions.Normal(m2, (0.5 * lv2).exp()))
    got = L.normal_kl(m1, lv1, m2, lv2)
    assert float(((got - want).abs() / want.abs().clamp_min(1e-300)).max()) < 1e-12


def test_tanh_cdf_within_its_approximation_error():
    x = torch.linspace(-8, 8, 160001, dtype=torch.float64)
    exact = 0.5 * (1 + torch.erf(x / math.sqrt(2)))
    err = float((L.approx_standard_normal_cdf(x) - exact).abs().max())
    assert 1e-4 < err < 2e-4, err            # the tanh form's known worst case, ~1.9e-4 near |x| = 2


@pytest.mark.parametrize("variance_type", ["fixed_small", "fixed_large"])
def test_epsilon_model_given_the_true_noise_has_rounding_level_kl(variance_type):
    x, noise = _inputs((2, 1, 6, 5, 4), 1)
    s = OracleDDPMScheduler(variance_type=variance_type, clip_sample=False, **LDM)
    _, inter = L.get_likelihood(s, x, lambda noisy, timesteps, context: noise, save_intermediates=True, noise=noise)
    worst = max(float(k.abs().max()) for t, k in zip(s.timesteps, inter) if int(t) > 0)
    assert worst < 1e-5, worst


@pytest.mark.parametrize("variance_type", ["fixed_small", "fixed_large"])
def test_sample_model_returning_the_input_gives_the_closed_form_bound(variance_type):
    """x0_hat = x0 exactly: every KL term is its constant part 0.5 (-1 + lv - lv + exp(0)) (fp32 rounding of -1 + lv),
    and the decoder mean is within 1e-5 of x0. fixed_small: a scale of 1e-10, so the decoder term is -log(1) = 0.
    fixed_large: a scale of sqrt(beta_0), so it is -log of the mass of the bin (inner) or half-line (the ends) around
    x0, a function of the branch alone."""
    x, noise = _inputs((2, 1, 6, 5, 4), 2)
    kw = dict(LDM, prediction_type="sample")
    s = OracleDDPMScheduler(variance_type=variance_type, clip_sample=False, **kw)
    total, inter = L.get_likelihood(s, x, lambda noisy, timesteps, context: x, save_intermediates=True, noise=noise)
    want = 0.0
    for t in range(1, 1000):
        lv = torch.log(s._variance(t))
        want += 0.5 * float(-1.0 + lv - lv + torch.exp(lv - lv))
    if variance_type == "fixed_small":
        assert float(inter[-1].abs().max()) == 0.0
        atol = 1e-9
    else:
        cdf = lambda v: 0.5 * (1 + math.tanh(math.sqrt(2 / math.pi) * (v + 0.044715 * v ** 3)))  # noqa: E731
        a = 0.5 / 255 / math.sqrt(float(s.betas[0]))
        ends = (x.abs() > 0.999).double()
        dec = ends * -math.log(cdf(a)) + (1 - ends) * -math.log(cdf(a) - cdf(-a))
        assert torch.allclose(inter[-1].double(), dec, rtol=0, atol=1e-3)
        want = want + dec.view(2, -1).mean(1)
        atol = 1e-4
    want = torch.as_tensor(want, dtype=torch.float64).expand(2)
    assert torch.allclose(total.double(), want, rtol=0, atol=atol), (total, want)


def test_decoder_branches():
    hb = 0.5 / 255
    x = torch.tensor([-1.0, 1.0, 0.3, -0.3])
    mu = torch.tensor([-0.98, 0.97, 0.31, -0.3])
    log_scale = torch.tensor(math.log(0.02))
    got = L.decoder_log_likelihood(x, mu, log_scale)
    cdf = lambda v: 0.5 * (1 + math.tanh(math.sqrt(2 / math.pi) * (v + 0.044715 * v ** 3)))  # noqa: E731
    want = []
    for xi, mi in zip(x.tolist(), mu.tolist()):
        hi, lo = cdf((xi - mi + hb) / 0.02), cdf((xi - mi - hb) / 0.02)
        want.append(math.log(hi) if xi < -0.999 else math.log(1 - lo) if xi > 0.999 else math.log(hi - lo))
    assert torch.allclose(got.double(), torch.tensor(want, dtype=torch.float64), rtol=2e-5, atol=0), (got, want)
    # the end bins reach to infinity: far more mass than an inner bin at the same distance
    assert got[0] > got[2] and got[1] > got[2]


def test_intermediates_sum_to_the_total_and_short_schedules_index_t_minus_one():
    """With set_timesteps(10) the loop visits 900, ..., 0 and, as upstream, the coefficients of timestep t use
    alphas_cumprod[t - 1] (not the previous timestep of the schedule). A sample model returning a fixed m gives
    kl = 0.5 (c + c0^2 (x0 - m)^2 / var) with c0 and var of t and t - 1, checked in fp64 (c is below 3e-7)."""
    x, noise = _inputs((3, 2, 4, 4, 4), 3)
    m = torch.rand(x.shape, generator=torch.Generator().manual_seed(4)) * 2 - 1
    s = OracleDDPMScheduler(clip_sample=False, **dict(LDM, prediction_type="sample"))
    s.set_timesteps(10)
    seen = []

    def model(noisy, timesteps, context):
        seen.append(int(timesteps[0]))
        return m

    total, inter = L.get_likelihood(s, x, model, save_intermediates=True, noise=noise)
    assert seen == list(range(900, -1, -100)) and len(inter) == 10
    means = torch.stack([k.view(3, -1).double().mean(1) for k in inter]).sum(0)
    assert torch.allclose(total.double(), means, rtol=1e-6, atol=0)
    acp = s.alphas_cumprod.double()
    for t, k in zip(seen[:-1], inter[:-1]):
        beta = float(s.betas[t])
        var = (1 - acp[t - 1]) / (1 - acp[t]) * beta
        c0 = acp[t - 1].sqrt() * beta / (1 - acp[t])
        want = 0.5 * c0 ** 2 * (x.double() - m.double()) ** 2 / var
        # fp32 cancellation in (c0 x0 + ct x_t) - (c0 m + ct x_t) when c0 << ct: measured 1.2e-4 at t = 900; indexing
        # with the schedule's previous timestep t - 100 instead would change c0^2 / var by orders of magnitude
        assert float(((k.double() - want).norm() / want.norm())) < 1e-3, t


def test_host_table_matches_the_oracle():
    """The table the vlb kernel reads: c0 and ct of `step` equal those of upstream `_get_mean` bit for bit, and the
    variance terms are those the oracle evaluates."""
    for vt in ("fixed_small", "fixed_large"):
        s = mig.DDPMScheduler(variance_type=vt, **LDM)
        o = OracleDDPMScheduler(variance_type=vt, **LDM)
        tab = s.vlb_coefficients()
        assert tab.shape == (1000, len(s.VLB_COEFS)) and tab.dtype == torch.float32
        for t in (0, 1, 2, 500, 998, 999):
            acp_prev = o.alphas_cumprod[t - 1] if t > 0 else o.one
            c0 = acp_prev.sqrt() * o.betas[t] / (1 - o.alphas_cumprod[t])
            ct = o.alphas[t].sqrt() * (1 - acp_prev) / (1 - o.alphas_cumprod[t])
            lv = torch.log(o._variance(t))
            want = [o.alphas_cumprod[t] ** 0.5, (1 - o.alphas_cumprod[t]) ** 0.5, c0, ct,
                    -1.0 + lv - lv + torch.exp(lv - lv), torch.exp(-lv), torch.exp(-(0.5 * lv))]
            assert torch.equal(tab[t], torch.stack([torch.as_tensor(w, dtype=torch.float32) for w in want])), (vt, t)


def test_errors():
    x = torch.zeros(1, 1, 4, 4, 4)
    model = lambda noisy, timesteps, context: noisy  # noqa: E731
    with pytest.raises(NotImplementedError, match="DDPMScheduler"):
        L.get_likelihood(OracleDDIMScheduler(**LDM), x, model)
    with pytest.raises(NotImplementedError):
        L.get_likelihood(OracleDDPMScheduler(**LDM), x, model, mode="add")
    with pytest.raises(ValueError):
        L.latent_get_likelihood(OracleDDPMScheduler(**LDM), 1.0, x, None, model, resample_latent_likelihoods=True)
    with pytest.raises(ValueError):
        L.latent_get_likelihood(OracleDDPMScheduler(**LDM), 1.0, x, None, model, save_intermediates=True,
                                resample_latent_likelihoods=True, resample_interpolation_mode="bicubic")
    # the package raises the same errors before touching a device
    with pytest.raises(NotImplementedError, match="only compatible with DDPMScheduler"):
        mig.DiffusionInferer(mig.DDIMScheduler(**LDM)).get_likelihood(x, model)
    with pytest.raises(NotImplementedError, match="condition is not supported"):
        mig.DiffusionInferer(mig.DDPMScheduler(**LDM)).get_likelihood(x, model, mode="add")
    lat = mig.LatentDiffusionInferer(mig.DDPMScheduler(**LDM))
    with pytest.raises(ValueError, match="save_intermediates"):
        lat.get_likelihood(x, None, model, resample_latent_likelihoods=True)
    with pytest.raises(ValueError, match="nearest, bilinear, or trilinear"):
        lat.get_likelihood(x, None, model, save_intermediates=True, resample_latent_likelihoods=True,
                           resample_interpolation_mode="bicubic")
