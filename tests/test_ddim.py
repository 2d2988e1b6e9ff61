"""DDIMScheduler host logic against the CPU oracle (oracle/ddim_oracle.py), and the closed-form identities that anchor
that oracle, whose parity with monai-generative is otherwise unpinned. No device needed."""
import pytest
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import planner
from oracle.ddim_oracle import OracleDDIMScheduler
from oracle.ddpm_oracle import OracleDDPMScheduler
from test_host_logic import SCHEDS

# DDIM takes no variance_type: keep the beta schedules (and prediction types) of the DDPM parity tests
DDIM_SCHEDS = [{k: v for k, v in kw.items() if k != "variance_type"} for kw in SCHEDS]
LDM = planner.LDM_SCHEDULER_KWARGS


def _kernel_formula(k, pred, clip, m, x, z):
    """What ddim_step_kernel computes per element from the scalars of `step_coefficients` (fp32)."""
    sa, sb = k["sqrt_acp"], k["sqrt_one_minus_acp"]
    if pred == "epsilon":
        x0, eps = (x - sb * m) / sa, m
    elif pred == "sample":
        x0 = m
        eps = (x - sa * x0) / sb
    else:
        x0, eps = sa * x - sb * m, sa * m + sb * x
    if clip:
        x0 = torch.clamp(x0, -1, 1)
    return k["sqrt_acp_prev"] * x0 + k["dir_coef"] * eps + k["sigma"] * z, x0


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("kw", DDIM_SCHEDS)
def test_tables_identical_to_ddpm(kw):
    d, p = mig.DDIMScheduler(**kw), mig.DDPMScheduler(**kw)
    for name in ("betas", "alphas", "alphas_cumprod"):
        assert torch.equal(getattr(d, name), getattr(p, name)), name
    o = OracleDDIMScheduler(**kw)
    assert torch.equal(d.alphas_cumprod, o.alphas_cumprod) and torch.equal(d.timesteps, o.timesteps)
    assert d.num_inference_steps == o.num_inference_steps == kw["num_train_timesteps"]


def test_constructor_takes_the_ldm_kwargs_and_upstream_arguments():
    s = mig.DDIMScheduler(**LDM)
    assert s.prediction_type == "epsilon" and s.clip_sample and float(s.final_alpha_cumprod) == 1.0
    s = mig.DDIMScheduler(**LDM, set_alpha_to_one=False, steps_offset=1, clip_sample=False)
    assert torch.equal(s.final_alpha_cumprod, s.alphas_cumprod[0]) and s.steps_offset == 1 and not s.clip_sample
    with pytest.raises(ValueError):
        mig.DDIMScheduler(prediction_type="x0")
    from medical_image_generation_b200.shims.generative.networks.schedulers import DDIMScheduler
    assert DDIMScheduler is mig.DDIMScheduler


@pytest.mark.parametrize("kw", DDIM_SCHEDS)
@pytest.mark.parametrize("offset", [0, 1])
def test_set_timesteps_bit_exact_vs_oracle(kw, offset):
    s, o = mig.DDIMScheduler(steps_offset=offset, **kw), OracleDDIMScheduler(steps_offset=offset, **kw)
    T = kw["num_train_timesteps"]
    checked = 0
    for n in (T, T // 2, 50, 7, 3, 1):
        if offset >= T // n:
            for sch in (s, o):
                with pytest.raises(ValueError):
                    sch.set_timesteps(n)
            continue
        s.set_timesteps(n)
        o.set_timesteps(n)
        assert s.timesteps.dtype == torch.int64 and torch.equal(s.timesteps, o.timesteps), n
        assert len(s.timesteps) == n and int(s.timesteps[-1]) == offset and s.num_inference_steps == n
        assert int(s.timesteps[0]) == (n - 1) * (T // n) + offset
        checked += 1
    assert checked == (6 if offset == 0 else 5)
    with pytest.raises(ValueError):
        s.set_timesteps(T + 1)


def _coefficient_cases(kw):
    """(n, timesteps) of the schedules checked: every step of a 50-step and a 7-step schedule, and the n = T steps
    around both ends."""
    T = kw["num_train_timesteps"]
    return [(50, None), (7, None), (T, [T - 1, T // 2, 2, 1, 0])]


@pytest.mark.parametrize("kw", DDIM_SCHEDS[:2] + [dict(LDM, prediction_type="v_prediction")])
@pytest.mark.parametrize("set_alpha_to_one", [True, False])
@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_step_coefficients_reproduce_the_oracle_step(kw, set_alpha_to_one, pred):
    kw = dict(kw, prediction_type=pred)
    g = torch.Generator().manual_seed(3)
    # values whose x0 prediction falls both inside and outside [-1, 1], so clipping and the unclipped eps both matter
    x = torch.tensor([0.3, 2.5, -3.0, 0.9, -0.05])
    m = torch.tensor([-0.7, 0.1, 0.9, 1.4, -2.2])
    z = torch.randn(5, generator=g)
    worst = 0.0
    for clip in (True, False):
        s = mig.DDIMScheduler(clip_sample=clip, set_alpha_to_one=set_alpha_to_one, **kw)
        o = OracleDDIMScheduler(clip_sample=clip, set_alpha_to_one=set_alpha_to_one, **kw)
        for n, ts in _coefficient_cases(kw):
            s.set_timesteps(n)
            o.set_timesteps(n)
            for t in (ts if ts is not None else [int(t) for t in s.timesteps]):
                for eta in (0.0, 1.0):
                    k = s.step_coefficients(t, eta)
                    assert k["t_prev"] == t - kw["num_train_timesteps"] // n
                    prev, x0 = _kernel_formula(k, pred, clip, m, x, z)
                    wprev, wx0 = o.step(m, t, x, eta=eta, noise=z)
                    err = float((prev - wprev).abs().max()) / max(1.0, float(wprev.abs().max()))
                    assert err <= 2e-6, (n, t, eta, clip, err)
                    assert float((x0 - wx0).abs().max()) <= 2e-6 * max(1.0, float(wx0.abs().max())), (n, t, clip)
                    worst = max(worst, err)
                if t + kw["num_train_timesteps"] // n < kw["num_train_timesteps"]:
                    k = s.reversed_step_coefficients(t)
                    assert k["sigma"] == 0.0
                    nxt, _ = _kernel_formula(k, pred, clip, m, x, z)
                    wnxt, _ = o.reversed_step(m, t, x)
                    assert float((nxt - wnxt).abs().max()) <= 2e-6 * max(1.0, float(wnxt.abs().max())), (n, t)
                else:
                    for sch in (s, o):
                        with pytest.raises(IndexError):
                            (sch.reversed_step_coefficients(t) if sch is s else o.reversed_step(m, t, x))
    assert worst <= 2e-6


def test_final_step_uses_final_alpha_cumprod():
    """The step past timestep 0 lands on x0 (alpha_bar = 1) or on alpha_bar[0] (set_alpha_to_one=False)."""
    for one in (True, False):
        s = mig.DDIMScheduler(set_alpha_to_one=one, **LDM)
        s.set_timesteps(50)
        k = s.step_coefficients(0)
        want = 1.0 if one else float(s.alphas_cumprod[0] ** 0.5)
        assert k["t_prev"] == -20 and k["sqrt_acp_prev"] == pytest.approx(want, abs=0, rel=1e-7)
        if one:
            assert k["dir_coef"] == 0.0


# ---- identities that anchor the oracle ----------------------------------------------------------------------------------
def _fixture(T_kw, seed=0):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(2, 1, 6, 5, 4, generator=g) * 1.6 - 0.8
    eps = torch.randn(2, 1, 6, 5, 4, generator=g)
    return x0, eps, OracleDDPMScheduler(**T_kw)


def _model_output(pred, ddpm, x0, eps, t):
    tt = torch.tensor([t, t])
    return {"epsilon": eps, "sample": x0, "v_prediction": ddpm.get_velocity(x0, eps, tt)}[pred]


@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_identity_exact_step_lands_on_the_previous_marginal(pred):
    """With the true eps, eta = 0 and clipping off, step(add_noise(x0, eps, t)) = add_noise(x0, eps, t_prev)."""
    x0, eps, ddpm = _fixture(LDM)
    o = OracleDDIMScheduler(clip_sample=False, **dict(LDM, prediction_type=pred))
    o.set_timesteps(50)
    worst = 0.0
    for t in [int(t) for t in o.timesteps]:
        xt = ddpm.add_noise(x0, eps, torch.tensor([t, t]))
        prev, x0h = o.step(_model_output(pred, ddpm, x0, eps, t), t, xt)
        want = ddpm.add_noise(x0, eps, torch.tensor([t - 20] * 2)) if t >= 20 else x0
        worst = max(worst, _rel(prev, want))
        assert _rel(x0h, x0) < 5e-5, t     # measured 5.3e-6: 1/sqrt(alpha_bar) amplifies fp32 rounding at large t
    assert worst < 1e-6, worst            # measured 8.8e-8


@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_identity_inversion_lands_on_the_next_marginal(pred):
    x0, eps, ddpm = _fixture(LDM, seed=1)
    o = OracleDDIMScheduler(clip_sample=False, **dict(LDM, prediction_type=pred))
    o.set_timesteps(50)
    worst = 0.0
    for t in [int(t) for t in o.timesteps.flip(0)][:-1]:
        xt = ddpm.add_noise(x0, eps, torch.tensor([t, t]))
        nxt, _ = o.reversed_step(_model_output(pred, ddpm, x0, eps, t), t, xt)
        worst = max(worst, _rel(nxt, ddpm.add_noise(x0, eps, torch.tensor([t + 20] * 2))))
    assert worst < 1e-6, worst            # measured 1.2e-7
    with pytest.raises(IndexError):
        o.reversed_step(eps, 980, x0)


@pytest.mark.parametrize("pred", ["epsilon", "sample", "v_prediction"])
def test_identity_full_schedule_eta_one_is_ddpm(pred):
    """n = T, eta = 1, clipping off: the DDIM step is the DDPM fixed_small posterior step given the same z."""
    kw = dict(LDM, prediction_type=pred)
    g = torch.Generator().manual_seed(2)
    o = OracleDDIMScheduler(clip_sample=False, **kw)
    p = OracleDDPMScheduler(clip_sample=False, variance_type="fixed_small", **kw)
    o.set_timesteps(1000)
    p.set_timesteps(1000)
    worst = 0.0
    for t in (999, 998, 700, 500, 100, 10, 2, 1, 0):
        m, x, z = (torch.randn(2, 1, 6, 5, 4, generator=g) for _ in range(3))
        got, gx0 = o.step(m, t, x, eta=1.0, noise=z)
        want, wx0 = p.step(m, t, x, noise=z)
        worst = max(worst, _rel(got, want))
        assert _rel(gx0, wx0) < 1e-6, t
    assert worst < 3e-5, worst            # measured 6.9e-6 (sqrt(1 - alpha_bar_prev - sigma^2) cancels near t = 1)
