"""The optimiser kernels through the C ABI (`_lib.call`), against an fp64 restatement of clip_grad_norm_ + one
torch.optim.AdamW step: `mig_sumsq`, `mig_sumsq_strided`, `mig_adamw_step` and `mig_adamw_step_strided`.

The strided entry points are what the sharded data-parallel optimiser runs: rank r owns slice r (`piece` = bucket / W
elements) of every gradient bucket and calls them at element r * piece with (piece, stride = bucket, count = nb). Here
W ranks are emulated on one device: before each rank's call every element the rank does not own is NaN, so a read of a
wrong element shows up in the result and a write to one shows up as a changed NaN.

Every comparison is one step: the reference is fed the kernel's own fp32 state from before the step, so only that step's
arithmetic is compared. Hyperparameters are rounded to fp32 before the reference sees them, because that is what crosses
the ABI (1 - f32(0.999) is 1.3e-5 away from 0.001)."""
import ctypes as C
import math

import pytest
import torch

from util import adam_step_scale, clip_adamw_reference, f32, ulp32

gpu = pytest.mark.gpu
DEV = "cuda"

# BASELINE config 3 (bench.py at 8 GPUs, bucket_mb 64): the sharded region is 26 buckets of 16,777,216 elements; the
# used region adds the replicated one. test_config3_layout_matches_bench_unet derives these from the bench U-Net.
C3_BUCKET, C3_NB, C3_SHARD, C3_USED = 16_777_216, 26, 436_207_616, 447_074_880

# bars, with the worst value measured on a B200 next to each. m and p are measured against the magnitude of the terms
# that make them up, because the terms can cancel: b1 m0 against (1 - b1) clip g in m, and in p the weight decay
# p lr wd against the Adam step lr / bc1 m / denom (taken with m's term magnitudes, see util.adam_step_scale).
SUMSQ_TOL = 1.5e-6     # relative to the fp64 sum of squares; 3.8e-7 (447,074,880 elements, scalar path)
M_TOL = 1e-6           # |m - m_ref| / (b1 |m0| + (1 - b1) |clip g|); 2.4e-7
V_TOL = 1.5e-6         # |v - v_ref| / v_ref; 4.1e-7
P_ULP, P_REL = 2.0, 1e-6   # |dp - dp_ref| <= P_ULP ulp(p) + P_REL (|p lr wd| + |Adam step|); beyond 2 ulp: 2.8e-7
HP = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _call(name, *args):
    from medical_image_generation_b200 import _lib
    _lib.call(name, *[_ptr(a) if isinstance(a, torch.Tensor) else a for a in args],
              C.c_void_p(torch.cuda.current_stream().cuda_stream))


def _hp32(hp):
    return dict(lr=f32(hp["lr"]), betas=tuple(f32(b) for b in hp["betas"]), eps=f32(hp["eps"]),
                weight_decay=f32(hp["weight_decay"]))


def _abi_hp(hp):
    return (hp["lr"], hp["betas"][0], hp["betas"][1], hp["eps"], hp["weight_decay"])


def _note(what, value):
    print(f"measured {what}: {value:.3e}")


def _sumsq(g, out=None):
    out = torch.zeros(1, device=DEV) if out is None else out
    _call("mig_sumsq", g, out, torch.zeros(2048, device=DEV), g.numel())
    return out


def _step_ratios(before, g, after, step, hp, max_norm, chunk=1 << 24):
    """Worst error ratios (m, v, p) of one kernel step against the reference fed the kernel's fp32 state `before`
    (p, m, v) and the gradient g: each ratio is the error over its bar, so every ratio must be <= 1. Computed in chunks
    (fp64 temporaries of the config-3 region would be several GB). The clip coefficient is taken from the fp64 norm of
    the whole of g. Also returns the raw worst values for the notes next to the bars."""
    p0, m0, v0 = before
    p1, m1, v1 = after
    hp = _hp32(hp)
    total = math.sqrt(sum(float(c.double().pow(2).sum()) for c in g.split(chunk)))
    coef = min(max_norm / (total + 1e-6), 1.0) if max_norm else 1.0
    b1 = hp["betas"][0]
    worst = dict(m=0.0, v=0.0, p=0.0, m_raw=0.0, v_raw=0.0, p_rel=0.0)
    for s in range(0, g.numel(), chunk):
        sl = slice(s, s + chunk)
        (pr,), (mr,), (vr,), _, _ = clip_adamw_reference([p0[sl]], [g[sl].double() * coef], [m0[sl]], [v0[sl]], step,
                                                         max_norm=0, **hp)
        em = (m1[sl].double() - mr).abs()
        m_scale = b1 * m0[sl].double().abs() + (1 - b1) * (g[sl].double() * coef).abs()
        ev = (v1[sl].double() - vr).abs()
        pd = p0[sl].double()
        dp_ref = pr - pd
        p_scale = (pd * hp["lr"] * hp["weight_decay"]).abs() + adam_step_scale(m_scale, vr, step, lr=hp["lr"],
                                                                                betas=hp["betas"], eps=hp["eps"])
        ep = ((p1[sl].double() - pd) - dp_ref).abs()
        ulp = ulp32(p0[sl])
        rm = em / (M_TOL * m_scale).clamp_min(1e-300)
        rv = ev / (V_TOL * vr).clamp_min(1e-300)
        rp = ep / (P_ULP * ulp + P_REL * p_scale).clamp_min(1e-300)
        worst["m"] = max(worst["m"], float(rm.max()))
        worst["v"] = max(worst["v"], float(rv.max()))
        worst["p"] = max(worst["p"], float(rp.max()))
        worst["m_raw"] = max(worst["m_raw"], float((em / m_scale.clamp_min(1e-300)).max()))
        worst["v_raw"] = max(worst["v_raw"], float((ev / vr.clamp_min(1e-300)).max()))
        worst["p_rel"] = max(worst["p_rel"], float(((ep - P_ULP * ulp).clamp_min(0) / p_scale.clamp_min(1e-300)).max()))
    return worst


def _assert_step(before, g, after, step, hp, max_norm, what):
    w = _step_ratios(before, g, after, step, hp, max_norm)
    _note(f"{what} m err / term scale", w["m_raw"])
    _note(f"{what} v rel err", w["v_raw"])
    _note(f"{what} p err beyond {P_ULP} ulp / p term scale", w["p_rel"])
    assert w["m"] <= 1 and w["v"] <= 1 and w["p"] <= 1, (what, w)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the fp64 reference itself, against torch
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_norm", [1.0, 0.0])
def test_reference_matches_torch_adamw_fp64(max_norm):
    """The fp64 restatement against clip_grad_norm_ + torch.optim.AdamW run in float64 over several steps, with several
    parameters (the norm is global), gradient scales that switch the clip on and off, and weight decay."""
    gen = torch.Generator().manual_seed(7)
    shapes = [(13, 7), (29,), (3, 5, 4)]
    init = [torch.randn(s, generator=gen, dtype=torch.float64) for s in shapes]
    params = [torch.nn.Parameter(t.clone()) for t in init]
    opt = torch.optim.AdamW(params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2)
    p, m, v = [t.clone() for t in init], [torch.zeros_like(t) for t in init], [torch.zeros_like(t) for t in init]
    for step, scale in enumerate([3.0, 0.01, 0.5, 20.0, 1e-3], 1):
        grads = [torch.randn(s, generator=gen, dtype=torch.float64) * scale for s in shapes]
        for q, gr in zip(params, grads):
            q.grad = gr.clone()
        norm = torch.nn.utils.clip_grad_norm_(params, max_norm) if max_norm else None
        opt.step()
        p, m, v, total, _ = clip_adamw_reference(p, grads, m, v, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                                                 weight_decay=1e-2, max_norm=max_norm)
        if norm is not None:
            assert abs(float(total) - float(norm)) <= 1e-14 * float(norm)
        for i, q in enumerate(params):
            st = opt.state[q]
            for got, want in ((p[i], q.detach()), (m[i], st["exp_avg"]), (v[i], st["exp_avg_sq"])):
                assert torch.allclose(got, want, rtol=1e-12, atol=1e-15), (step, i)


@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_reference_matches_torch_on_nonfinite_gradients(bad):
    """clip_grad_norm_ + AdamW with a NaN gradient element: every parameter becomes NaN. With an inf: the clip
    coefficient is 0, the inf element becomes NaN (inf * 0) and the others only decay."""
    gen = torch.Generator().manual_seed(8)
    init = torch.randn(10, generator=gen, dtype=torch.float64)
    grad = torch.randn(10, generator=gen, dtype=torch.float64)
    grad[3] = float(bad)
    q = torch.nn.Parameter(init.clone())
    q.grad = grad.clone()
    opt = torch.optim.AdamW([q], lr=1e-3)
    torch.nn.utils.clip_grad_norm_([q], 1.0)
    opt.step()
    (p,), _, _, _, coef = clip_adamw_reference([init], [grad], [torch.zeros(10, dtype=torch.float64)],
                                               [torch.zeros(10, dtype=torch.float64)], 1, lr=1e-3, betas=(0.9, 0.999),
                                               eps=1e-8, weight_decay=1e-2, max_norm=1.0)
    if bad == "nan":
        assert torch.isnan(q.detach()).all() and torch.isnan(p).all() and math.isnan(float(coef))
    else:
        assert float(coef) == 0.0
        fin = torch.arange(10) != 3
        assert torch.isnan(q.detach()[3]) and torch.isnan(p[3])
        assert torch.equal(q.detach()[fin], init[fin] * (1 - 1e-3 * 1e-2))
        assert torch.allclose(p[fin], q.detach()[fin], rtol=1e-15, atol=0)


def test_config3_layout_matches_bench_unet():
    """The config-3 constants above, from the bench U-Net built on the meta device, with FlatAdamW's layout rules:
    parameters padded to 64 elements, the fp32-consumed ones (1-D, FP32_CONSUMED names) replicated, proj_attn in the
    unused tail, the sharded region rounded up to whole buckets of bucket_mb = 64 (bench.py's default) at 8 GPUs."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200.engine import FlatAdamW
    with torch.device("meta"):
        model = mig.DiffusionModelUNet(**bench.unet_kwargs(), compute_dtype=torch.bfloat16)
    pad = lambda k: (k + 63) // 64 * 64  # noqa: E731
    used = [(n, p) for n, p in model.named_parameters() if "proj_attn" not in n]
    repl = lambda n, p: p.ndim <= 1 or any(tag in n for tag in FlatAdamW.FP32_CONSUMED)  # noqa: E731
    shard_raw = sum(pad(p.numel()) for n, p in used if not repl(n, p))
    repl_numel = sum(pad(p.numel()) for n, p in used if repl(n, p))
    unit = 8 * 64
    bucket = max(unit, (int(64.0 * (1 << 20) / 4) + unit - 1) // unit * unit)
    nb = -(-shard_raw // bucket)
    assert (bucket, nb, nb * bucket, nb * bucket + repl_numel) == (C3_BUCKET, C3_NB, C3_SHARD, C3_USED)


# ------------------------------------------------------------------------------------------------------------------
# mig_sumsq
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 10007, (1 << 20) + 3, C3_USED])
def test_sumsq_matches_fp64(n, path):
    """Sum of squares against an fp64 sum; the scalar path runs from a base one float past an aligned address.
    Elements outside [base, base + n) are NaN, so a read past either end shows. Two calls are bit-identical."""
    off = 0 if path == "vector" else 1
    buf = torch.full((n + off + 8,), float("nan"), device=DEV)
    g = buf[off:off + n]
    gen = torch.Generator(device=DEV).manual_seed(n)
    g.copy_(torch.randn(n, device=DEV, generator=gen) * torch.exp(torch.randn(n, device=DEV, generator=gen)))
    a, b = _sumsq(g), _sumsq(g)
    want = sum(float(c.double().pow(2).sum()) for c in g.split(1 << 26))
    err = abs(float(a) - want) / want
    _note(f"sumsq n={n} {path} rel err", err)
    assert torch.equal(a, b)
    assert err <= SUMSQ_TOL, err


# ------------------------------------------------------------------------------------------------------------------
# mig_sumsq_strided: W ranks emulated on one device
# ------------------------------------------------------------------------------------------------------------------
# (W, bucket, nb): piece 4 with one bucket, piece 64 with three, W = 1 (piece == stride, contiguous), config 3
STRIDED = ([(w, 4 * w, 1) for w in (2, 4, 8)] + [(w, 64 * w, 3) for w in (2, 4, 8)] + [(1, 1000, 5)] +
           [(w, C3_BUCKET, C3_NB) for w in (2, 4, 8)])


def _owned(buf, world, bucket, nb, r):
    """Rank r's slices of the strided region at the front of `buf`, as an (nb, piece) view."""
    return buf[:nb * bucket].view(nb, world, bucket // world)[:, r]


def _not_owned_is_nan(buf, world, bucket, nb, r):
    """Every element of `buf` outside rank r's slices still holds the canonical NaN it was filled with."""
    bits = buf.view(torch.int16 if buf.dtype == torch.bfloat16 else torch.int32)
    nan = int(torch.tensor(float("nan"), dtype=buf.dtype).view(bits.dtype))
    v = bits[:nb * bucket].view(nb, world, bucket // world)
    others = [q for q in range(world) if q != r]
    return bool((v[:, others] == nan).all()) and bool((bits[nb * bucket:] == nan).all())


@gpu
@pytest.mark.parametrize("world,bucket,nb", STRIDED)
def test_sumsq_strided_per_rank(world, bucket, nb):
    piece = bucket // world
    region = nb * bucket
    gen = torch.Generator(device=DEV).manual_seed(world * 7 + nb)
    g = torch.randn(region, device=DEV, generator=gen)
    g *= torch.exp(torch.randn(region, device=DEV, generator=gen))
    total = 0.0
    for r in range(world):
        work = torch.full((region + 64,), float("nan"), device=DEV)
        _owned(work, world, bucket, nb, r).copy_(_owned(g, world, bucket, nb, r))
        out = torch.zeros(1, device=DEV)
        _call("mig_sumsq_strided", work[r * piece:], out, torch.zeros(2048, device=DEV), piece, bucket, nb)
        got = float(out)
        want = float(_owned(g, world, bucket, nb, r).double().pow(2).sum())
        assert math.isfinite(got), (r, got)
        _note(f"sumsq_strided W={world} bucket={bucket} rank {r} rel err", abs(got - want) / want)
        assert abs(got - want) <= SUMSQ_TOL * want, (r, got, want)
        total += got
    want = sum(float(c.double().pow(2).sum()) for c in g.split(1 << 26))
    assert abs(total - want) <= SUMSQ_TOL * want, (total, want)
    if bucket == C3_BUCKET:
        _note(f"sumsq_strided config 3 W={world} peak memory GB", torch.cuda.max_memory_allocated() / 1e9)


# ------------------------------------------------------------------------------------------------------------------
# mig_adamw_step
# ------------------------------------------------------------------------------------------------------------------
def _state(n, gen, fresh=False):
    p = torch.randn(n, device=DEV, generator=gen)
    if fresh:
        return p, torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    m = torch.randn(n, device=DEV, generator=gen) * 1e-2
    v = (torch.randn(n, device=DEV, generator=gen) * 1e-2) ** 2
    return p, m, v


def _run_adamw(bufs, n, off, soff, step, hp, max_norm, sumsq, step_device=None):
    """One mig_adamw_step on views at element `off` of the fp32 buffers and byte `soff` of the shadow buffer."""
    p, g, m, v, sh = bufs
    shadow = sh.view(torch.uint8)[soff:soff + 2 * n].view(torch.bfloat16)
    _call("mig_adamw_step", p[off:off + n], g[off:off + n], m[off:off + n], v[off:off + n], n, *_abi_hp(hp),
          0 if step_device is not None else step, sumsq if max_norm else None, max_norm, shadow, step_device)
    return shadow


ADAM_CASES = {                           # gradient scale per step (norm ~ scale * sqrt(n)), max_norm, weight decay
    "clip_inactive": ([1e-4], 1.0, 1e-2),
    "clip_active": ([1.0], 1.0, 1e-2),
    "no_clip": ([1.0], 0.0, 1e-2),
    "no_weight_decay": ([1.0], 1.0, 0.0),
    "six_steps": ([3.0, 1e-5, 0.1, 1e-4, 10.0, 1e-3], 1.0, 1e-2),
}


@gpu
@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("case", list(ADAM_CASES))
def test_adamw_step_one_step_against_fp64(case, path):
    """Each step against the fp64 reference from the kernel's own state; host and device step counters give bit-identical
    results; the bf16 shadow is exactly bf16(master); elements outside [base, base + n) are never written. The scalar
    path: n not a multiple of 4, the base one float past an aligned address, the shadow 2 bytes off."""
    scales, max_norm, wd = ADAM_CASES[case]
    hp = dict(HP, weight_decay=wd)
    n, off, soff = ((1 << 20), 0, 0) if path == "vector" else ((1 << 20) + 3, 1, 2)
    gen = torch.Generator(device=DEV).manual_seed(len(case) * 31 + off)
    total = n + off + 16
    bufs = [torch.full((total,), 1234.5, device=DEV) for _ in range(4)] + \
           [torch.full((total,), -7.0, device=DEV, dtype=torch.bfloat16)]
    p, g, m, v, _ = bufs
    for b, t in zip((p, m, v), _state(n, gen, fresh=len(scales) > 1)):
        b[off:off + n] = t
    first = 1 if len(scales) > 1 else 3
    step_dev = torch.zeros(1, dtype=torch.int32, device=DEV)
    for k, scale in enumerate(scales):
        step = first + k
        g[off:off + n] = torch.randn(n, device=DEV, generator=gen) * scale
        sumsq = _sumsq(g[off:off + n])
        before = [b[off:off + n].clone() for b in (p, m, v)]
        twin = [b.clone() for b in bufs]
        step_dev.fill_(step)
        shadow = _run_adamw(bufs, n, off, soff, step, hp, max_norm, sumsq)
        _run_adamw(twin, n, off, soff, step, hp, max_norm, sumsq, step_device=step_dev)
        for a, b in zip(bufs, twin):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), "host and device step counters differ"
        assert torch.equal(shadow, p[off:off + n].to(torch.bfloat16)), "shadow != bf16(master)"
        for b in (p, g, m, v):
            assert bool((b[:off] == 1234.5).all()) and bool((b[off + n:] == 1234.5).all()), "wrote outside [0, n)"
        sb = bufs[4].view(torch.uint8)
        fill = torch.full((total,), -7.0, dtype=torch.bfloat16, device=DEV).view(torch.uint8)
        assert torch.equal(sb[:soff], fill[:soff]) and torch.equal(sb[soff + 2 * n:], fill[soff + 2 * n:]), \
            "shadow written outside [0, n)"
        after = [b[off:off + n] for b in (p, m, v)]
        _assert_step(before, g[off:off + n], after, step, hp, max_norm, f"adamw {case} {path} step {step}")


@gpu
@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_adamw_nonfinite_gradient_matches_torch(bad):
    """A NaN gradient element: the norm is NaN and, as in torch, every parameter and moment becomes NaN (a clamp that
    turns the NaN coefficient into 1 would take an unclipped step instead). An inf: the clip coefficient is 0, the inf
    element becomes NaN and the finite ones only decay (first step, zero moments)."""
    n = 4096
    gen = torch.Generator(device=DEV).manual_seed(5)
    p, m, v = _state(n, gen, fresh=True)
    g = torch.randn(n, device=DEV, generator=gen)
    g[1000] = float(bad)
    p0 = p.clone()
    shadow = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    sumsq = _sumsq(g)
    _call("mig_adamw_step", p, g, m, v, n, *_abi_hp(HP), 1, sumsq, 1.0, shadow, None)
    q = torch.nn.Parameter(p0.cpu().clone())
    q.grad = g.cpu().clone()
    opt = torch.optim.AdamW([q], **HP)
    torch.nn.utils.clip_grad_norm_([q], 1.0)
    opt.step()
    if bad == "nan":
        assert torch.isnan(q.detach()).all()
        assert torch.isnan(p).all() and torch.isnan(m).all() and torch.isnan(v).all() and torch.isnan(shadow).all()
        return
    fin = torch.arange(n, device=DEV) != 1000
    assert torch.isnan(p[1000]) and torch.isnan(q.detach()[1000])
    assert bool((m[fin] == 0).all()) and bool((v[fin] == 0).all())
    decay = 1 - f32(HP["lr"]) * f32(HP["weight_decay"])
    assert float(((p[fin].double() - p0[fin].double() * decay).abs() / ulp32(p0[fin])).max()) <= P_ULP
    assert float(((p[fin].cpu() - q.detach()[fin.cpu()]).double().abs() / ulp32(p0[fin]).cpu()).max()) <= P_ULP


# ------------------------------------------------------------------------------------------------------------------
# mig_adamw_step_strided: W ranks emulated on one device
# ------------------------------------------------------------------------------------------------------------------
ADAMW_STRIDED = ([(w, 4 * w, 1) for w in (2, 4, 8)] + [(w, 64 * w, 3) for w in (2, 4, 8)] + [(1, 1000, 5)] +
                 [(8, C3_BUCKET, C3_NB)])


@gpu
@pytest.mark.parametrize("world,bucket,nb", ADAMW_STRIDED)
def test_adamw_step_strided_emulated_ranks(world, bucket, nb):
    """Rank r's call with every element it does not own NaN (p, g, m, v and the shadow): those elements keep their bits,
    the owned ones are finite, and the owned results of all W ranks together are bit-identical to ONE mig_adamw_step over
    the whole region with the same sumsq pointer and device step counter, which matches the fp64 reference."""
    piece, region = bucket // world, nb * bucket
    gen = torch.Generator(device=DEV).manual_seed(world + 3 * nb)
    p0, m0, v0 = _state(region, gen)
    g = torch.randn(region, device=DEV, generator=gen) * 10.0 / math.sqrt(region)   # norm ~10: the clip is active
    sumsq = _sumsq(g)
    step_dev = torch.full((1,), 4, dtype=torch.int32, device=DEV)
    whole = [t.clone() for t in (p0, m0, v0)] + [torch.empty(region, dtype=torch.bfloat16, device=DEV)]
    _call("mig_adamw_step", whole[0], g, whole[1], whole[2], region, *_abi_hp(HP), 0, sumsq, 1.0, whole[3], step_dev)
    merged = [torch.full_like(t, float("nan")) for t in whole]
    for r in range(world):
        bufs = [torch.full((region + 64,), float("nan"), device=DEV) for _ in range(4)] + \
               [torch.full((region + 64,), float("nan"), device=DEV, dtype=torch.bfloat16)]
        for b, src in zip(bufs, (p0, g, m0, v0)):
            _owned(b, world, bucket, nb, r).copy_(_owned(src, world, bucket, nb, r))
        p, gg, m, v, sh = (b[r * piece:] for b in bufs)
        _call("mig_adamw_step_strided", p, gg, m, v, piece, bucket, nb, *_abi_hp(HP), 0, sumsq, 1.0, sh, step_dev)
        for name, b in zip("pgmvs", bufs):
            assert _not_owned_is_nan(b, world, bucket, nb, r), f"rank {r} changed a {name} element it does not own"
            assert bool(torch.isfinite(_owned(b, world, bucket, nb, r)).all()), f"rank {r}: non-finite owned {name}"
        for dst, b in zip(merged, (bufs[0], bufs[2], bufs[3], bufs[4])):
            _owned(dst, world, bucket, nb, r).copy_(_owned(b, world, bucket, nb, r))
        del bufs, p, gg, m, v, sh
    for name, a, b in zip(("master", "m", "v", "shadow"), merged, whole):
        assert torch.equal(a, b), f"{name}: the ranks' strided steps differ from one step over the whole region"
    assert torch.equal(whole[3], whole[0].to(torch.bfloat16))
    _assert_step((p0, m0, v0), g, whole[:3], 4, HP, 1.0, f"adamw_strided W={world} bucket={bucket}")
    if bucket == C3_BUCKET:
        _note(f"adamw_strided config 3 W={world} peak memory GB", torch.cuda.max_memory_allocated() / 1e9)


@gpu
def test_strided_entry_points_reject_misaligned_layouts():
    """piece or stride not a multiple of 4 elements, or a base that is not 16-byte aligned, is refused on the host."""
    buf = torch.zeros(4096, device=DEV)
    sh = torch.zeros(4096, dtype=torch.bfloat16, device=DEV)
    out, parts = torch.zeros(1, device=DEV), torch.zeros(2048, device=DEV)
    step_dev = torch.ones(1, dtype=torch.int32, device=DEV)
    for piece, stride, base in ((6, 64, 0), (64, 66, 0), (64, 128, 1)):
        g = buf[base:]
        with pytest.raises(RuntimeError, match="aligned"):
            _call("mig_sumsq_strided", g, out, parts, piece, stride, 3)
        with pytest.raises(RuntimeError, match="aligned"):
            _call("mig_adamw_step_strided", g, g, g, g, piece, stride, 3, *_abi_hp(HP), 1, out, 1.0, sh, step_dev)
    shadow_off = sh.view(torch.uint8)[2:].view(torch.bfloat16)
    with pytest.raises(RuntimeError, match="aligned"):
        _call("mig_adamw_step_strided", buf, buf, buf, buf, 64, 128, 3, *_abi_hp(HP), 1, out, 1.0, shadow_off, step_dev)
    torch.cuda.synchronize()
    assert bool((buf == 0).all()) and bool((sh == 0).all())
