"""The benchmarked workloads, kernel call by kernel call, at their own shapes.

bench.py times one LDMTrainer step of the 441 M-parameter U-Net (BASELINE config 3: 256/512/768 channels, batch 8 of
3 x 24^3 latents, bf16, every dispatch policy on `auto`) and the sampling forward of config 4 (32/64/128 channels on
1 x 1 x 128 x 128 x 64, attention at L = 32768). Tile sizes, split-K, the persistent tile loop, the upsample fold, the
GroupNorm statistics in the conv epilogue and the attention routing are all chosen from the shapes, so a test at a
smaller shape runs other code. Here every call the model makes to the ops entry points is recorded during one real
step and compared with an fp32 reference of the same operation on the same bf16 operands (TF32 off), per voxel and
per channel as well as globally: an error confined to one TMA box, one halo plane or one channel tile fails.

Bars (worst value observed on a B200 in the comment beside each):
  * one bf16 rounding of the result is off by at most 2^-8 = 3.9e-3 relative per element, 1.7e-3 rms on normally
    distributed values;
  * fp32 results (weight, bias and norm-gain gradients, the fp32 time-embedding path) only reorder fp32 sums;
  * attention stores P (forward) and dS (backward) in bf16 before the second product.
"""
import math
import types

import pytest
import torch
import torch.nn.functional as F

from util import BF16_TOL, assert_close_local, graph_vs_eager, local_errors, local_failure, rel_err

DEV = "cuda"

BARS = {
    # bf16 outputs and input gradients; worst 2.41e-3 / 3.89e-3 / 2.85e-3 (folded upsample conv forward, conv_in dx)
    "bf16": dict(glob=5e-3, row=1e-2, col=1e-2),
    # fp32 outputs (wgrad, bias / gain / time-embedding gradients, fp32 linears); worst 2.4e-5 / 2.6e-5 / 2.7e-5
    "fp32": dict(glob=1e-4, row=5e-4, col=5e-4),
    # attention output and dq / dk / dv; worst 2.7e-3 / 4.8e-3 / 6.3e-3 (dqkv of the 6^3 flash block)
    "attn": dict(glob=1e-2, row=2e-2, col=2e-2),
}
GN_SUMS_BAR = 5e-5   # epilogue GroupNorm statistics; worst 4.7e-8 (sum y^2, relative), 7.4e-6 (sum y, see below)


@pytest.fixture
def no_tf32():
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


# ------------------------------------------------------------------------------------------------------------------
# the checker catches what rel_err misses (CPU)
# ------------------------------------------------------------------------------------------------------------------
def test_local_checker_catches_tile_faults():
    """On an 8 x 256 x 24^3 activation (level 0 of the benchmark): bf16 rounding noise passes; one 64-voxel box off by
    50 %, one channel off by 5 % and one boundary plane off by 10 % fail, and the message names the box / channel /
    plane -- while the global rel_err of all three stays under the 2e-2 bar the other parity tests use."""
    g = torch.Generator().manual_seed(0)
    want = torch.randn(8, 256, 24, 24, 24, generator=g)
    noise = want.to(torch.bfloat16).float()
    errs = assert_close_local(noise, want, what="bf16 rounding", **BARS["bf16"])
    assert errs["glob"] < 2e-3 and errs["row"] < 2.5e-3   # 1.66e-3 and 2.06e-3
    faults = {
        "box": (lambda t: t[5, :, 8:12, 4:8, 20:24].mul_(1.5), r"voxel \(n, \*spatial\) \(5, (8|9|10|11), [4-7], (2[0-3])\)"),
        "channel": (lambda t: t[:, 77].mul_(1.05), r"worst channel 77 "),
        "plane": (lambda t: t[3, :, :, :, 23].mul_(1.1), r"voxel \(n, \*spatial\) \(3, \d+, \d+, 23\)"),
    }
    for name, (inject, where) in faults.items():
        got = noise.clone()
        inject(got)
        assert rel_err(got, want) < BF16_TOL, name
        with pytest.raises(AssertionError, match=where):
            assert_close_local(got, want, what=name, **BARS["bf16"])


# ------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------
def _tup(v, n):
    return tuple(int(a) for a in v) if isinstance(v, (list, tuple)) else (int(v),) * n


def _nearest(x, factors):
    for ax, f in enumerate(factors):
        x = x.repeat_interleave(f, dim=2 + ax) if f != 1 else x
    return x


def _conv_ref(x, w, b, stride, padding, chan_bias=None, residual=None):
    nd = x.ndim - 2
    y = (F.conv3d if nd == 3 else F.conv2d)(x, w, b, stride=stride, padding=padding)
    if chan_bias is not None:
        y = y + chan_bias.reshape(*chan_bias.shape, *([1] * nd))
    if residual is not None:
        y = y + residual
    return y


def _attn_ref(q, k, v, heads, scale, rows=4096):
    """softmax(scale q k^T) v per head for (B, L, C) matrices, over blocks of query rows (differentiable)."""
    B, _, Cc = q.shape
    dh = Cc // heads

    def split(t):
        return t.reshape(B, t.shape[1], heads, dh).transpose(1, 2)

    outs = []
    for i in range(0, q.shape[1], rows):
        p = torch.softmax(split(q[:, i:i + rows]) @ split(k).transpose(-1, -2) * scale, dim=-1)
        outs.append((p @ split(v)).transpose(1, 2).reshape(B, -1, Cc))
    return torch.cat(outs, 1)


def _kernel_weight(w, dtype):
    """The filter the kernels read for compute dtype `dtype`: the optimiser's bf16 shadow, else the cached cast."""
    if w.dtype == dtype:
        return w.detach()
    shadow = getattr(w, "_mig_shadow", None)
    if shadow is not None:
        return shadow
    hit = w.__dict__.get("_mig_filter_cache", {}).get(dtype)
    return hit[1] if hit is not None else w.detach().to(dtype)


# ------------------------------------------------------------------------------------------------------------------
# recording the calls of one real step
# ------------------------------------------------------------------------------------------------------------------
def _clone(v):
    if isinstance(v, torch.Tensor):
        return v.detach().clone()
    if isinstance(v, list):
        return [_clone(t) for t in v]
    return v


class _Recorder:
    """Wraps the module-level ops entry points the model calls through `ops.`; keeps clones of the inputs (with the
    bf16 filters the kernels read) and outputs of the first call of every distinct signature, and the gradient that
    reaches each output in the backward pass. Also collects the C entry points launched while `on`."""

    OPS = ("conv_nd", "upsample_conv_nd", "group_norm", "linear", "temb_projections", "sdpa_qkv")

    def __init__(self, monkeypatch, ops):
        self.ops, self.calls, self.names, self.on = ops, {}, set(), True
        self.real = {n: getattr(ops, n) for n in self.OPS + ("call",)}
        real_call = self.real["call"]

        def call(name, *a):
            if self.on:
                self.names.add(name)
            return real_call(name, *a)

        monkeypatch.setattr(ops, "call", call)
        for n in self.OPS:
            monkeypatch.setattr(ops, n, getattr(self, "_" + n))

    def _keep(self, sig, outs, **inputs):
        if not self.on or sig in self.calls:
            return
        rec = dict(op=sig[0], sig=sig, outs=[_clone(o) for o in outs], dys=[None] * len(outs),
                   **{k: _clone(v) for k, v in inputs.items()})
        self.calls[sig] = rec
        for i, o in enumerate(outs):
            if isinstance(o, torch.Tensor) and o.requires_grad:
                o.register_hook(lambda g, i=i: rec["dys"].__setitem__(i, g.detach().clone()))

    def _conv_nd(self, x, weight, bias=None, stride=1, padding=0, chan_bias=None, residual=None, gn_groups=0):
        y = self.real["conv_nd"](x, weight, bias, stride, padding, chan_bias=chan_bias, residual=residual,
                                 gn_groups=gn_groups)
        nd = x.ndim - 2
        s, p = _tup(stride, nd), _tup(padding, nd)
        sums = getattr(y, "_mig_gn_sums", None)
        sig = ("conv", x.dtype, tuple(x.shape), tuple(weight.shape), s, p, bias is not None, chan_bias is not None,
               residual is not None, int(gn_groups or 0), sums is not None)
        self._keep(sig, [y], x=x, w=_kernel_weight(weight, x.dtype), bias=bias, chan_bias=chan_bias, residual=residual,
                   stride=s, padding=p, gn_groups=int(gn_groups or 0), sums=None if sums is None else sums[0])
        return y

    def _upsample_conv_nd(self, x, weight, bias, factors, padding):
        y = self.real["upsample_conv_nd"](x, weight, bias, factors, padding)
        nd = x.ndim - 2
        f, p = _tup(factors, nd), _tup(padding, nd)
        sig = ("upconv", x.dtype, tuple(x.shape), tuple(weight.shape), f, p, self.ops.upconv_usable(x, weight, f, p))
        self._keep(sig, [y], x=x, w=_kernel_weight(weight, x.dtype), bias=bias, factors=f, padding=p)
        return y

    def _group_norm(self, x, gamma, beta, groups, eps, silu=False, with_skip=False):
        out = self.real["group_norm"](x, gamma, beta, groups, eps, silu=silu, with_skip=with_skip)
        sig = ("gn", x.dtype, tuple(x.shape), int(groups), bool(silu), bool(with_skip),
               getattr(x, "_mig_gn_sums", None) is not None)
        self._keep(sig, list(out) if with_skip else [out], x=x, gamma=gamma, beta=beta, groups=int(groups),
                   eps=float(eps), silu=bool(silu), with_skip=bool(with_skip))
        return out

    def _linear(self, x, weight, bias=None):
        y = self.real["linear"](x, weight, bias)
        sig = ("linear", x.dtype, tuple(x.shape), tuple(weight.shape), weight.dtype, bias is not None)
        self._keep(sig, [y], x=x, w=_kernel_weight(weight, x.dtype), bias=bias)
        return y

    def _temb_projections(self, x, linears):
        outs = self.real["temb_projections"](x, linears)
        if outs is not None:
            sig = ("temb", tuple(x.shape), tuple(tuple(m.weight.shape) for m in linears))
            self._keep(sig, outs, x=x, ws=[m.weight for m in linears], bs=[m.bias for m in linears])
        return outs

    def _sdpa_qkv(self, qkv, heads, scale_, order=("q", "k", "v")):
        o = self.real["sdpa_qkv"](qkv, heads, scale_, order)
        sig = ("sdpa_qkv", qkv.dtype, tuple(qkv.shape), int(heads), tuple(order), bool(o.requires_grad))
        self._keep(sig, [o], qkv=qkv, heads=int(heads), scale=float(scale_), order=tuple(order))
        return o


# differentiable tensor inputs of each op, in the order `_run` and `_reference` take them
_DIFF = {"conv": ("x", "w", "bias", "chan_bias", "residual"), "upconv": ("x", "w", "bias"), "gn": ("x", "gamma", "beta"),
         "linear": ("x", "w", "bias"), "temb": ("x", "ws", "bs"), "sdpa_qkv": ("qkv",)}


def _reference(rec, t):
    """fp32 reference outputs of a recorded call from the tensors `t` (name -> tensor or list of tensors)."""
    op = rec["op"]
    if op == "conv":
        return [_conv_ref(t["x"], t["w"], t["bias"], rec["stride"], rec["padding"], t["chan_bias"], t["residual"])]
    if op == "upconv":
        return [_conv_ref(_nearest(t["x"], rec["factors"]), t["w"], t["bias"], 1, rec["padding"])]
    if op == "gn":
        y = F.group_norm(t["x"], rec["groups"], t["gamma"], t["beta"], rec["eps"])
        y = F.silu(y) if rec["silu"] else y
        return [y, t["x"]] if rec["with_skip"] else [y]
    if op == "linear":
        return [F.linear(t["x"], t["w"], t["bias"])]
    if op == "temb":
        return [F.linear(t["x"], w, b) for w, b in zip(t["ws"], t["bs"])]
    qkv = t["qkv"]
    Cc = qkv.shape[-1] // 3
    sl = {n: qkv[..., i * Cc:(i + 1) * Cc] for i, n in enumerate(rec["order"])}
    return [_attn_ref(sl["q"], sl["k"], sl["v"], rec["heads"], rec["scale"])]


def _run(real, rec, t):
    """The recorded call again, through the production op, on the tensors `t`."""
    op = rec["op"]
    if op == "conv":
        return [real["conv_nd"](t["x"], t["w"], t["bias"], rec["stride"], rec["padding"], chan_bias=t["chan_bias"],
                                residual=t["residual"], gn_groups=rec["gn_groups"])]
    if op == "upconv":
        return [real["upsample_conv_nd"](t["x"], t["w"], t["bias"], rec["factors"], rec["padding"])]
    if op == "gn":
        out = real["group_norm"](t["x"], t["gamma"], t["beta"], rec["groups"], rec["eps"], silu=rec["silu"],
                                 with_skip=rec["with_skip"])
        return list(out) if rec["with_skip"] else [out]
    if op == "linear":
        return [real["linear"](t["x"], t["w"], t["bias"])]
    if op == "temb":
        return real["temb_projections"](t["x"], [types.SimpleNamespace(weight=w, bias=b) for w, b in zip(t["ws"], t["bs"])])
    return [real["sdpa_qkv"](t["qkv"], rec["heads"], rec["scale"], rec["order"])]


def _leaves(rec, dtype=None):
    """Fresh leaf tensors (requires_grad) for the differentiable inputs; `dtype` None keeps the kernels' dtypes, except
    that filters become fp32 leaves holding the bf16 values (the op casts them back exactly, like a master weight)."""
    def leaf(v, as_filter=False):
        if v is None:
            return None
        v = v.detach().clone()
        v = v.to(dtype) if dtype is not None else (v.float() if as_filter else v)
        return v.requires_grad_(True)

    out = {}
    for k in _DIFF[rec["op"]]:
        v = rec[k]
        out[k] = [leaf(a, k == "ws") for a in v] if isinstance(v, list) else leaf(v, k == "w")
    return out


def _flat(t):
    for k, v in t.items():
        for i, a in enumerate(v if isinstance(v, list) else [v]):
            if a is not None:
                yield (f"{k}[{i}]" if isinstance(v, list) else k), a


def _nc(t):
    """(N, C, *spatial) view for the local checker: token matrices (B, L, C) become (B, C, L)."""
    return t.transpose(1, 2) if t.ndim == 3 else t


class _Report:
    """Collects every check of a test so one run reports all of them, and the worst value of each kind."""

    def __init__(self, title):
        self.title, self.failures, self.worst = title, [], {}

    def local(self, kind, got, want, what):
        errs = local_errors(_nc(got), _nc(want))
        msg = local_failure(errs, what=what, **BARS[kind])
        if msg:
            self.failures.append(msg)
        w = self.worst.setdefault(kind, {})
        for key in ("glob", "row", "col"):
            if errs[key] >= w.get(key, (-1.0, ""))[0]:
                w[key] = (errs[key], what)

    def value(self, kind, err, bar, what):
        if not err <= bar:
            self.failures.append(f"{what}: {err:.3e} (bar {bar:.1e})")
        if err >= self.worst.get(kind, (-1.0, ""))[0]:
            self.worst[kind] = (err, what)

    def require(self, ok, what):
        if not ok:
            self.failures.append(what)

    def finish(self):
        lines = [f"[{self.title}] worst observed:"]
        for kind, w in sorted(self.worst.items()):
            if isinstance(w, dict):
                lines += [f"  {kind:6s} {key:4s} {v:.3e}  {what}" for key, (v, what) in sorted(w.items())]
            else:
                lines.append(f"  {kind:16s} {w[0]:.3e}  {w[1]}")
        print("\n".join(lines))
        assert not self.failures, f"{len(self.failures)} check(s) failed:\n" + "\n".join(self.failures[:40])


def _name(rec):
    sig = rec["sig"]
    return f"{sig[0]} {' '.join(str(s) for s in sig[1:])}"


def _kind(rec, t):
    if rec["op"] == "sdpa_qkv":
        return "attn"
    return "bf16" if t.dtype == torch.bfloat16 else "fp32"


def _check_forward(rep, rec):
    """The output recorded in the model run against the fp32 reference built from the recorded inputs."""
    def f32(v):
        return [f32(a) for a in v] if isinstance(v, list) else (None if v is None else v.float())

    with torch.no_grad():
        want = _reference(rec, {k: f32(rec[k]) for k in _DIFF[rec["op"]]})
    for i, (got, w) in enumerate(zip(rec["outs"], want)):
        rep.local(_kind(rec, got), got, w, f"fwd {_name(rec)} out{i}")
    if rec["op"] == "conv" and rec["sums"] is not None:
        # the GroupNorm statistics the epilogue accumulated, (sum y, sum y^2) per (sample, group) of the bf16 output
        y = rec["outs"][0]
        N, Cout, G = y.shape[0], y.shape[1], rec["gn_groups"]
        yg = y.double().reshape(N, G, Cout // G, -1)
        s1, s2 = yg.sum(dim=(2, 3)), (yg * yg).sum(dim=(2, 3))
        rep.value("gn_sums_sq", rel_err(rec["sums"][..., 1], s2), GN_SUMS_BAR, f"epilogue sum y^2 {_name(rec)}")
        err1 = float((rec["sums"][..., 0] - s1).abs().max() / s2.sqrt().max())
        rep.value("gn_sums", err1, GN_SUMS_BAR, f"epilogue sum y {_name(rec)} (abs / sqrt(max sum y^2))")


def _check_backward(rep, real, rec):
    """The production op once more on plain leaf clones with the recorded output gradients as probes, against autograd
    of the fp32 reference. (Plain leaves: the trainer's parameters accumulate into `main_grad` instead.)"""
    pairs = [(i, d) for i, d in enumerate(rec["dys"]) if d is not None]
    if not pairs:
        return
    kern, ref = _leaves(rec), _leaves(rec, torch.float32)
    outs = _run(real, rec, kern)
    torch.autograd.backward([outs[i] for i, _ in pairs], [d for _, d in pairs])
    want = _reference(rec, ref)
    torch.autograd.backward([want[i] for i, _ in pairs], [d.float() for _, d in pairs])
    for (name, a), (_, b) in zip(_flat(kern), _flat(ref)):
        if b.grad is None:
            continue
        rep.require(a.grad is not None, f"bwd {_name(rec)} d{name}: no gradient")
        if a.grad is not None:
            rep.local(_kind(rec, a.grad), a.grad, b.grad, f"bwd {_name(rec)} d{name}")


# ------------------------------------------------------------------------------------------------------------------
# the benchmark's models
# ------------------------------------------------------------------------------------------------------------------
def _bench_trainer(cuda_graph=True):
    """Model and trainer exactly as bench.run_b200 builds them."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import LDMTrainer
    torch.manual_seed(0)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.unet_kwargs(), compute_dtype=torch.bfloat16))
    model = model.to(DEV).train()
    sched = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    tr = LDMTrainer(model, sched, lr=2e-5, grad_clip_max_norm=1.0, cuda_graph=cuda_graph, bucket_mb=64.0,
                    graph_warmup_steps=2, shard_optimizer=None)
    return model, tr


def _bench_batch(seed, batch=8):
    import bench
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn((batch, *bench.LATENT), generator=g)
    noise = torch.randn(x0.shape, generator=g)
    t = torch.randint(0, 1000, (batch,), generator=g)
    return x0.to(DEV), noise.to(DEV), t.to(DEV)


@pytest.fixture(scope="module")
def bench_trainer():
    model, tr = _bench_trainer()
    yield model, tr
    tr.opt.close()
    del model, tr
    torch.cuda.empty_cache()


def _peak(rep, what):
    rep.worst[f"peak GB {what}"] = (torch.cuda.max_memory_allocated() / 1e9, "torch.cuda.max_memory_allocated")


# C entry points one eager training step launches through ops (bench shape, defaults; recorded on a B200): the upsample
# fold at 12^3 -> 24^3 (mig_upconv_*, mig_class_interleave), the unfolded nearest upsample + conv at 6^3 -> 12^3 (too
# few tiles to fold), the unfused attention chain at 12^3 (d = 512: mig_gemm_strided, mig_softmax_fwd,
# mig_softmax_bwd_narrow), flash at 6^3 (d = 768, L = 216) and the GroupNorm statistics in the conv epilogue
# (mig_conv_fwd_stats, mig_groupnorm_apply). A routing change that moves the benchmark onto another path fails here:
# make sure the new path is among the calls checked in this file, then update the list.
TRAIN_STEP_CALLS = sorted([
    "mig_add", "mig_class_interleave", "mig_colsum", "mig_concat_channels", "mig_conv_dgrad", "mig_conv_fwd",
    "mig_conv_fwd_stats", "mig_conv_wgrad", "mig_flash_attention_bwd", "mig_flash_attention_fwd_ld",
    "mig_gemm_strided", "mig_groupnorm_apply", "mig_groupnorm_bwd", "mig_groupnorm_fwd", "mig_mse_bwd", "mig_mse_fwd",
    "mig_nchw_to_nhwc", "mig_nhwc_to_nchw", "mig_silu_bwd", "mig_silu_fwd", "mig_softmax_bwd_narrow",
    "mig_softmax_fwd", "mig_split_channels", "mig_temb_proj_all_bwd", "mig_temb_proj_all_fwd", "mig_timestep_embedding",
    "mig_upconv_fold_filter", "mig_upconv_fwd", "mig_upconv_unfold_wgrad", "mig_upsample_nearest_bwd",
    "mig_upsample_nearest_fwd",
])

# ... and of one config-4 sampling forward: both upsample convs folded, flash at L = 32768, the filters cast to bf16
# once (mig_cast: no optimiser keeps a shadow), the one-channel input already channels-last.
SAMPLING_CALLS = sorted([
    "mig_add", "mig_cast", "mig_concat_channels", "mig_conv_fwd", "mig_conv_fwd_stats", "mig_flash_attention_fwd_ld",
    "mig_groupnorm_apply", "mig_groupnorm_fwd", "mig_nhwc_to_nchw", "mig_silu_fwd", "mig_temb_proj_all_fwd",
    "mig_timestep_embedding", "mig_upconv_fold_filter", "mig_upconv_fwd",
])


@pytest.mark.gpu
def test_training_step_calls_at_bench_shape(bench_trainer, monkeypatch, no_tf32):
    """Every distinct ops call of one eager LDMTrainer step at the benchmark shape: forward in place, backward
    standalone, plus the epilogue GroupNorm statistics, the bf16 shadow and the C entry points the step used."""
    from medical_image_generation_b200 import ops
    model, tr = bench_trainer
    torch.cuda.reset_peak_memory_stats()
    rep = _Report("training step, BASELINE config 3")
    recorder = _Recorder(monkeypatch, ops)
    x0, noise, t = _bench_batch(1000)
    tr._eager_step(x0, noise, t)
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(TRAIN_STEP_CALLS), f"entry points: {sorted(recorder.names)} (expected "
                f"{TRAIN_STEP_CALLS}; missing {sorted(set(TRAIN_STEP_CALLS) - recorder.names)}, new "
                f"{sorted(recorder.names - set(TRAIN_STEP_CALLS))})")
    # the bf16 filters every tensor-core kernel reads are the round-to-nearest of the fp32 masters, bit for bit
    rep.require(torch.equal(tr.opt.shadow, tr.opt.master.to(torch.bfloat16)), "bf16 shadow != bf16(master)")
    ops_seen = {}
    for rec in recorder.calls.values():
        ops_seen[rec["op"]] = ops_seen.get(rec["op"], 0) + 1
        _check_forward(rep, rec)
        _check_backward(rep, recorder.real, rec)
    rep.require({"conv", "upconv", "gn", "linear", "temb", "sdpa_qkv"} <= set(ops_seen), f"ops recorded: {ops_seen}")
    rep.require(any(r["op"] == "conv" and r["sums"] is not None for r in recorder.calls.values()),
                "no conv delivered epilogue GroupNorm statistics")
    rep.require(any(r["op"] == "upconv" and r["sig"][-1] for r in recorder.calls.values()), "the upsample fold did not run")
    print(f"distinct calls checked: {ops_seen}")
    _peak(rep, "training calls")
    rep.finish()


@pytest.mark.gpu
def test_sampling_forward_calls_at_bench_shape(monkeypatch, no_tf32):
    """Every distinct ops call of one config-4 sampling forward (1 x 1 x 128 x 128 x 64, no_grad): the 32-channel
    halo kernels at a million voxels, the narrow tiles with epilogue statistics and flash attention at L = 32768."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import ops
    torch.cuda.reset_peak_memory_stats()
    torch.manual_seed(7)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.SAMPLING_CFG, compute_dtype=torch.bfloat16))
    model = model.to(DEV).eval()
    x = torch.randn((1, *bench.VOLUME), generator=torch.Generator().manual_seed(42)).to(DEV)
    rep = _Report("sampling forward, BASELINE config 4")
    recorder = _Recorder(monkeypatch, ops)
    with torch.no_grad():
        model(x, torch.tensor([500], device=DEV))
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(SAMPLING_CALLS), f"entry points: {sorted(recorder.names)} (expected {SAMPLING_CALLS})")
    attn = [r for r in recorder.calls.values() if r["op"] == "sdpa_qkv"]
    rep.require([r["qkv"].shape[1] for r in attn] == [32768], f"attention lengths {[r['qkv'].shape for r in attn]}")
    for rec in recorder.calls.values():
        _check_forward(rep, rec)
    _peak(rep, "sampling calls")
    rep.finish()


# ------------------------------------------------------------------------------------------------------------------
# attention at the lengths the benchmarks use
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C", [(1, 8192, 128), (1, 32768, 128)])
def test_flash_attention_at_sampling_lengths(B, L, C, monkeypatch, no_tf32):
    """Fused forward and backward at L = 8192 and 32768 (64 / 256 KV blocks per query tile), checked per query row."""
    from medical_image_generation_b200 import ops
    g = torch.Generator().manual_seed(L)
    q, k, v, dO = (torch.randn(B, L, C, generator=g).to(DEV, torch.bfloat16) for _ in range(4))
    scale = 1 / math.sqrt(C)
    seen = []
    real = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.append(name), real(name, *a))[1])
    qd, kd, vd = (t.clone().requires_grad_(True) for t in (q, k, v))
    out = ops.sdpa(qd, kd, vd, 1, scale)
    out.backward(dO)
    monkeypatch.setattr(ops, "call", real)
    rep = _Report(f"flash attention B={B} L={L} C={C}")
    rep.require(seen == ["mig_flash_attention_fwd_ld", "mig_flash_attention_bwd"], f"calls {seen}")
    qr, kr, vr = (t.float().requires_grad_(True) for t in (q, k, v))
    want = _attn_ref(qr, kr, vr, 1, scale)
    want.backward(dO.float())
    for name, got, ref in (("out", out, want), ("dq", qd.grad, qr.grad), ("dk", kd.grad, kr.grad), ("dv", vd.grad, vr.grad)):
        rep.local("attn", got, ref, f"flash L={L} {name}")
    rep.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C,path", [(8, 1728, 512, "unfused"), (8, 216, 768, "flash")])
def test_sdpa_qkv_routing_at_training_shapes(B, L, C, path, monkeypatch, no_tf32):
    """The two attention blocks of the training step in `auto`: d = 512 at L = 1728 takes the unfused GEMM + softmax
    chain (row stride 3C, dS narrowed to bf16), d = 768 at L = 216 the fused kernels; order as the flat optimiser lays
    out the projections."""
    from medical_image_generation_b200 import ops
    order = ("v", "k", "q")
    g = torch.Generator().manual_seed(L + C)
    qkv = torch.randn(B, L, 3 * C, generator=g).to(DEV, torch.bfloat16)
    dO = torch.randn(B, L, C, generator=g).to(DEV, torch.bfloat16)
    scale = 1 / math.sqrt(C)
    seen = set()
    real = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.add(name), real(name, *a))[1])
    qd = qkv.clone().requires_grad_(True)
    out = ops.sdpa_qkv(qd, 1, scale, order)
    out.backward(dO)
    monkeypatch.setattr(ops, "call", real)
    expected = ({"mig_gemm_strided", "mig_softmax_fwd", "mig_softmax_bwd_narrow"} if path == "unfused" else
                {"mig_flash_attention_fwd_ld", "mig_flash_attention_bwd", "mig_concat_channels"})
    rep = _Report(f"sdpa_qkv B={B} L={L} C={C}")
    rep.require(seen == expected, f"calls {sorted(seen)}, expected {sorted(expected)}")
    qr = qkv.float().requires_grad_(True)
    sl = {n: qr[..., i * C:(i + 1) * C] for i, n in enumerate(order)}
    want = _attn_ref(sl["q"], sl["k"], sl["v"], 1, scale)
    want.backward(dO.float())
    rep.local("attn", out, want, f"sdpa_qkv {path} out")
    rep.local("attn", qd.grad, qr.grad, f"sdpa_qkv {path} dqkv")
    rep.finish()


@pytest.mark.gpu
def test_fp32_reference_matches_fp64(no_tf32):
    """The references above run in fp32 on the GPU with TF32 off; on bf16 operands they agree with fp64 on the CPU."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 64, 6, 6, 6, generator=g).bfloat16().float()
    w = (torch.randn(96, 64, 3, 3, 3, generator=g) / 40).bfloat16().float()
    b, cb = torch.randn(96, generator=g), torch.randn(2, 96, generator=g)
    want = _conv_ref(x.double(), w.double(), b.double(), (1, 1, 1), (1, 1, 1), cb.double())
    got = _conv_ref(x.to(DEV), w.to(DEV), b.to(DEV), (1, 1, 1), (1, 1, 1), cb.to(DEV))
    assert rel_err(got, want) < 1e-6
    gn = F.silu(F.group_norm(x.to(DEV), 32, b[:64].to(DEV), cb[0, :64].to(DEV), 1e-6))
    assert rel_err(gn, F.silu(F.group_norm(x.double(), 32, b[:64].double(), cb[0, :64].double(), 1e-6))) < 1e-6
    q, k, v = (torch.randn(2, 216, 256, generator=g).bfloat16().float() for _ in range(3))
    got = _attn_ref(q.to(DEV), k.to(DEV), v.to(DEV), 2, 1 / 16, rows=100)
    assert rel_err(got, _attn_ref(q.double(), k.double(), v.double(), 2, 1 / 16)) < 1e-6


# ------------------------------------------------------------------------------------------------------------------
# the whole step against the oracle, and the graph replay against eager steps
# ------------------------------------------------------------------------------------------------------------------
# whole step against the oracle (the golden model tests use 2e-2 output, 8e-2 gradient)
OUT_BAR = 1e-2       # worst 3.7e-3
GRAD_BAR = 6e-2      # worst 3.1e-2 (up_blocks.1.attentions.1.to_q.bias)
LOSS_BAR = 5e-3      # worst 5.2e-4
NORM_BAR = 5e-3      # worst 6.4e-4

# graphed vs eager steps on the same inputs: GroupNorm / split-K atomics reorder fp32 sums between the two runs
GRAPH_LOSS_BAR = 2e-3    # worst 1.3e-4
GRAPH_NORM_BAR = 5e-3    # worst 8.1e-4
GRAPH_DRIFT_BAR = 0.2    # worst 3.7e-2; a stale input, noise or shadow gives about 1


@pytest.mark.gpu
def test_training_step_matches_oracle_at_bench_shape(bench_trainer, monkeypatch, no_tf32):
    """One production step (batch 8) and the fp32 oracle (plain torch, pinned to the reference goldens) on the same
    weights and batch: loss, U-Net output, every parameter's full gradient and the global gradient norm."""
    import bench
    from oracle import torch_oracle as O
    model, tr = bench_trainer
    torch.cuda.reset_peak_memory_stats()
    cfg = bench.unet_kwargs()
    params = {k: v.detach().float().contiguous().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    x0, noise, t = _bench_batch(2000)
    got = {}
    hook = model.register_forward_hook(lambda m, a, kw, out: got.update(x=kw["x"].detach().clone(), out=out.detach().clone()),
                                       with_kwargs=True)
    try:
        loss = float(tr._eager_step(x0, noise, t).detach())
    finally:
        hook.remove()
    real_temb = O.timestep_embedding    # (builds its frequency table on the CPU)
    monkeypatch.setattr(O, "timestep_embedding", lambda ts, dim, max_period=10000: real_temb(ts.cpu(), dim, max_period).to(ts.device))
    pred = O.unet_forward(params, cfg, got["x"], t)
    ref_loss = F.mse_loss(pred, noise)
    ref_loss.backward()
    rep = _Report("training step vs oracle, BASELINE config 3")
    rep.value("loss", abs(loss - float(ref_loss)) / float(ref_loss), LOSS_BAR, "loss")
    rep.value("output", rel_err(got["out"], pred), OUT_BAR, "U-Net output (rel_err)")
    e = local_errors(got["out"], pred)
    print(f"U-Net output: per-voxel {e['row']:.3e} at {e['row_at']}, per-channel {e['col']:.3e}")
    named = dict(model.named_parameters())
    sq = 0.0
    for k, p in named.items():
        ref = params[k].grad
        if ref is None:
            rep.require("proj_attn" in k, f"oracle gives no gradient for {k}")
            continue
        sq += float(ref.double().pow(2).sum())
        if k.endswith("to_k.bias"):
            continue    # exactly zero mathematically (softmax is shift invariant): noise on both sides
        rep.value("param grad", rel_err(p.main_grad, ref, floor=1e-12), GRAD_BAR, k)
    rep.value("grad_norm", abs(float(tr.opt.grad_norm()) - sq ** 0.5) / sq ** 0.5, NORM_BAR, "opt.grad_norm()")
    _peak(rep, "oracle step")
    rep.finish()


@pytest.mark.gpu
def test_graph_replay_matches_eager_at_bench_shape():
    """Capture and three replays of the benchmarked CUDA-graph step against eager steps of a second trainer fed the
    same batch, noise and timesteps: a replay that reads a stale input, noise or shadow weights moves the masters
    elsewhere (drift ratio near 1)."""
    torch.cuda.reset_peak_memory_stats()
    model_a, tr_a = _bench_trainer(cuda_graph=True)
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import LDMTrainer
    model_b = mig.DiffusionModelUNet(**bench.unet_kwargs(), compute_dtype=torch.bfloat16)
    model_b.load_state_dict(model_a.state_dict())
    tr_b = LDMTrainer(model_b.to(DEV).train(), mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS), lr=2e-5,
                      grad_clip_max_norm=1.0)
    batches = [_bench_batch(3000 + i)[0] for i in range(6)]
    rows, noises, drift = graph_vs_eager(tr_a, tr_b, batches)
    rep = _Report("graph replay vs eager, BASELINE config 3")
    rep.require(tr_a._graph is not None and int(tr_a.opt.step_dev) == 6, "capture did not happen")
    rep.require(not any(torch.equal(noises[i], noises[i + 1]) for i in range(2, 5)), "replays drew the same noise")
    for i, (la, lb, ga, gb) in enumerate(rows):
        rep.value("loss", abs(la - lb) / abs(lb), GRAPH_LOSS_BAR, f"step {i} loss {la:.5f} vs {lb:.5f}")
        rep.value("grad_norm", abs(ga - gb) / gb, GRAPH_NORM_BAR, f"step {i} grad norm {ga:.5f} vs {gb:.5f}")
    rep.value("master drift", drift, GRAPH_DRIFT_BAR, "||master_A - master_B|| / ||master_A - master_0||")
    _peak(rep, "two trainers")
    tr_a.opt.close()
    tr_b.opt.close()
    del tr_a, tr_b, model_a, model_b
    torch.cuda.empty_cache()
    rep.finish()
