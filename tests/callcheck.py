"""Kernel-call checks for whole training and sampling steps at their real shapes (TEST CODE, not collected).

`_Recorder` wraps the module-level ops entry points the models and trainers call through `ops.`, keeps the inputs and
outputs of the first call of every distinct signature together with the gradient that reaches each output, and
collects the C entry points launched. `_check_forward` compares each recorded output with an fp32 reference of the same
operation on the same bf16 operands (TF32 off), per voxel and per channel as well as globally; scalar losses are compared
with fp64. `_check_backward` runs the production op once more on leaf clones with the recorded output gradient as probe,
against autograd of the fp32 reference. `_Report` collects every check of a test and prints the worst value of each kind.

Bars (worst value observed on a B200 in the comment beside each):
  * one bf16 rounding of the result is off by at most 2^-8 = 3.9e-3 relative per element, 1.7e-3 rms on normally
    distributed values;
  * fp32 results (weight, bias and norm-gain gradients, the fp32 time-embedding path) only reorder fp32 sums;
  * attention stores P (forward) and dS (backward) in bf16 before the second product.
"""
import types

import torch
import torch.nn.functional as F

from util import local_errors, local_failure, rel_err

BARS = {
    # bf16 outputs and input gradients; worst 2.41e-3 / 3.89e-3 / 2.85e-3 (folded upsample conv forward, conv_in dx)
    "bf16": dict(glob=5e-3, row=1e-2, col=1e-2),
    # fp32 outputs (wgrad, bias / gain / time-embedding gradients, fp32 linears); worst 2.4e-5 / 2.6e-5 / 2.7e-5
    "fp32": dict(glob=1e-4, row=5e-4, col=5e-4),
    # attention output and dq / dk / dv; worst 2.7e-3 / 4.8e-3 / 6.3e-3 (dqkv of the 6^3 flash block)
    "attn": dict(glob=1e-2, row=2e-2, col=2e-2),
}
GN_SUMS_BAR = 5e-5   # epilogue GroupNorm statistics; worst 4.7e-8 (sum y^2, relative), 7.4e-6 (sum y, see below)
# scalar losses (L1, KL) against fp64: fp32 partial sums over up to 1.8 M terms; worst 3.4e-8 (L1 over 2 x 96^3)
LOSS_CALL_BAR = 1e-6


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


def _kl_ref(mu, sigma):
    """0.5 sum(mu^2 + sigma^2 - log sigma^2 - 1) / batch (train_autoencoder.py:67-72)."""
    s2 = sigma * sigma
    return 0.5 * (mu * mu + s2 - torch.log(s2) - 1).sum() / mu.shape[0]


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

    OPS = ("conv_nd", "upsample_conv_nd", "group_norm", "linear", "temb_projections", "sdpa_qkv", "conv_transpose_nd",
           "vae_sigma", "vae_reparam", "l1_loss", "kl_loss")

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

    def _conv_transpose_nd(self, x, weight, bias=None, stride=1, padding=0, output_padding=0):
        y = self.real["conv_transpose_nd"](x, weight, bias, stride, padding, output_padding)
        nd = x.ndim - 2
        s, p, op = _tup(stride, nd), _tup(padding, nd), _tup(output_padding, nd)
        sig = ("convT", x.dtype, tuple(x.shape), tuple(weight.shape), s, p, op, bias is not None)
        self._keep(sig, [y], x=x, w=_kernel_weight(weight, x.dtype), bias=bias, stride=s, padding=p, output_padding=op)
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

    def _vae_sigma(self, logvar):
        sigma = self.real["vae_sigma"](logvar)
        self._keep(("sigma", logvar.dtype, tuple(logvar.shape)), [sigma], lv=logvar)
        return sigma

    def _vae_reparam(self, mu, sigma, eps):
        z = self.real["vae_reparam"](mu, sigma, eps)
        self._keep(("reparam", mu.dtype, tuple(mu.shape)), [z], mu=mu, sigma=sigma, eps=eps.to(mu.dtype))
        return z

    def _l1_loss(self, pred, target):
        # the kernel reads the target in the prediction's dtype
        out = self.real["l1_loss"](pred, target)
        cast = pred.dtype if pred.dtype in (torch.float32, torch.bfloat16) else torch.float32
        self._keep(("l1", pred.dtype, tuple(pred.shape)), [out], pred=pred, target=target.to(cast))
        return out

    def _kl_loss(self, z_mu, z_sigma):
        out = self.real["kl_loss"](z_mu, z_sigma)
        cast = z_mu.dtype if z_mu.dtype in (torch.float32, torch.bfloat16) else torch.float32
        self._keep(("kl", z_mu.dtype, tuple(z_mu.shape)), [out], mu=z_mu, sigma=z_sigma.to(cast))
        return out


# differentiable tensor inputs of each op, in the order `_run` and `_reference` take them
_DIFF = {"conv": ("x", "w", "bias", "chan_bias", "residual"), "upconv": ("x", "w", "bias"), "gn": ("x", "gamma", "beta"),
         "linear": ("x", "w", "bias"), "temb": ("x", "ws", "bs"), "sdpa_qkv": ("qkv",), "convT": ("x", "w", "bias"),
         "sigma": ("lv",), "reparam": ("mu", "sigma"), "l1": ("pred",), "kl": ("mu", "sigma")}
# ops whose output is a scalar loss: compared with an fp64 reference (the backward still with fp32 autograd)
_SCALAR = ("l1", "kl")


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
    if op == "convT":
        fn = F.conv_transpose3d if t["x"].ndim == 5 else F.conv_transpose2d
        return [fn(t["x"], t["w"], t["bias"], stride=rec["stride"], padding=rec["padding"],
                   output_padding=rec["output_padding"])]
    if op == "sigma":
        return [torch.exp(torch.clamp(t["lv"], -30.0, 20.0) / 2)]
    if op == "reparam":
        return [t["mu"] + rec["eps"].to(t["mu"].dtype) * t["sigma"]]
    if op == "l1":
        return [(t["pred"] - rec["target"].to(t["pred"].dtype)).abs().mean()]
    if op == "kl":
        return [_kl_ref(t["mu"], t["sigma"])]
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
    if op == "convT":
        return [real["conv_transpose_nd"](t["x"], t["w"], t["bias"], rec["stride"], rec["padding"], rec["output_padding"])]
    if op == "sigma":
        return [real["vae_sigma"](t["lv"])]
    if op == "reparam":
        return [real["vae_reparam"](t["mu"], t["sigma"], rec["eps"])]
    if op == "l1":
        return [real["l1_loss"](t["pred"], rec["target"])]
    if op == "kl":
        return [real["kl_loss"](t["mu"], t["sigma"])]
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
    dtype = torch.float64 if rec["op"] in _SCALAR else torch.float32

    def up(v):
        return [up(a) for a in v] if isinstance(v, list) else (None if v is None else v.to(dtype))

    with torch.no_grad():
        want = _reference(rec, {k: up(rec[k]) for k in _DIFF[rec["op"]]})
    for i, (got, w) in enumerate(zip(rec["outs"], want)):
        if rec["op"] in _SCALAR:
            rep.value("loss call", abs(float(got) - float(w)) / abs(float(w)), LOSS_CALL_BAR, f"fwd {_name(rec)}")
        else:
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


def _peak(rep, what):
    rep.worst[f"peak GB {what}"] = (torch.cuda.max_memory_allocated() / 1e9, "torch.cuda.max_memory_allocated")
