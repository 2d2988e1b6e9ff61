"""Autograd-aware operators over the C ABI (libmedimgen_b200.so).

Every function here launches hand-written sm_100a kernels through `_lib.call`; torch supplies only
device memory, the current CUDA stream and the autograd tape. Activations are logical
(N, C, *spatial) tensors in channels-last memory (NDHWC / NHWC), conv filters are logical
(Cout, Cin, *k) tensors in channels-last memory ([Cout][taps][Cin]) -- exactly the layouts the
kernels consume, so no repacking happens on the hot path.

Reference call sites are cited per operator (unet:N = medimgen/diffusion_model_unet_with_strides.py:N,
ae:N = medimgen/autoencoderkl_with_strides.py:N).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional, Sequence

import torch
from torch.autograd import Function

from . import _lib
from ._lib import BF16, F32, call

_ENGINE = _lib.ENGINE_AUTO


def set_engine(engine: int) -> None:
    """0 = auto (tcgen05 where eligible), 1 = force the SIMT family, 2 = require tcgen05."""
    global _ENGINE
    _ENGINE = engine


def get_engine() -> int:
    return _ENGINE


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {t.dtype}: the B200 path computes in float32 or bfloat16")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensor is on {t.device}; medical_image_generation_b200 runs on CUDA (sm_100a) "
                           "only and has no CPU path")


_workspaces: dict = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only scratch buffer per (device, stream): kernels on one stream are serialised, so reuse is safe."""
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _mf(ndim: int):
    return {4: torch.channels_last, 5: torch.channels_last_3d}.get(ndim, torch.contiguous_format)


def _is_cl(t: torch.Tensor) -> bool:
    return t.is_contiguous(memory_format=_mf(t.ndim)) if t.ndim in (4, 5) else t.is_contiguous()


def empty_cl(shape, dtype, device) -> torch.Tensor:
    return torch.empty(tuple(shape), dtype=dtype, device=device, memory_format=_mf(len(shape)))


def _sp3(spatial: Sequence[int]) -> tuple:
    s = tuple(int(v) for v in spatial)
    return (1,) * (3 - len(s)) + s


# ----------------------------------------------------------------------------------------------
# layout / dtype at the module boundary
# ----------------------------------------------------------------------------------------------
def _relayout(x: torch.Tensor, dtype: torch.dtype, to_cl: bool) -> torch.Tensor:
    N, Cc = x.shape[0], x.shape[1]
    S = x.numel() // max(N * Cc, 1)
    if to_cl:
        y = empty_cl(x.shape, dtype, x.device)
        call("mig_nchw_to_nhwc", _dt(x), _dt(y), _ptr(x), _ptr(y), N, Cc, S, _stream())
    else:
        y = torch.empty(x.shape, dtype=dtype, device=x.device)
        call("mig_nhwc_to_nchw", _dt(x), _dt(y), _ptr(x), _ptr(y), N, Cc, S, _stream())
    return y


class _ToChannelsLast(Function):
    @staticmethod
    def forward(ctx, x, dtype):
        ctx.src_dtype = x.dtype
        ctx.was_cl = _is_cl(x)
        if ctx.was_cl:
            if x.dtype == dtype:
                return x.view_as(x)
            y = empty_cl(x.shape, dtype, x.device)
            call("mig_cast", _dt(x), _dt(y), _ptr(x), _ptr(y), x.numel(), _stream())
            return y
        return _relayout(x.contiguous(), dtype, True)

    @staticmethod
    def backward(ctx, dy):
        dy = as_cl(dy)
        if ctx.was_cl:
            if dy.dtype == ctx.src_dtype:
                return dy, None
            dx = empty_cl(dy.shape, ctx.src_dtype, dy.device)
            call("mig_cast", _dt(dy), _dt(dx), _ptr(dy), _ptr(dx), dy.numel(), _stream())
            return dx, None
        return _relayout(dy, ctx.src_dtype, False), None


class _FromChannelsLast(Function):
    @staticmethod
    def forward(ctx, x, dtype):
        ctx.src_dtype = x.dtype
        return _relayout(as_cl(x), dtype, False)

    @staticmethod
    def backward(ctx, dy):
        return _relayout(dy.contiguous(), ctx.src_dtype, True), None


def as_cl(x: torch.Tensor) -> torch.Tensor:
    """Non-differentiable: make sure the memory is channels-last (used on incoming gradients)."""
    if _is_cl(x):
        return x
    return _relayout(x.contiguous(), x.dtype, True)


def _grad_in(g: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """An incoming gradient in the layout the backward kernels read (channels-last activations, contiguous row
    matrices) and in `dtype`."""
    g = as_cl(g) if g.ndim in (4, 5) else g.contiguous()
    return g if g.dtype == dtype else g.to(dtype)


def to_channels_last(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """(N,C,*sp) any layout/dtype -> channels-last memory in the compute dtype (differentiable)."""
    _require_cuda(x, "to_channels_last")
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    if _is_cl(x) and x.dtype == dtype:
        return x
    return _ToChannelsLast.apply(x, dtype)


def from_channels_last(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """channels-last compute tensor -> standard contiguous (N,C,*sp) tensor of `dtype` (differentiable)."""
    return _FromChannelsLast.apply(x, dtype)


_PROFILE = None  # list of (kind, algorithmic flops, (Cin, Cout, out_dims, ksize), start_event, end_event) or None
_PROFILE_SAVED = {}   # kind -> FLOPs the reference's algorithm would have spent that a folded operator did not execute


def _profile_saved(kind: str, flops: float) -> None:
    if _PROFILE is not None:
        _PROFILE_SAVED[kind] = _PROFILE_SAVED.get(kind, 0.0) + flops


def profile_start() -> None:
    """bench.py: record CUDA events (on the launching stream) around every conv implicit-GEMM launch."""
    global _PROFILE
    _PROFILE_SAVED.clear()
    _PROFILE = []


def profile_saved_flops() -> dict:
    """FLOPs NOT executed since profile_start() because an operator ran an algebraically reduced form (the folded
    Upsample convolutions, ops.upsample_conv_nd): reference-algorithm FLOPs minus executed FLOPs, per kind."""
    return dict(_PROFILE_SAVED)


def profile_stop() -> list:
    global _PROFILE
    out, _PROFILE = _PROFILE or [], None
    return out


def _conv_call(kind, geom, name, *args):
    if _PROFILE is None:
        return call(name, *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    call(name, *args)
    e1.record()
    od, ks = tuple(geom.out_dims), tuple(geom.ksize)
    flops = 2.0 * geom.N * od[0] * od[1] * od[2] * geom.Cout * geom.Cin * ks[0] * ks[1] * ks[2]
    _PROFILE.append((kind, flops, (geom.Cin, geom.Cout, od, ks), e0, e1))


def _conv_launch(name, which, kind, geom, dt, device, *args):
    """Launch the implicit-GEMM entry point `name` as `name(geom, dt, *args, engine, workspace, bytes, stream)` with the
    workspace that `mig_conv_workspace_bytes` asks for pass `which` (0 = fwd, 1 = dgrad, 2 = wgrad), profiled as `kind`.
    `which` and `kind` name the pass the kernel serves, which is not always the entry point's own (conv-transpose,
    upconv dgrad)."""
    ws = _workspace(_lib.load().mig_conv_workspace_bytes(C.byref(geom), dt, which, _ENGINE), device)
    _conv_call(kind, geom, name, C.byref(geom), dt, *args, _ENGINE, _ptr(ws), ws.numel(), _stream())


def _deliver(param, grad):
    """Route a parameter gradient: into `param.main_grad` (flat-buffer view owned by engine.FlatAdamW) when present --
    returning None to autograd -- else hand it to autograd unchanged. `grad=None` means the kernel already accumulated
    into main_grad."""
    if param is None:
        return grad
    mg = getattr(param, "main_grad", None)
    if mg is None:
        return grad
    if grad is not None:
        mg.add_(grad)
    hook = getattr(param, "_mig_grad_ready", None)   # set per parameter by the engine.FlatAdamW that owns it
    if hook is not None:
        hook(param)
    return None


def _grad_buf(param) -> torch.Tensor:
    """The fp32 buffer a backward kernel ACCUMULATES `param`'s gradient into: its flat gradient buffer slot
    (`main_grad`) when engine.FlatAdamW owns it, else a zeroed buffer of its shape and memory format. Finish with
    `_grad_done`."""
    mg = getattr(param, "main_grad", None)
    if mg is not None:
        return mg
    return empty_cl(param.shape, torch.float32, param.device).zero_()


def _grad_done(param, buf):
    """What autograd receives for a gradient accumulated into `_grad_buf(param)`: None once it is in main_grad (the
    owner is told it is ready), else the buffer."""
    return _deliver(param, None) if getattr(param, "main_grad", None) is not None else buf


# ----------------------------------------------------------------------------------------------
# filter cache: compute-dtype copy of an fp32 master filter, refreshed when the parameter changes
# ----------------------------------------------------------------------------------------------
def _filter_for(weight: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    if dtype == torch.bfloat16:
        shadow = getattr(weight, "_mig_shadow", None)  # bf16 copy kept current by the fused AdamW kernel
        if shadow is not None:
            # The fused AdamW kernel writes master + shadow together and never bumps the autograd version counter, so
            # a version that differs from the one recorded at the last refresh means somebody ELSE changed the fp32
            # master in place (load_state_dict after the trainer was built -- the reference's resume order,
            # train_ldm.py:522-525 --, AutoencoderKL.initialize, zero_module, copy_): re-cast this parameter's slot.
            if weight._version != weight._mig_shadow_version:
                refresh_shadow(weight)
            return shadow
    w = weight.detach()
    if not _is_cl(w):
        w = w.contiguous(memory_format=_mf(w.ndim))
    if w.dtype == dtype:
        return w
    # The cache lives ON the parameter object (never keyed by address: freed storage is reused by other
    # tensors). An entry is valid only for the same storage address AND the same in-place version counter.
    cache = weight.__dict__.setdefault("_mig_filter_cache", {})
    stamp = (weight.data_ptr(), weight._version)
    hit = cache.get(dtype)
    if hit is not None and hit[0] == stamp and hit[1].shape == w.shape:
        return hit[1]
    wk = torch.empty_like(w, dtype=dtype)  # preserves the channels-last strides
    call("mig_cast", _dt(w), _dt(wk), _ptr(w), _ptr(wk), w.numel(), _stream())
    cache[dtype] = (stamp, wk)
    return wk


def refresh_shadow(weight) -> None:
    """Re-cast one parameter's fp32 master slot into its bf16 shadow slot (both are the same strided view of a
    contiguous, 64-element aligned slot of the flat buffers owned by engine.FlatAdamW)."""
    shadow = weight._mig_shadow
    call("mig_cast", F32, BF16, _ptr(weight), _ptr(shadow), weight.numel(), _stream())
    weight._mig_shadow_version = weight._version


class FusedLinearParams:
    """Several nn.Linear layers that read the same input, presented as ONE (sum of out_features, in_features) weight and
    one bias: possible when engine.FlatAdamW laid their parameters out next to each other in its flat buffers (it does
    for to_q / to_k / to_v of every attention block). `weight` / `bias` are leaf views of the fp32 master buffer that
    carry the same attributes the kernels' wrappers look for on real parameters (main_grad, bf16 shadow, grad-ready
    callback), `order` is the order of the layers' rows in the fused matrix."""

    def __init__(self, weight, bias, order, members):
        self.weight, self.bias, self.order, self.members = weight, bias, order, members

    def refresh(self):
        for m in self.members:   # a member changed in place behind the optimiser's back (load_state_dict, copy_)
            if getattr(m, "_mig_shadow", None) is not None and m._version != m._mig_shadow_version:
                refresh_shadow(m)


def fuse_linears(named_linears):
    """[(name, Linear-like module with .weight/.bias)] -> FusedLinearParams or None (parameters not flat-owned or not
    adjacent)."""
    ws = [(n, m.weight) for n, m in named_linears]
    bs = [(n, m.bias) for n, m in named_linears]
    opt = getattr(ws[0][1], "_mig_flat", None)
    if opt is None or any(getattr(w, "_mig_flat", None) is not opt for _, w in ws):
        return None
    if any(b is None or getattr(b, "_mig_flat", None) is not opt for _, b in bs):
        return None
    ws.sort(key=lambda t: t[1]._mig_slot[0])
    order = tuple(n for n, _ in ws)
    bs.sort(key=lambda t: order.index(t[0]))
    out_f, in_f = ws[0][1].shape

    def adjacent(ps):
        off = ps[0][1]._mig_slot[0]
        for _, p in ps:
            o, k = p._mig_slot
            if o != off or k % 64 != 0 or not p.is_contiguous():
                return None
            off += k
        return ps[0][1]._mig_slot[0]

    if any(tuple(w.shape) != (out_f, in_f) for _, w in ws):
        return None
    wo, bo = adjacent(ws), adjacent(bs)
    if wo is None or bo is None:
        return None
    n = len(ws)
    members = [w for _, w in ws] + [b for _, b in bs]

    def ready(_p):
        for m in members:
            opt._grad_ready(m)

    W = opt.master[wo:wo + n * out_f * in_f].view(n * out_f, in_f).requires_grad_(True)
    W.main_grad = opt.grad[wo:wo + n * out_f * in_f].view(n * out_f, in_f)
    W._mig_shadow = opt.shadow[wo:wo + n * out_f * in_f].view(n * out_f, in_f)
    W._mig_shadow_version = W._version
    W._mig_grad_ready = ready
    Bv = opt.master[bo:bo + n * out_f].requires_grad_(True)
    Bv.main_grad = opt.grad[bo:bo + n * out_f]
    Bv._mig_grad_ready = lambda _p: None      # the weight's callback reports all members
    return FusedLinearParams(W, Bv, order, members)


def clear_caches() -> None:
    _workspaces.clear()


# ----------------------------------------------------------------------------------------------
# convolution (K1/K2/K3) and linear (1x1x1 conv over rows)
# ----------------------------------------------------------------------------------------------
def _geom(N, in_sp, Cin, Cout, ksize, stride, pad):
    in3, k3, s3 = _sp3(in_sp), _sp3(ksize), _sp3(stride)
    p3 = (0,) * (3 - len(pad)) + tuple(int(v) for v in pad)
    out3 = tuple((in3[i] + 2 * p3[i] - k3[i]) // s3[i] + 1 for i in range(3))
    if min(out3) < 1:
        raise RuntimeError(f"conv: kernel {k3} with padding {p3} does not fit input {in3}")
    return _lib.conv_geom(N, in3, out3, Cin, Cout, k3, s3, p3), out3


def _gn_split_ok(x_dtype, N, S, Cc, groups) -> bool:
    if x_dtype != torch.bfloat16 or _ENGINE == _lib.ENGINE_SIMT or not groups:
        return False
    return bool(_lib.load().mig_groupnorm_can_split(BF16, int(N), int(S), int(Cc), int(groups)))


def _conv_forward(x, weight, bias, chan_bias, residual, stride, padding, gn_groups=0):
    """The convolution kernel launch of conv_nd on prepared operands -> (y, geom, gn_sums). gn_sums is
    (sums, gn_groups) when the epilogue also accumulated the GroupNorm statistics of y, else None."""
    N, Cin = x.shape[0], x.shape[1]
    nd = x.ndim - 2
    Cout = weight.shape[0]
    if weight.shape[1] != Cin:
        raise RuntimeError(f"conv: input has {Cin} channels but the filter expects {weight.shape[1]}")
    geom, out3 = _geom(N, x.shape[2:], Cin, Cout, weight.shape[2:], stride, padding)
    wk = _filter_for(weight, x.dtype)
    y = empty_cl((N, Cout, *out3[3 - nd:]), x.dtype, x.device)
    if residual is not None and residual.shape != y.shape:
        raise RuntimeError(f"Sizes of tensors must match: residual {tuple(residual.shape)} vs conv output "
                           f"{tuple(y.shape)}")
    args = (_ptr(x), _ptr(wk), _ptr(bias), _ptr(chan_bias), _ptr(residual), _ptr(y))
    if gn_groups and _gn_split_ok(x.dtype, N, out3[0] * out3[1] * out3[2], Cout, gn_groups):
        # the epilogue also accumulates the GroupNorm statistics of y for the norm that consumes it
        sums = torch.empty((N, gn_groups, 2), dtype=torch.float64, device=x.device)
        _conv_launch("mig_conv_fwd_stats", 0, "fwd", geom, _dt(x), x.device, *args, _ptr(sums), int(gn_groups))
        return y, geom, (sums, int(gn_groups))
    _conv_launch("mig_conv_fwd", 0, "fwd", geom, _dt(x), x.device, *args)
    return y, geom, None


def _conv_backward(x, weight, bias, geom, dy, want_dx, want_dw, want_db, want_dcb, want_dres):
    """Gradients (dx, dw, db, dcb, dres) of _conv_forward; those not wanted are None. weight / bias are the parameter
    objects (they carry main_grad and the bf16 shadow)."""
    # per-(n, c) column sums of dy, when the GroupNorm that consumed this conv's output computed them in its own
    # backward (ops._GroupNormFn): they ARE the time-embedding gradient, and summed over n the bias gradient
    colsum = getattr(dy, "_mig_colsum", None)
    if colsum is not None and tuple(colsum.shape) != (dy.shape[0], dy.shape[1]):
        colsum = None
    dy = _grad_in(dy, x.dtype)
    dt = _dt(x)
    dx = dw = db = dcb = dres = None
    if want_dx:
        wk = _filter_for(weight, x.dtype)
        dx = torch.empty_like(x)
        _conv_launch("mig_conv_dgrad", 1, "dgrad", geom, dt, x.device, _ptr(dy), _ptr(wk), _ptr(dx))
    if want_dw or want_db:
        # the kernels ACCUMULATE: straight into the flat gradient buffer when the engine owns the parameter
        dw_buf = _grad_buf(weight) if want_dw else None
        db_buf = _grad_buf(bias) if want_db else None
        db_arg = db_buf
        if want_db and colsum is not None:   # bias gradient = sum over samples of the ready-made column sums
            call("mig_colsum", F32, _ptr(colsum), _ptr(db_buf), colsum.shape[0], colsum.shape[1], 1, _stream())
            db_arg = None
        if want_dw or db_arg is not None:
            _conv_launch("mig_conv_wgrad", 2, "wgrad", geom, dt, x.device, _ptr(x), _ptr(dy), _ptr(dw_buf),
                         _ptr(db_arg))
        if want_dw:
            dw = _grad_done(weight, dw_buf)
        if want_db:
            db = _grad_done(bias, db_buf)
    if want_dcb:
        N, Cout = dy.shape[0], dy.shape[1]
        if colsum is not None:
            dcb = colsum
        else:
            dcb = torch.empty((N, Cout), dtype=torch.float32, device=dy.device)
            call("mig_chan_bias_bwd", dt, _ptr(dy), _ptr(dcb), N, dy.numel() // (N * Cout), Cout, _stream())
    if want_dres:
        dres = dy
    return dx, dw, db, dcb, dres


class _ConvFn(Function):
    @staticmethod
    def forward(ctx, x, weight, bias, chan_bias, residual, stride, padding, gn_groups=0):
        y, ctx.geom, gn_sums = _conv_forward(x, weight, bias, chan_bias, residual, stride, padding, gn_groups)
        if gn_sums is not None:
            y._mig_gn_sums = gn_sums   # Function.apply hands the caller this very tensor object, attribute included
        ctx.bias_ref, ctx.weight_ref = bias, weight  # the Parameter objects (carry main_grad / shadow attributes)
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, _ = ctx.saved_tensors
        return (*_conv_backward(x, ctx.weight_ref, ctx.bias_ref, ctx.geom, dy, *ctx.needs_input_grad[:5]), None, None,
                None)


def conv_nd(x, weight, bias=None, stride=1, padding=0, chan_bias=None, residual=None, gn_groups=0):
    """Conv{2,3}d with fused epilogue: + bias[c] + chan_bias[n,c] (time embedding, unet:691-695)
    + residual (skip add, unet:701 / ae:204). x, residual: channels-last compute dtype.
    gn_groups > 0: the epilogue also accumulates the statistics of a GroupNorm(gn_groups) over the output; they ride on
    the returned tensor (`_mig_gn_sums`) and ops.group_norm on that tensor skips its statistics pass."""
    _require_cuda(x, "conv_nd")
    nd = x.ndim - 2
    s = tuple(stride) if isinstance(stride, (list, tuple)) else (stride,) * nd
    p = tuple(padding) if isinstance(padding, (list, tuple)) else (padding,) * nd
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    if chan_bias is not None:
        # (rows, C) with rows = N, or ONE row broadcast over the batch: the reference adds temb[:, :, None, None, None]
        # (unet:691-695) and the inferers pass a single timestep for a whole batch (`torch.Tensor((t,))`). The kernels index
        # chan_bias[n * C + c], so the broadcast is made explicit here (expand is differentiable: its backward sums).
        if chan_bias.ndim != 2 or chan_bias.shape[1] != weight.shape[0] or chan_bias.shape[0] not in (1, x.shape[0]):
            raise RuntimeError(f"conv_nd: chan_bias {tuple(chan_bias.shape)} does not broadcast to "
                               f"({x.shape[0]}, {weight.shape[0]})")
        if chan_bias.shape[0] != x.shape[0]:
            chan_bias = chan_bias.expand(x.shape[0], -1)
        chan_bias = chan_bias.float().contiguous()
    if residual is not None and (not _is_cl(residual) or residual.dtype != x.dtype):
        residual = to_channels_last(residual, x.dtype)
    return _ConvFn.apply(x, weight, bias, chan_bias, residual, s, p, int(gn_groups or 0))


class _ConvTransposeFn(Function):
    """nn.ConvTranspose{2,3}d (monai Convolution(is_transposed=True), ae:66-76) on the convolution kernels: a transposed
    convolution IS the data gradient of the strided convolution with the same filter, so
        forward  = mig_conv_dgrad   (stride-residue classes on the tcgen05 kernels, no zero-insertion),
        d/dx     = mig_conv_fwd     (the strided convolution itself),
        d/dw     = mig_conv_wgrad   with the roles of input and output gradient exchanged.
    weight: (Cin, Cout, *k) like torch's ConvTranspose, channels-last memory = [Cin][tap][Cout] = the [Cout'][tap][Cin']
    filter of the underlying convolution (Cout' = Cin, Cin' = Cout)."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride, padding, output_padding):
        N, Cin = x.shape[0], x.shape[1]
        nd = x.ndim - 2
        if weight.shape[0] != Cin:
            raise RuntimeError(f"conv_transpose: input has {Cin} channels but the filter expects {weight.shape[0]}")
        Cout = weight.shape[1]
        k = tuple(weight.shape[2:])
        out_sp = tuple((x.shape[2 + i] - 1) * stride[i] - 2 * padding[i] + k[i] + output_padding[i] for i in range(nd))
        # geometry of the underlying convolution: it maps the transposed conv's OUTPUT to its INPUT
        geom, back3 = _geom(N, out_sp, Cout, Cin, k, stride, padding)
        if tuple(back3[3 - nd:]) != tuple(x.shape[2:]):
            raise RuntimeError(f"conv_transpose: output_padding {output_padding} is inconsistent with stride {stride}")
        wk = _filter_for(weight, x.dtype)
        y = empty_cl((N, Cout, *out_sp), x.dtype, x.device)
        dt = _dt(x)
        _conv_launch("mig_conv_dgrad", 1, "dgrad", geom, dt, x.device, _ptr(x), _ptr(wk), _ptr(y))
        if bias is not None:
            call("mig_add_channel_bias", dt, _ptr(y), _ptr(bias), _ptr(y), y.numel() // Cout, Cout, _stream())
        ctx.geom = geom
        ctx.bias_ref, ctx.weight_ref = bias, weight
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, _ = ctx.saved_tensors
        weight, bias, geom = ctx.weight_ref, ctx.bias_ref, ctx.geom
        dy = _grad_in(dy, x.dtype)
        dt = _dt(x)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wk = _filter_for(weight, x.dtype)
            dx = torch.empty_like(x)
            _conv_launch("mig_conv_fwd", 0, "fwd", geom, dt, x.device, _ptr(dy), _ptr(wk), None, None, None, _ptr(dx))
        if ctx.needs_input_grad[1]:
            dw_buf = _grad_buf(weight)
            # underlying convolution: input = dy (of this op), output gradient = x (of this op)
            _conv_launch("mig_conv_wgrad", 2, "wgrad", geom, dt, x.device, _ptr(dy), _ptr(x), _ptr(dw_buf), None)
            dw = _grad_done(weight, dw_buf)
        if ctx.needs_input_grad[2]:
            db_buf = _grad_buf(bias)
            Cout = dy.shape[1]
            call("mig_colsum", dt, _ptr(dy), _ptr(db_buf), dy.numel() // Cout, Cout, 1, _stream())
            db = _grad_done(bias, db_buf)
        return dx, dw, db, None, None, None


def conv_transpose_nd(x, weight, bias=None, stride=1, padding=0, output_padding=0):
    """ConvTranspose{2,3}d; x channels-last compute dtype, weight (Cin, Cout, *k)."""
    _require_cuda(x, "conv_transpose_nd")
    nd = x.ndim - 2
    tup = lambda v: tuple(v) if isinstance(v, (list, tuple)) else (v,) * nd  # noqa: E731
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    return _ConvTransposeFn.apply(x, weight, bias, tup(stride), tup(padding), tup(output_padding))


class _LinearFn(Function):
    """y[r, o] = sum_i x[r, i] w[o, i] + b[o]  -- a 1x1x1 conv over `rows` voxels (unet:436-438,1832-1834)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        rows, K = x.shape
        O = weight.shape[0]
        geom, _ = _geom(1, (1, 1, rows), K, O, (1, 1, 1), (1, 1, 1), (0, 0, 0))
        wk = _filter_for(weight, x.dtype)
        y = torch.empty((rows, O), dtype=x.dtype, device=x.device)
        _conv_launch("mig_conv_fwd", 0, "fwd", geom, _dt(x), x.device, _ptr(x), _ptr(wk), _ptr(bias), None, None,
                     _ptr(y))
        ctx.geom = geom
        ctx.bias_ref, ctx.weight_ref = bias, weight
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, _ = ctx.saved_tensors
        weight, bias, geom = ctx.weight_ref, ctx.bias_ref, ctx.geom
        dy = _grad_in(dy, x.dtype)
        dt = _dt(x)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wk = _filter_for(weight, x.dtype)
            dx = torch.empty_like(x)
            _conv_launch("mig_conv_dgrad", 1, "dgrad", geom, dt, x.device, _ptr(dy), _ptr(wk), _ptr(dx))
        want_w, want_b = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        if want_w or want_b:
            dw_buf = _grad_buf(weight) if want_w else None
            db_buf = _grad_buf(bias) if want_b else None
            _conv_launch("mig_conv_wgrad", 2, "wgrad", geom, dt, x.device, _ptr(x), _ptr(dy), _ptr(dw_buf),
                         _ptr(db_buf))
            if want_w:
                dw = _grad_done(weight, dw_buf)
            if want_b:
                db = _grad_done(bias, db_buf)
        return dx, dw, db


def linear(x, weight, bias=None):
    """nn.Linear over the last dim; x (..., in) contiguous."""
    _require_cuda(x, "linear")
    shp = x.shape
    y = _LinearFn.apply(x.reshape(-1, shp[-1]).contiguous(), weight, bias)
    return y.reshape(*shp[:-1], weight.shape[0])


class _TembProjAllFn(Function):
    """time_emb_proj of every ResnetBlock applied to the same silu(emb) in one launch per pass (unet:691-695, SURVEY K6).
    forward(x, w0, b0, w1, b1, ...) -> (y0, y1, ...); the layers stay separate fp32 parameters."""

    @staticmethod
    def forward(ctx, x, *params):
        ws, bs = params[0::2], params[1::2]
        n = len(ws)
        rows, K = x.shape
        outs = [torch.empty((rows, w.shape[0]), dtype=torch.float32, device=x.device) for w in ws]
        PA, IA = C.c_void_p * n, C.c_int32 * n
        call("mig_temb_proj_all_fwd", _ptr(x), PA(*[w.data_ptr() for w in ws]),
             PA(*[None if b is None else b.data_ptr() for b in bs]), PA(*[o.data_ptr() for o in outs]),
             IA(*[w.shape[0] for w in ws]), n, rows, K, _stream())
        ctx.save_for_backward(x, *[w.detach() for w in ws])
        ctx.refs = (ws, bs)
        ctx.set_materialize_grads(False)   # a layer whose output is unused gets grad None (not zeros): skipped like torch
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        x, *wt = ctx.saved_tensors
        ws, bs = ctx.refs
        n = len(ws)
        rows, K = x.shape
        keep, dw_b, db_b = [], [None] * n, [None] * n
        for i in range(n):
            if grads[i] is None:     # this layer received no gradient: the kernels skip it (null dy)
                keep.append(None)
                continue
            keep.append(grads[i].float().contiguous())
            dw_b[i] = _grad_buf(ws[i])
            if bs[i] is not None:
                db_b[i] = _grad_buf(bs[i])
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        PA, IA = C.c_void_p * n, C.c_int32 * n
        ptrs = lambda ts: PA(*[None if t is None else t.data_ptr() for t in ts])  # noqa: E731
        call("mig_temb_proj_all_bwd", _ptr(x), ptrs(wt), ptrs(keep), ptrs(dw_b), ptrs(db_b), _ptr(dx),
             IA(*[w.shape[0] for w in wt]), n, rows, K, _stream())
        out = [dx]
        for i in range(n):
            if keep[i] is None:
                out += [None, None]
                continue
            out.append(_grad_done(ws[i], dw_b[i]))
            out.append(None if bs[i] is None else _grad_done(bs[i], db_b[i]))
        return tuple(out)


def temb_projections(x, linears):
    """[Linear-like modules with fp32 .weight/.bias] applied to the same fp32 input x (rows, K) -> list of (rows, C_i)
    tensors, or None when the batched kernels do not apply (more than 32 layers, more than 8 rows, non-fp32)."""
    if not linears or len(linears) > 32 or x.dtype != torch.float32 or x.ndim != 2 or x.shape[0] > 8 or x.shape[1] % 4:
        return None
    if any(m.weight.dtype != torch.float32 or not m.weight.is_contiguous() or m.weight.shape[1] != x.shape[1]
           for m in linears):
        return None
    _require_cuda(x, "temb_projections")
    params = []
    for m in linears:
        params += [m.weight, m.bias]
    return list(_TembProjAllFn.apply(x.contiguous(), *params))


# ----------------------------------------------------------------------------------------------
# GroupNorm (+SiLU), LayerNorm, SiLU
# ----------------------------------------------------------------------------------------------
def _gn_forward(x, gamma, beta, groups, eps, silu):
    """GroupNorm (+SiLU) of channels-last x -> (y, mean, rstd)."""
    N, Cc = x.shape[0], x.shape[1]
    S = x.numel() // (N * Cc)
    y = torch.empty_like(x)
    mean = torch.empty((N, groups), dtype=torch.float32, device=x.device)
    rstd = torch.empty_like(mean)
    pre = getattr(x, "_mig_gn_sums", None)   # statistics accumulated by the producing convolution's epilogue
    if pre is not None and pre[1] == groups and tuple(pre[0].shape) == (N, groups, 2) and \
            _gn_split_ok(x.dtype, N, S, Cc, groups):
        call("mig_groupnorm_apply", _dt(x), _ptr(x), _ptr(gamma), _ptr(beta), _ptr(pre[0]), _ptr(y), _ptr(mean),
             _ptr(rstd), N, S, Cc, groups, float(eps), int(silu), _stream())
    else:
        need = _lib.load().mig_groupnorm_workspace_bytes(N, S, Cc, groups)
        ws = _workspace(need, x.device)
        call("mig_groupnorm_fwd", _dt(x), _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(mean), _ptr(rstd), N, S, Cc,
             groups, float(eps), int(silu), _ptr(ws), ws.numel(), _stream())
    return y, mean, rstd


def _gn_backward(x, gamma, beta, mean, rstd, groups, silu, want_colsum, dy, dskip=None):
    """-> (dx, dgamma, dbeta). gamma / beta are the parameter objects (they carry main_grad).
    dskip: the gradient that reaches x through the block's skip path (x also feeds the residual add / skip conv): it is
    added inside the GroupNorm backward kernel instead of by a separate accumulation pass.
    want_colsum: x is the output of a convolution that only this norm consumes; hand that convolution's backward the
    column sums of dx (`_mig_colsum`)."""
    N, Cc = x.shape[0], x.shape[1]
    S = x.numel() // (N * Cc)
    if dy is None:   # the normalised branch got no gradient: only the skip path contributes
        return (None if dskip is None else as_cl(dskip)), None, None
    dy = _grad_in(dy, x.dtype)
    if dskip is not None:
        dskip = _grad_in(dskip, x.dtype)
    dx = torch.empty_like(x)
    g_main, b_main = getattr(gamma, "main_grad", None), getattr(beta, "main_grad", None)
    into_main = g_main is not None and b_main is not None     # accumulate straight into the flat gradient buffer
    dgamma = g_main if into_main else torch.empty_like(gamma)
    dbeta = b_main if into_main else torch.empty_like(beta)
    need = _lib.load().mig_groupnorm_workspace_bytes(N, S, Cc, groups)
    ws = _workspace(need, x.device)
    colsum = torch.empty((N, Cc), dtype=torch.float32, device=x.device) if (want_colsum and dskip is None) else None
    call("mig_groupnorm_bwd", _dt(x), _ptr(x), _ptr(dy), _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(rstd), _ptr(dx),
         _ptr(dgamma), _ptr(dbeta), _ptr(colsum), _ptr(dskip), int(into_main), N, S, Cc, groups, int(silu), _ptr(ws),
         ws.numel(), _stream())
    if colsum is not None:
        # rides on the gradient tensor to the backward of the convolution that produced x (its bias and
        # time-embedding gradients are these column sums); if autograd hands that node a different tensor
        # (several consumers -> accumulated gradient) the attribute is simply absent and the conv sums dy itself
        dx._mig_colsum = colsum
    if into_main:
        return dx, _deliver(gamma, None), _deliver(beta, None)
    return dx, _deliver(gamma, dgamma), _deliver(beta, dbeta)


class _GroupNormFn(Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, groups, eps, silu):
        y, mean, rstd = _gn_forward(x, gamma, beta, groups, eps, silu)
        ctx.save_for_backward(x, gamma, beta, mean, rstd)
        ctx.refs = (gamma, beta)   # the Parameter objects (carry main_grad)
        ctx.cfg = (groups, silu, bool(getattr(x, "_mig_sole_consumer_gn", False)))
        return y

    @staticmethod
    def backward(ctx, dy):
        x, _, _, mean, rstd = ctx.saved_tensors
        return (*_gn_backward(x, *ctx.refs, mean, rstd, *ctx.cfg, dy), None, None, None)


class _GroupNormSkipFn(Function):
    """GroupNorm whose input ALSO feeds the block's skip path (ResnetBlock: unet:674-701, x -> norm1 and x -> skip /
    residual add; AttentionBlock: unet:418-458). Returns (norm(x), x): the second output is x itself for the skip path,
    so both gradients arrive at this node together and are summed inside the backward kernel."""

    @staticmethod
    def forward(ctx, x, gamma, beta, groups, eps, silu):
        y, mean, rstd = _gn_forward(x, gamma, beta, groups, eps, silu)
        ctx.save_for_backward(x, gamma, beta, mean, rstd)
        ctx.refs = (gamma, beta)   # the Parameter objects (carry main_grad)
        ctx.cfg = (groups, silu, bool(getattr(x, "_mig_sole_consumer_gn", False)))
        return y, x.view_as(x)

    @staticmethod
    def backward(ctx, dy, dskip):
        x, _, _, mean, rstd = ctx.saved_tensors
        return (*_gn_backward(x, *ctx.refs, mean, rstd, *ctx.cfg, dy, dskip), None, None, None)


def group_norm(x, gamma, beta, groups: int, eps: float, silu: bool = False, with_skip: bool = False):
    """nn.GroupNorm (fp32 statistics) with optional fused SiLU (unet:628-629,648,1932-1933; ae:157,194).
    with_skip=True returns (y, x_skip): use x_skip instead of x for the block's skip path."""
    _require_cuda(x, "group_norm")
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    if with_skip:
        if torch.is_grad_enabled() and x.requires_grad:
            return _GroupNormSkipFn.apply(x, gamma, beta, int(groups), float(eps), bool(silu))
        return _GroupNormFn.apply(x, gamma, beta, int(groups), float(eps), bool(silu)), x
    return _GroupNormFn.apply(x, gamma, beta, int(groups), float(eps), bool(silu))


class _LayerNormFn(Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, eps):
        rows, Cc = x.shape
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty_like(mean)
        call("mig_layernorm_fwd", _dt(x), _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(mean), _ptr(rstd), rows, Cc,
             float(eps), _stream())
        ctx.save_for_backward(x, gamma, mean, rstd)
        ctx.refs = (gamma, beta)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, mean, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        rows, Cc = x.shape
        dx = torch.empty_like(x)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        call("mig_layernorm_bwd", _dt(x), _ptr(x), _ptr(dy), _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dx),
             _ptr(dgamma), _ptr(dbeta), rows, Cc, _stream())
        return dx, _deliver(ctx.refs[0], dgamma), _deliver(ctx.refs[1], dbeta), None


def layer_norm(x, gamma, beta, eps: float = 1e-5):
    shp = x.shape
    return _LayerNormFn.apply(x.reshape(-1, shp[-1]).contiguous(), gamma, beta, float(eps)).reshape(shp)


class _SiluFn(Function):
    @staticmethod
    def forward(ctx, x):
        y = torch.empty_like(x)
        call("mig_silu_fwd", _dt(x), _ptr(x), _ptr(y), x.numel(), _stream())
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dy = dy.contiguous() if x.is_contiguous() else as_cl(dy)
        dx = torch.empty_like(x)
        call("mig_silu_bwd", _dt(x), _ptr(x), _ptr(dy), _ptr(dx), x.numel(), _stream())
        return dx


def silu(x):
    _require_cuda(x, "silu")
    if not (x.is_contiguous() or _is_cl(x)):
        x = x.contiguous()
    return _SiluFn.apply(x)


class _AddFn(Function):
    @staticmethod
    def forward(ctx, a, b):
        y = torch.empty_like(a)
        call("mig_add", _dt(a), _ptr(a), _ptr(b), _ptr(y), a.numel(), _stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        return dy, dy


def add(a, b):
    """Elementwise add of two tensors with identical shape, dtype and memory layout."""
    if a.shape != b.shape:
        raise RuntimeError(f"Sizes of tensors must match: {tuple(a.shape)} vs {tuple(b.shape)}")
    if b.dtype != a.dtype:
        b = b.to(a.dtype)
    if a.stride() != b.stride():
        b = as_cl(b) if _is_cl(a) else b.contiguous()
        if a.stride() != b.stride():
            a = a.contiguous()
            b = b.contiguous()
    return _AddFn.apply(a, b)


class _ScaleFn(Function):
    @staticmethod
    def forward(ctx, x, s):
        ctx.s = s
        y = torch.empty_like(x)
        call("mig_scale", _dt(x), _ptr(x), _ptr(y), float(s), x.numel(), _stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = dy.contiguous() if not _is_cl(dy) else dy
        dx = torch.empty_like(dy)
        call("mig_scale", _dt(dy), _ptr(dy), _ptr(dx), float(ctx.s), dy.numel(), _stream())
        return dx, None


def scale(x, s: float):
    if not (x.is_contiguous() or _is_cl(x)):
        x = x.contiguous()
    return _ScaleFn.apply(x, float(s))


class _GegluFn(Function):
    @staticmethod
    def forward(ctx, x):
        rows, H2 = x.shape
        y = torch.empty((rows, H2 // 2), dtype=x.dtype, device=x.device)
        call("mig_geglu_fwd", _dt(x), _ptr(x), _ptr(y), rows, H2 // 2, _stream())
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dx = torch.empty_like(x)
        call("mig_geglu_bwd", _dt(x), _ptr(x), _ptr(dy.contiguous()), _ptr(dx), x.shape[0], x.shape[1] // 2, _stream())
        return dx


def geglu(x):
    """x[..., :H] * gelu(x[..., H:]) (monai MLPBlock act="GEGLU", unet:213)."""
    shp = x.shape
    return _GegluFn.apply(x.reshape(-1, shp[-1]).contiguous()).reshape(*shp[:-1], shp[-1] // 2)


# ----------------------------------------------------------------------------------------------
# concat / upsample
# ----------------------------------------------------------------------------------------------
class _CatFn(Function):
    @staticmethod
    def forward(ctx, a, b):
        N, Ca, Cb = a.shape[0], a.shape[1], b.shape[1]
        y = empty_cl((N, Ca + Cb, *a.shape[2:]), a.dtype, a.device)
        rows = a.numel() // Ca
        call("mig_concat_channels", _dt(a), _ptr(a), _ptr(b), _ptr(y), rows, Ca, Cb, _stream())
        ctx.split = (Ca, Cb)
        return y

    @staticmethod
    def backward(ctx, dy):
        Ca, Cb = ctx.split
        dy = as_cl(dy)
        N = dy.shape[0]
        da = empty_cl((N, Ca, *dy.shape[2:]), dy.dtype, dy.device)
        db = empty_cl((N, Cb, *dy.shape[2:]), dy.dtype, dy.device)
        call("mig_split_channels", _dt(dy), _ptr(dy), _ptr(da), _ptr(db), dy.numel() // (Ca + Cb), Ca, Cb, _stream())
        return da, db


def cat_channels(a, b):
    """torch.cat([a, b], dim=1) on channels-last tensors (unet:1263,1377,1504)."""
    if a.shape[0] != b.shape[0] or a.shape[2:] != b.shape[2:]:
        raise RuntimeError(f"Sizes of tensors must match except in dimension 1. Expected size {tuple(a.shape)} but got "
                           f"size {tuple(b.shape)}")
    if b.dtype != a.dtype:
        b = b.to(a.dtype)
    return _CatFn.apply(to_channels_last(a, a.dtype), to_channels_last(b, b.dtype))


class _UpsampleFn(Function):
    @staticmethod
    def forward(ctx, x, factors):
        N, Cc = x.shape[0], x.shape[1]
        nd = x.ndim - 2
        in3, f3 = _sp3(x.shape[2:]), (1,) * (3 - nd) + tuple(factors)
        out_sp = tuple(x.shape[2 + i] * factors[i] for i in range(nd))
        y = empty_cl((N, Cc, *out_sp), x.dtype, x.device)
        I3 = C.c_int32 * 3
        call("mig_upsample_nearest_fwd", _dt(x), _ptr(x), _ptr(y), N, I3(*in3), I3(*f3), Cc, _stream())
        ctx.cfg = (in3, f3, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        in3, f3, shape = ctx.cfg
        dy = as_cl(dy)
        dx = empty_cl(shape, dy.dtype, dy.device)
        I3 = C.c_int32 * 3
        call("mig_upsample_nearest_bwd", _dt(dy), _ptr(dy), _ptr(dx), shape[0], I3(*in3), I3(*f3), shape[1], _stream())
        return dx, None


class _AvgPoolFn(Function):
    @staticmethod
    def forward(ctx, x, ksize, stride):
        N, Cc = x.shape[0], x.shape[1]
        nd = x.ndim - 2
        in3, k3, s3 = _sp3(x.shape[2:]), (1,) * (3 - nd) + tuple(ksize), (1,) * (3 - nd) + tuple(stride)
        if any(x.shape[2 + i] < ksize[i] for i in range(nd)):
            raise RuntimeError(f"avg_pool: kernel {tuple(ksize)} is larger than the input {tuple(x.shape[2:])}")
        out_sp = tuple((x.shape[2 + i] - ksize[i]) // stride[i] + 1 for i in range(nd))
        y = empty_cl((N, Cc, *out_sp), x.dtype, x.device)
        I3 = C.c_int32 * 3
        call("mig_avgpool_fwd", _dt(x), _ptr(x), _ptr(y), N, I3(*in3), I3(*k3), I3(*s3), Cc, _stream())
        ctx.cfg = (in3, k3, s3, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        in3, k3, s3, shape = ctx.cfg
        dy = as_cl(dy)
        dx = empty_cl(shape, dy.dtype, dy.device)
        I3 = C.c_int32 * 3
        call("mig_avgpool_bwd", _dt(dy), _ptr(dy), _ptr(dx), shape[0], I3(*in3), I3(*k3), I3(*s3), shape[1], _stream())
        return dx, None, None


def avg_pool(x, kernel_size, stride):
    """nn.AvgPool{2,3}d(kernel_size, stride), no padding (unet:517-518)."""
    _require_cuda(x, "avg_pool")
    nd = x.ndim - 2
    tup = lambda v: tuple(int(a) for a in v) if isinstance(v, (list, tuple)) else (int(v),) * nd  # noqa: E731
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    return _AvgPoolFn.apply(x, tup(kernel_size), tup(stride))


def upsample_nearest(x, factors):
    """F.interpolate(x, scale_factor=factors, mode='nearest') for integer per-axis factors (unet:580, ae:99)."""
    nd = x.ndim - 2
    f = tuple(factors) if isinstance(factors, (list, tuple)) else (factors,) * nd
    fi = tuple(int(v) for v in f)
    if any(float(a) != float(b) for a, b in zip(f, fi)) or min(fi) < 1:
        raise RuntimeError(f"upsample_nearest: only positive integer scale factors are supported, got {f}")
    if all(v == 1 for v in fi):
        return x
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    return _UpsampleFn.apply(x, fi)


# ----------------------------------------------------------------------------------------------
# nearest upsample folded into the convolution that follows it (K8; unet:576-584, ae:97-106)
# ----------------------------------------------------------------------------------------------
_UPCONV = os.environ.get("MIG_UPCONV", "auto")    # auto | always | never (A/B switch and tests)
_UPCONV_MIN_TILES = int(os.environ.get("MIG_UPCONV_MIN_TILES", "96"))     # 256 x 256 tiles per class for 'auto'
_UPCONV_DIRECT = os.environ.get("MIG_UPCONV_DIRECT", "1") != "0"          # forward scatters straight into y (A/B)


def set_upconv(mode: str) -> None:
    """'auto' (fold where the cost model says it pays), 'always' (wherever the kernels can), 'never'."""
    global _UPCONV
    if mode not in ("auto", "always", "never"):
        raise ValueError("set_upconv: mode must be 'auto', 'always' or 'never'")
    _UPCONV = mode


def _axis_fold(k: int, f: int, p: int):
    """Per output residue class r of one axis: (base, folded tap count). An output o = f*j + r reads low-resolution voxels
    j + floor((r + t - p) / f), t = 0..k-1: `base` is the smallest offset, the count how many distinct ones there are."""
    out = []
    for r in range(f):
        d = [(r + t - p) // f for t in range(k)]
        out.append((min(d), max(d) - min(d) + 1))
    return out


def upconv_usable(x, weight, factors, padding) -> bool:
    """Can (and should) `upsample_nearest(x, factors)` + `conv_nd(weight, stride 1, padding)` run folded?"""
    if _UPCONV == "never" or x.dtype != torch.bfloat16 or _ENGINE == _lib.ENGINE_SIMT or not x.is_cuda:
        return False
    nd = x.ndim - 2
    k, f, p = tuple(weight.shape[2:]), tuple(int(v) for v in factors), tuple(int(v) for v in padding)
    if all(v == 1 for v in f) or any(v not in (1, 2) for v in f):
        return False
    if any(ki != 2 * pi + 1 or ki > 3 for ki, pi in zip(k, p)):     # "same" convolutions only: output = f * input
        return False
    Cout, Cin = weight.shape[0], weight.shape[1]
    if Cin % 64 != 0 or Cout % 64 != 0:      # every piece on the TMA box kernels (wgrad panels: multiples of 64)
        return False
    if not _lib.load().mig_has_tcgen05():
        return False
    if _UPCONV == "always":
        return True
    # cost model: the per-class convolutions run one after the other, each over 1/f^n of the output voxels; on a small
    # level a class no longer fills the 148 SMs with 256 x 256 tiles and the fold loses to one big launch
    return _upconv_tiles(x, Cout) >= _UPCONV_MIN_TILES


def _upconv_tiles(x, Cout) -> int:
    rows = x.shape[0] * math.prod(x.shape[2:])
    return -(-rows // 256) * -(-Cout // 256)


class _UpConvFn(Function):
    """y = conv(nearest_upsample(x, f), w, b, stride 1, padding p) without the upsampled tensor (csrc/upconv.cu)."""

    @staticmethod
    def forward(ctx, x, weight, bias, factors, padding):
        N, Cin = x.shape[0], x.shape[1]
        nd = x.ndim - 2
        Cout = weight.shape[0]
        if weight.shape[1] != Cin:
            raise RuntimeError(f"conv: input has {Cin} channels but the filter expects {weight.shape[1]}")
        low3 = _sp3(x.shape[2:])
        k3 = _sp3(weight.shape[2:])
        f3 = (1,) * (3 - nd) + tuple(factors)
        p3 = (0,) * (3 - nd) + tuple(padding)
        I3 = C.c_int32 * 3
        kk, ff, pp = I3(*k3), I3(*f3), I3(*p3)
        lib = _lib.load()
        wk = _filter_for(weight, x.dtype)
        folded = torch.empty(int(lib.mig_upconv_folded_elems(Cout, Cin, kk, ff, pp, 0)), dtype=x.dtype, device=x.device)
        call("mig_upconv_fold_filter", _ptr(wk), _ptr(folded), Cout, Cin, kk, ff, pp, 0, _stream())
        folds = [_axis_fold(k3[i], f3[i], p3[i]) for i in range(3)]
        classes = [(r0, r1, r2) for r0 in range(f3[0]) for r1 in range(f3[1]) for r2 in range(f3[2])]
        per_class = N * low3[0] * low3[1] * low3[2] * Cout
        dt = _dt(x)
        out_sp = tuple(low3[i] * f3[i] for i in range(3))[3 - nd:]
        y = empty_cl((N, Cout, *out_sp), x.dtype, x.device)
        geoms, off = [], 0
        for r in classes:
            base = [folds[i][r[i]][0] for i in range(3)]
            nu = [folds[i][r[i]][1] for i in range(3)]
            geoms.append((_lib.conv_geom(N, low3, low3, Cin, Cout, nu, (1, 1, 1), [-b for b in base]), off))
            off += nu[0] * nu[1] * nu[2] * Cout * Cin
        # Large levels: every class goes through the persistent box kernel and its epilogue writes rows j to f*j + r of y
        # (the strided dgrad's row mapping). Small levels need split-K to fill the GPU, which wants rows 1:1 with the
        # output: per-class convolutions into class buffers, then one interleave pass.
        same_taps = all(tuple(g.ksize) == tuple(geoms[0][0].ksize) for g, _ in geoms)
        direct = (_UPCONV_DIRECT and same_taps and _upconv_tiles(x, Cout) >= _UPCONV_MIN_TILES
                  and lib.mig_upconv_fwd_direct_ok(N, I3(*low3), Cin, Cout))
        if direct:
            g0 = geoms[0][0]
            total = _lib.conv_geom(N * len(classes), low3, low3, Cin, Cout, tuple(g0.ksize), (1, 1, 1), tuple(g0.pad))
            _conv_call("fwd", total, "mig_upconv_fwd", _ptr(x), _ptr(folded), _ptr(bias), _ptr(y), N, I3(*low3), Cin, Cout,
                       kk, ff, pp, _stream())
        else:
            yc = torch.empty(len(classes) * per_class, dtype=x.dtype, device=x.device)
            for ci, (geom, goff) in enumerate(geoms):
                _conv_launch("mig_conv_fwd", 0, "fwd", geom, dt, x.device, _ptr(x),
                             C.c_void_p(folded.data_ptr() + 2 * goff), _ptr(bias), None, None,
                             C.c_void_p(yc.data_ptr() + 2 * ci * per_class))
            call("mig_class_interleave", dt, _ptr(yc), _ptr(y), N, I3(*low3), ff, Cout, 0, _stream())
        ref = 2.0 * N * math.prod(low3) * math.prod(f3) * Cout * Cin * math.prod(k3)      # the reference's k^n taps
        _profile_saved("fwd", ref - sum(2.0 * N * math.prod(low3) * Cout * Cin * math.prod(g.ksize) for g, _ in geoms))
        ctx.cfg = (low3, k3, f3, p3, geoms, per_class, off)
        ctx.bias_ref, ctx.weight_ref = bias, weight
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, _ = ctx.saved_tensors
        weight, bias = ctx.weight_ref, ctx.bias_ref
        low3, k3, f3, p3, geoms, per_class, folded_elems = ctx.cfg
        N, Cin, Cout = x.shape[0], x.shape[1], weight.shape[0]
        I3 = C.c_int32 * 3
        kk, ff, pp = I3(*k3), I3(*f3), I3(*p3)
        lib = _lib.load()
        dy = _grad_in(dy, x.dtype)
        dt = _dt(x)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            # dx = a stride-f convolution of dy with the (f + k - 1)^n-tap folded filter [Cin][s][Cout]
            wk = _filter_for(weight, x.dtype)
            wd = torch.empty(int(lib.mig_upconv_folded_elems(Cout, Cin, kk, ff, pp, 1)), dtype=x.dtype, device=x.device)
            call("mig_upconv_fold_filter", _ptr(wk), _ptr(wd), Cout, Cin, kk, ff, pp, 1, _stream())
            full3 = tuple(low3[i] * f3[i] for i in range(3))
            geom = _lib.conv_geom(N, full3, low3, Cout, Cin, [f3[i] + k3[i] - 1 for i in range(3)], f3,
                                  [k3[i] - 1 - p3[i] for i in range(3)])
            dx = torch.empty_like(x)
            _conv_launch("mig_conv_fwd", 0, "dgrad", geom, dt, x.device, _ptr(dy), _ptr(wd), None, None, None, _ptr(dx))
            ref = 2.0 * N * math.prod(full3) * Cout * Cin * math.prod(k3)
            _profile_saved("dgrad", ref - 2.0 * N * math.prod(low3) * Cout * Cin * math.prod(geom.ksize))
        want_w, want_b = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        if want_w or want_b:
            dw_buf = _grad_buf(weight) if want_w else None
            db_buf = _grad_buf(bias) if want_b else None
            # dy split into its residue classes (contiguous low-resolution tensors), one wgrad per class into the folded
            # layout, then unfolded onto the k^n taps; the bias gradient rides on the class wgrads
            dyc = torch.empty(len(geoms) * per_class, dtype=x.dtype, device=x.device)
            call("mig_class_interleave", dt, _ptr(dy), _ptr(dyc), N, I3(*low3), ff, Cout, 1, _stream())
            dwc = torch.zeros(folded_elems, dtype=torch.float32, device=x.device) if want_w else None
            for ci, (geom, off) in enumerate(geoms):
                _conv_launch("mig_conv_wgrad", 2, "wgrad", geom, dt, x.device, _ptr(x),
                             C.c_void_p(dyc.data_ptr() + 2 * ci * per_class),
                             C.c_void_p(dwc.data_ptr() + 4 * off) if want_w else None, _ptr(db_buf))
            ref = 2.0 * N * math.prod(low3) * math.prod(f3) * Cout * Cin * math.prod(k3)
            _profile_saved("wgrad", ref - sum(2.0 * N * math.prod(low3) * Cout * Cin * math.prod(g.ksize) for g, _ in geoms))
            if want_w:
                call("mig_upconv_unfold_wgrad", _ptr(dwc), _ptr(dw_buf), Cout, Cin, kk, ff, pp, _stream())
                dw = _grad_done(weight, dw_buf)
            if want_b:
                db = _grad_done(bias, db_buf)
        return dx, dw, db, None, None


def upsample_conv_nd(x, weight, bias, factors, padding):
    """conv_nd(upsample_nearest(x, factors), weight, bias, stride 1, padding): folded into per-class convolutions of the
    low-resolution tensor where `upconv_usable` says so, the two separate operators otherwise."""
    _require_cuda(x, "upsample_conv_nd")
    nd = x.ndim - 2
    f = tuple(factors) if isinstance(factors, (list, tuple)) else (factors,) * nd
    p = tuple(padding) if isinstance(padding, (list, tuple)) else (padding,) * nd
    fi = tuple(int(v) for v in f)
    if any(float(a) != float(b) for a, b in zip(f, fi)) or min(fi) < 1 or not upconv_usable(x, weight, fi, p):
        return conv_nd(upsample_nearest(x, f), weight, bias, 1, p)
    if not _is_cl(x):
        x = to_channels_last(x, x.dtype)
    return _UpConvFn.apply(x, weight, bias, fi, tuple(int(v) for v in p))


# ----------------------------------------------------------------------------------------------
# attention core: softmax(scale * Q K^T) V with heads inside the channel dim (unet:406-416)
# ----------------------------------------------------------------------------------------------
def _gemm(A, B, Cm, M, N, K, bo, bi, a, b, c, alpha=1.0, accumulate=False):
    d = _lib.GemmDesc()
    d.M, d.N, d.K, d.batch_outer, d.batch_inner = M, N, K, bo, bi
    d.a_m, d.a_k, d.a_outer, d.a_inner = a
    d.b_k, d.b_n, d.b_outer, d.b_inner = b
    d.c_m, d.c_n, d.c_outer, d.c_inner = c
    d.alpha, d.accumulate = float(alpha), int(accumulate)
    call("mig_gemm_strided", C.byref(d), _dt(A), _dt(Cm), _ptr(A), _ptr(B), _ptr(Cm), _ENGINE, _stream())


def _sdpa_fwd_unfused(q, k, v, B, Lq, Lk, Cc, heads, scale_, ld):
    """softmax(scale q k^T) v with q/k/v given as (B, L, Cc) views whose rows lie `ld` elements apart (ld = Cc for
    contiguous tensors, 3*Cc for the column slices of a fused QKV projection). Returns (O contiguous, P)."""
    dh = Cc // heads
    dev = q.device
    # scores in fp32 (softmax statistics in fp32 as under autocast), probabilities in the compute dtype
    S = torch.empty((B * heads, Lq, Lk), dtype=torch.float32, device=dev)
    _gemm(q, k, S, Lq, Lk, dh, B, heads, (ld, 1, Lq * ld, dh), (1, ld, Lk * ld, dh), (Lk, 1, heads * Lq * Lk, Lq * Lk))
    P = torch.empty((B * heads, Lq, Lk), dtype=q.dtype, device=dev)
    call("mig_softmax_fwd", F32, _dt(P), _ptr(S), _ptr(P), B * heads * Lq, Lk, float(scale_), _stream())
    del S
    O = torch.empty((B, Lq, Cc), dtype=q.dtype, device=dev)
    _gemm(P, v, O, Lq, dh, Lk, B, heads, (Lk, 1, heads * Lq * Lk, Lq * Lk), (ld, 1, Lk * ld, dh), (Cc, 1, Lq * Cc, dh))
    return O, P


def _sdpa_bwd_unfused(q, k, v, P, dO, dQ, dK, dV, B, Lq, Lk, Cc, heads, scale_, ld, ldg):
    """Gradients of the above into dQ / dK / dV, (B, L, Cc) views with row stride `ldg`."""
    dh = Cc // heads
    dev = q.device
    sP = (Lk, 1, heads * Lq * Lk, Lq * Lk)
    # dV[key, d] = sum_q P[q, key] dO[q, d]
    _gemm(P, dO, dV, Lk, dh, Lq, B, heads, (1, Lk, heads * Lq * Lk, Lq * Lk), (Cc, 1, Lq * Cc, dh), (ldg, 1, Lk * ldg, dh))
    # dP[q, key] = sum_d dO[q, d] V[key, d]
    dP = torch.empty((B * heads, Lq, Lk), dtype=torch.float32, device=dev)
    _gemm(dO, v, dP, Lq, Lk, dh, B, heads, (Cc, 1, Lq * Cc, dh), (1, ld, Lk * ld, dh), sP)
    # dS = scale * P * (dP - rowsum(dP * P))   (gradient w.r.t. the UNscaled scores)
    dS = torch.empty((B * heads, Lq, Lk), dtype=q.dtype, device=dev)
    if q.dtype == torch.float32:
        call("mig_softmax_bwd", F32, F32, _ptr(P), _ptr(dP), _ptr(dS), B * heads * Lq, Lk, float(scale_), _stream())
    else:
        # bf16 P, fp32 dP -> bf16 dS in one pass
        call("mig_softmax_bwd_narrow", _ptr(P), _ptr(dP), _ptr(dS), B * heads * Lq, Lk, float(scale_), _stream())
    del dP
    # dQ[q, d] = sum_key dS[q, key] K[key, d] ; dK[key, d] = sum_q dS[q, key] Q[q, d]
    _gemm(dS, k, dQ, Lq, dh, Lk, B, heads, sP, (ld, 1, Lk * ld, dh), (ldg, 1, Lq * ldg, dh))
    _gemm(dS, q, dK, Lk, dh, Lq, B, heads, (1, Lk, heads * Lq * Lk, Lq * Lk), (ld, 1, Lq * ld, dh), (ldg, 1, Lk * ldg, dh))


class _SdpaFn(Function):
    @staticmethod
    def forward(ctx, q, k, v, heads, scale_):
        B, Lq, Cc = q.shape
        Lk = k.shape[1]
        O, P = _sdpa_fwd_unfused(q, k, v, B, Lq, Lk, Cc, heads, scale_, Cc)
        ctx.save_for_backward(q, k, v, P)
        ctx.cfg = (heads, scale_)
        return O

    @staticmethod
    def backward(ctx, dO):
        q, k, v, P = ctx.saved_tensors
        heads, scale_ = ctx.cfg
        B, Lq, Cc = q.shape
        Lk = k.shape[1]
        dO = _grad_in(dO, q.dtype)
        dQ, dK, dV = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        _sdpa_bwd_unfused(q, k, v, P, dO, dQ, dK, dV, B, Lq, Lk, Cc, heads, scale_, Cc, Cc)
        return dQ, dK, dV, None, None


class _QkvSdpaFn(Function):
    """Self-attention on the output of ONE fused QKV projection: qkv (B, L, 3C) holds the three projections side by side
    (`order`, e.g. ("v", "k", "q") -- the order the flat optimiser lays the three weight matrices out). The unfused GEMMs
    read the column slices in place (row stride 3C) and the backward writes dq / dk / dv straight into the slices of
    ONE gradient tensor, so the projection's dgrad and wgrad are single GEMMs as well (unet:436-438 as one Linear)."""

    @staticmethod
    def forward(ctx, qkv, heads, scale_, order):
        B, L, C3 = qkv.shape
        Cc = C3 // 3
        sl = {name: qkv[:, :, i * Cc:(i + 1) * Cc] for i, name in enumerate(order)}
        q, k, v = sl["q"], sl["k"], sl["v"]
        use_flash = flash_attention_usable(qkv[:, :, :Cc], qkv[:, :, :Cc], qkv[:, :, :Cc], heads, needs_grad=bool(ctx.needs_input_grad[0]))
        if use_flash:
            # the forward kernel reads the three column blocks in place (row pitch 3C); contiguous copies are only made
            # when a backward will need them
            if ctx.needs_input_grad[0]:
                qc, kc, vc = q.contiguous(), k.contiguous(), v.contiguous()
                O, lse = _flash_fwd(qc, kc, vc, heads, scale_)
                ctx.save_for_backward(qc, kc, vc, O, lse)
            else:
                O, lse = _flash_fwd(q, k, v, heads, scale_)
        else:
            O, P = _sdpa_fwd_unfused(q, k, v, B, L, L, Cc, heads, scale_, C3)
            ctx.save_for_backward(qkv, P)
        ctx.cfg = (heads, scale_, tuple(order), use_flash, (B, L, Cc))
        return O

    @staticmethod
    def backward(ctx, dO):
        heads, scale_, order, use_flash, (B, L, Cc) = ctx.cfg
        C3 = 3 * Cc
        if use_flash:
            qc, kc, vc, O, lse = ctx.saved_tensors
            dO = _grad_in(dO, qc.dtype)
            dqkv = torch.empty((B, L, C3), dtype=qc.dtype, device=qc.device)
            dq, dk, dv = _flash_bwd(qc, kc, vc, O, lse, dO, heads, scale_)
            parts = {"q": dq, "k": dk, "v": dv}
            rows = B * L
            a, b_, c = (parts[n] for n in order)
            # three column blocks -> one (rows, 3C) matrix: concat(concat(a, b), c) with the channel-concat kernel
            ab = torch.empty((rows, 2 * Cc), dtype=qc.dtype, device=qc.device)
            call("mig_concat_channels", _dt(a), _ptr(a), _ptr(b_), _ptr(ab), rows, Cc, Cc, _stream())
            call("mig_concat_channels", _dt(a), _ptr(ab), _ptr(c), _ptr(dqkv), rows, 2 * Cc, Cc, _stream())
            return dqkv, None, None, None
        qkv, P = ctx.saved_tensors
        dO = _grad_in(dO, qkv.dtype)
        dqkv = torch.empty_like(qkv)
        sl = {name: qkv[:, :, i * Cc:(i + 1) * Cc] for i, name in enumerate(order)}
        dsl = {name: dqkv[:, :, i * Cc:(i + 1) * Cc] for i, name in enumerate(order)}
        _sdpa_bwd_unfused(sl["q"], sl["k"], sl["v"], P, dO, dsl["q"], dsl["k"], dsl["v"], B, L, L, Cc, heads, scale_, C3, C3)
        return dqkv, None, None, None


def sdpa_qkv(qkv, heads: int, scale_: float, order=("q", "k", "v")):
    """Self-attention over a fused projection output qkv (B, L, 3C); see _QkvSdpaFn."""
    _require_cuda(qkv, "sdpa_qkv")
    return _QkvSdpaFn.apply(qkv.contiguous(), int(heads), float(scale_), tuple(order))


def sdpa(q, k, v, heads: int, scale_: float):
    """softmax(scale * q k^T) v per head; q (B,Lq,C), k/v (B,Lk,C), heads split the channel dim."""
    _require_cuda(q, "sdpa")
    q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
    if flash_attention_usable(q, k, v, heads):
        if torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad):
            return _FlashSdpaFn.apply(q, k, v, int(heads), float(scale_))
        return flash_attention(q, k, v, int(heads), float(scale_))
    return _SdpaFn.apply(q, k, v, int(heads), float(scale_))


_FLASH = True
_FLASH_TRAIN = "auto"
_FLASH_TRAIN_BYTES = 2 << 30   # "auto": L x L buffers of the unfused chain above this size -> fused kernels regardless


def set_flash_attention(enabled: bool, training=None) -> None:
    """enabled: use the fused tcgen05 attention kernels at all. training (calls that need gradients): True = always the
    fused forward + backward (no L x L tensor), False = always the unfused GEMM + softmax chain, "auto" (default) = the
    faster of the two as measured on B200 (profiles/r02_attention_training.log):
      * head dim <= 256: fused (one pass, the accumulators of a whole head fit tensor memory: 3.6x faster at d = 128,
        L = 32768, and 8.6 GB of score buffers disappear);
      * head dim 512 / 768 (the LDM's single heads): the accumulators must be column-sliced and every slice recomputes
        Q K^T and dO V^T, which triples the tensor work -- the unfused chain is 2x faster at L = 1728..6400; the fused
        path is taken for short sequences (L <= 256, launch-bound: 9 kernels vs 3) and when the unfused chain's L x L
        buffers (12 bytes per score) would exceed 2 GiB."""
    global _FLASH, _FLASH_TRAIN
    _FLASH = bool(enabled)
    if training is not None:
        _FLASH_TRAIN = training if training == "auto" else bool(training)


def flash_attention_usable(q, k, v, heads: int, needs_grad=None) -> bool:
    """The fused tcgen05 kernels need bf16 and a head dim that is a multiple of 64 (above 256: a multiple of 256)."""
    if not _FLASH or _ENGINE == _lib.ENGINE_SIMT or q.dtype != torch.bfloat16:
        return False
    dh = q.shape[-1] // heads
    if dh % 64 != 0 or (dh > 256 and dh % 256 != 0) or q.shape[0] * heads >= 65536:
        return False
    if needs_grad is None:
        needs_grad = torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad)
    if needs_grad:
        if _FLASH_TRAIN is False:
            return False
        if _FLASH_TRAIN == "auto" and dh > 256:
            Lq, Lk = q.shape[1], k.shape[1]
            if Lq > 256 and q.shape[0] * heads * Lq * Lk * 12 <= _FLASH_TRAIN_BYTES:
                return False
    return bool(_lib.load().mig_has_tcgen05())


def _row_pitch(t):
    """Row pitch (elements) of a (B, L, C) matrix stack the strided attention entry point can read in place: unit column
    stride, rows `ld` apart, batches L * ld apart, 16-byte aligned -- e.g. a column block of a fused q/k/v projection
    output. None if `t` is laid out otherwise."""
    B, L, Cc = t.shape
    ld = t.stride(1) if L > 1 else max(t.stride(1), Cc)
    if t.stride(2) != 1 or ld < Cc or ld % 8 or (B > 1 and t.stride(0) != L * ld) or t.data_ptr() % 16:
        return None
    return ld


def _flash_fwd(q, k, v, heads: int, scale_: float):
    B, Lq, Cc = q.shape
    Lk = k.shape[1]
    lds = [_row_pitch(t) for t in (q, k, v)]
    if any(ld is None for ld in lds):
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        lds = [Cc, Cc, Cc]
    out = torch.empty((B, Lq, Cc), dtype=q.dtype, device=q.device)
    lse = torch.empty((B * heads, Lq), dtype=torch.float32, device=q.device)
    call("mig_flash_attention_fwd_ld", _ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(lse), B, heads, Lq, Lk, Cc // heads,
         int(lds[0]), int(lds[1]), int(lds[2]), float(scale_), _stream())
    return out, lse


def _flash_bwd(q, k, v, out, lse, dO, heads: int, scale_: float):
    """Gradients (dq, dk, dv) of _flash_fwd on contiguous q / k / v; dO contiguous in q's dtype."""
    B, Lq, Cc = q.shape
    Lk = k.shape[1]
    dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    delta = torch.empty((B * heads, Lq), dtype=torch.float32, device=q.device)
    call("mig_flash_attention_bwd", _ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(dO), _ptr(lse), _ptr(delta), _ptr(dq),
         _ptr(dk), _ptr(dv), B, heads, Lq, Lk, Cc // heads, float(scale_), _stream())
    return dq, dk, dv


def flash_attention(q, k, v, heads: int, scale_: float):
    """softmax(scale * q k^T) v without materialising the score matrix (unet:128-135 / 406-416). No autograd."""
    return _flash_fwd(q, k, v, heads, scale_)[0]


class _FlashSdpaFn(Function):
    """Training attention on the fused kernels: forward saves only O and the per-row log-sum-exp; backward recomputes P
    tile by tile (mig_flash_attention_bwd). No L x L tensor is ever allocated."""

    @staticmethod
    def forward(ctx, q, k, v, heads, scale_):
        out, lse = _flash_fwd(q, k, v, heads, scale_)
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.cfg = (heads, scale_)
        return out

    @staticmethod
    def backward(ctx, dO):
        q, k, v, out, lse = ctx.saved_tensors
        return (*_flash_bwd(q, k, v, out, lse, _grad_in(dO, q.dtype), *ctx.cfg), None, None)


# ----------------------------------------------------------------------------------------------
# timestep embedding, scheduler, losses
# ----------------------------------------------------------------------------------------------
def timestep_embedding(timesteps, dim: int, dtype=torch.float32, max_period: int = 10000):
    """unet:461-485 (cos first, then sin; odd dims zero-padded). No gradient flows to timesteps."""
    if timesteps.ndim != 1:
        raise ValueError("Timesteps should be a 1d-array")
    _require_cuda(timesteps, "timestep_embedding")
    t = timesteps.detach().float().contiguous()
    out = torch.empty((t.shape[0], dim), dtype=dtype, device=t.device)
    call("mig_timestep_embedding", _ptr(t), _ptr(out), _dt(out), t.shape[0], dim, float(max_period), _stream())
    return out


def _mse_forward(a, b, l1):
    """mean((a - b)^2), or mean |a - b| when l1, as an fp32 scalar; a and b share shape, dtype and strides."""
    out = torch.empty((), dtype=torch.float32, device=a.device)
    partials = torch.empty(2048, dtype=torch.float32, device=a.device)
    call("mig_mse_fwd", _dt(a), _ptr(a), _ptr(b), _ptr(out), _ptr(partials), a.numel(), int(l1), _stream())
    return out


def _mse_backward(a, b, l1, g):
    """Gradient w.r.t. a of _mse_forward, given the gradient g of the scalar."""
    g = g.float().contiguous()
    da = torch.empty_like(a)
    call("mig_mse_bwd", _dt(a), _ptr(a), _ptr(b), _ptr(g), _ptr(da), a.numel(), int(l1), _stream())
    return da


class _MseFn(Function):
    @staticmethod
    def forward(ctx, a, b, l1):
        ctx.save_for_backward(a, b)
        ctx.l1 = l1
        return _mse_forward(a, b, l1)

    @staticmethod
    def backward(ctx, g):
        return _mse_backward(*ctx.saved_tensors, ctx.l1, g), None, None


def _pair(a, b):
    if a.shape != b.shape:
        raise RuntimeError(f"loss: shape mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    if a.dtype not in (torch.float32, torch.bfloat16):
        a = a.float()
    b = b.to(a.dtype)
    if a.stride() != b.stride() or not (a.is_contiguous() or _is_cl(a)):
        a, b = a.contiguous(), b.contiguous()
    return a, b


def mse_loss(pred, target):
    """F.mse_loss(pred.float(), target.float()) (ldm:169): mean reduction, fp32 scalar. Grad flows to pred."""
    a, b = _pair(pred, target.detach())
    return _MseFn.apply(a, b, False)


def l1_loss(pred, target):
    """L1Loss()(pred.float(), target.float()) (aetrain:414)."""
    a, b = _pair(pred, target.detach())
    return _MseFn.apply(a, b, True)


class _KlFn(Function):
    @staticmethod
    def forward(ctx, mu, sigma):
        out = torch.empty((), dtype=torch.float32, device=mu.device)
        partials = torch.empty(2048, dtype=torch.float32, device=mu.device)
        call("mig_kl_fwd", _dt(mu), _ptr(mu), _ptr(sigma), _ptr(out), _ptr(partials), mu.numel(), mu.shape[0], _stream())
        ctx.save_for_backward(mu, sigma)
        return out

    @staticmethod
    def backward(ctx, g):
        mu, sigma = ctx.saved_tensors
        g = g.float().contiguous()
        dmu, dsig = torch.empty_like(mu), torch.empty_like(sigma)
        call("mig_kl_bwd", _dt(mu), _ptr(mu), _ptr(sigma), _ptr(g), _ptr(dmu), _ptr(dsig), mu.numel(), mu.shape[0],
             _stream())
        return dmu, dsig


def kl_loss(z_mu, z_sigma):
    """0.5*sum(mu^2 + sigma^2 - log(sigma^2) - 1) over non-batch dims, mean over batch (aetrain:67-72)."""
    a, b = _pair(z_mu, z_sigma)
    if not b.requires_grad and z_sigma.requires_grad:
        b = z_sigma.contiguous()
    return _KlFn.apply(a, b)


class _VaeSigmaFn(Function):
    """sigma = exp(clamp(logvar, -30, 20) / 2)  (ae:766-769); gradient is zero outside the clamp."""

    @staticmethod
    def forward(ctx, logvar):
        sigma = torch.empty_like(logvar)
        call("mig_vae_sample_fwd", _dt(logvar), None, _ptr(logvar), None, _ptr(sigma), None, logvar.numel(), _stream())
        ctx.save_for_backward(logvar, sigma)
        return sigma

    @staticmethod
    def backward(ctx, dsigma):
        logvar, sigma = ctx.saved_tensors
        if dsigma.stride() != sigma.stride():
            dsigma = as_cl(dsigma) if _is_cl(sigma) else dsigma.contiguous()
        if dsigma.dtype != sigma.dtype:
            dsigma = dsigma.to(sigma.dtype)
        dlv = torch.empty_like(sigma)
        call("mig_vae_sample_bwd", _dt(sigma), _ptr(logvar), None, _ptr(sigma), None, _ptr(dsigma), None, _ptr(dlv),
             sigma.numel(), _stream())
        return dlv


def vae_sigma(logvar):
    if not (logvar.is_contiguous() or _is_cl(logvar)):
        logvar = logvar.contiguous()
    return _VaeSigmaFn.apply(logvar)


class _ReparamFn(Function):
    """z = mu + eps * sigma (ae:786-787)."""

    @staticmethod
    def forward(ctx, mu, sigma, eps):
        z = torch.empty_like(mu)
        call("mig_addcmul", _dt(mu), _ptr(mu), _ptr(eps), _ptr(sigma), _ptr(z), mu.numel(), _stream())
        ctx.save_for_backward(eps)
        return z

    @staticmethod
    def backward(ctx, dz):
        (eps,) = ctx.saved_tensors
        if dz.stride() != eps.stride():
            dz = as_cl(dz) if _is_cl(eps) else dz.contiguous()
        if dz.dtype != eps.dtype:
            dz = dz.to(eps.dtype)
        dsigma = torch.empty_like(eps)
        call("mig_mul", _dt(eps), _ptr(dz), _ptr(eps), _ptr(dsigma), eps.numel(), _stream())
        return dz, dsigma, None


def vae_reparam(mu, sigma, eps):
    eps = eps.to(mu.dtype)
    if not (mu.stride() == sigma.stride() == eps.stride()) or not (mu.is_contiguous() or _is_cl(mu)):
        mu, sigma, eps = mu.contiguous(), sigma.contiguous(), eps.contiguous()
    return _ReparamFn.apply(mu, sigma, eps)
