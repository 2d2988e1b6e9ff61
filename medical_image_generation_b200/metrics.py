"""SSIM and multi-scale SSIM for 2-D and 3-D images: monai-generative's `generative.metrics.SSIMMetric` and
`MultiScaleSSIMMetric` (validation of reconstructions and samples, train_ldm.py:241-330), plus `pairwise_ms_ssim`, the
mean-MS-SSIM-over-sample-pairs diversity score of generative models.

Every SSIM evaluation runs `mig_ssim_pairs` (csrc/ssim.cu): the Gaussian or uniform window is an outer product of 1-D
windows, so the five local moments are filtered separably (5 x (kd + kh + kw) multiply-adds per output voxel instead
of upstream's 5 x kd*kh*kw dense depthwise convolutions) and reduced to per-pair means on chip. MS-SSIM scales are
built with the 2x average pool of the U-Net (`mig_avgpool_fwd`, floor, as upstream's avg_pool(kernel_size=2)). The
window taps are computed on the host exactly as upstream computes them (fp32). CUDA tensors only: there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Union

import numpy as np
import torch

from . import _lib, ops
from ._lib import call

MS_SSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)
KERNEL_MAX = 16  # longest 1-D window the kernel takes per axis
_REDUCTIONS = ("mean", "sum", "none")


def _per_axis(v, n: int, name: str) -> tuple:
    t = tuple(v) if isinstance(v, Sequence) else (v,) * n
    if len(t) != n:
        raise ValueError(f"{name} must have {n} entries (one per spatial axis), got {t}")
    return t


def _gaussian_1d(k: int, sigma: float) -> torch.Tensor:
    """Upstream's 1-D window: the Gaussian at offsets (1-k)/2 ... (k-1)/2 (between voxels for even k), sum 1, fp32."""
    dist = torch.arange(start=(1 - k) / 2, end=(1 + k) / 2, step=1, dtype=torch.float32)
    gauss = torch.exp(-torch.pow(dist / sigma, 2) / 2)
    return gauss / gauss.sum()


def window_taps(spatial_dims: int, kernel_type: str = "gaussian", kernel_size=11, kernel_sigma=1.5) -> list:
    """Per-axis 1-D windows (fp32 tensors, spatial axes in order) whose outer product is upstream's dense window."""
    ks = tuple(int(k) for k in _per_axis(kernel_size, spatial_dims, "kernel_size"))
    if any(k < 1 or k > KERNEL_MAX for k in ks):
        raise ValueError(f"kernel_size must lie in 1..{KERNEL_MAX} per axis, got {ks}")
    if kernel_type == "gaussian":
        sig = tuple(float(s) for s in _per_axis(kernel_sigma, spatial_dims, "kernel_sigma"))
        return [_gaussian_1d(k, s) for k, s in zip(ks, sig)]
    if kernel_type == "uniform":
        return [torch.full((k,), 1.0 / k, dtype=torch.float32) for k in ks]
    raise ValueError(f"kernel_type must be 'gaussian' or 'uniform', got {kernel_type!r}")


def _check_pair(y_pred: torch.Tensor, y: torch.Tensor, spatial_dims: int) -> None:
    if y_pred.shape != y.shape:
        raise ValueError(f"y_pred and y must have the same shape, got {tuple(y_pred.shape)} and {tuple(y.shape)}")
    if y_pred.ndim != spatial_dims + 2:
        raise ValueError(f"y_pred should have {spatial_dims + 2} dimensions (batch, channel, {spatial_dims} spatial) "
                         f"when using {spatial_dims} spatial dimensions, got {y_pred.ndim}")
    if y_pred.dtype != y.dtype:
        raise ValueError(f"y_pred and y must have the same dtype, got {y_pred.dtype} and {y.dtype}")


def _channels_last(x: torch.Tensor, what: str) -> torch.Tensor:
    ops._require_cuda(x, what)
    ops._dt(x)
    x = x.detach()
    return x if ops._is_cl(x) else ops.as_cl(x)


def _pair_stats(a: torch.Tensor, b: torch.Tensor, pairs: torch.Tensor, taps: list, c1: float, c2: float):
    """(P, 2) fp64 (mean ssim, mean cs) of the pairs (a[i], b[j]); a, b channels-last (N, C, *spatial)."""
    P, Cc = pairs.shape[0], a.shape[1]
    pad = 3 - len(taps)
    dims = ops._sp3(a.shape[2:])
    I3 = C.c_int32 * 3
    ks = I3(*((1,) * pad + tuple(t.numel() for t in taps)))
    for ax, (s, k) in enumerate(zip(a.shape[2:], taps)):
        if s < k.numel():
            raise ValueError(f"kernel_size {k.numel()} is larger than spatial axis {ax} of the input ({s})")
    nbytes = _lib.load().mig_ssim_workspace_bytes(P, Cc, I3(*dims), ks)
    out = torch.empty((P, 2), dtype=torch.float64, device=a.device)
    ws = ops._workspace(nbytes, a.device)
    flat = np.concatenate([np.ones(pad, np.float32)] + [t.numpy() for t in taps]).astype(np.float32)
    call("mig_ssim_pairs", ops._dt(a), ops._ptr(a), ops._ptr(b), a.shape[0], b.shape[0], ops._ptr(pairs), P,
         I3(*dims), Cc, ks, flat.ctypes.data_as(C.c_void_p), float(c1), float(c2), ops._ptr(out), ops._ptr(ws),
         ws.numel(), ops._stream())
    return out


def _pool(x: torch.Tensor) -> torch.Tensor:
    """One MS-SSIM scale down: 2x average pool, floor. The pyramid is kept in fp32 (a bf16 input is widened once)."""
    if x.dtype != torch.float32:
        x = ops.to_channels_last(x, torch.float32)
    return ops.avg_pool(x, 2, 2)


def _ms_ssim(a, b, pairs, taps, weights, c1, c2) -> torch.Tensor:
    """(P,) fp64 MS-SSIM of the pairs: prod_s value_s ** w_s, value = relu(mean cs), relu(mean ssim) at the last scale.
    a is b (the pairwise case) builds one pyramid."""
    values = []
    for s in range(len(weights)):
        st = _pair_stats(a, b, pairs, taps, c1, c2)
        values.append(torch.relu(st[:, 0] if s == len(weights) - 1 else st[:, 1]))
        if s < len(weights) - 1:
            same = a is b
            a = _pool(a)
            b = a if same else _pool(b)
    w = torch.tensor(weights, dtype=torch.float64, device=pairs.device).view(-1, 1)
    return torch.prod(torch.stack(values) ** w, dim=0)


def _diagonal_pairs(B: int, device) -> torch.Tensor:
    i = torch.arange(B, dtype=torch.int32, device=device)
    return torch.stack([i, i], dim=1)


def compute_ssim_and_cs(y_pred: torch.Tensor, y: torch.Tensor, spatial_dims: int, kernel_size=11,
                        kernel_sigma=1.5, data_range: float = 1.0, kernel_type: str = "gaussian", k1: float = 0.01,
                        k2: float = 0.03):
    """Per-item means of upstream's SSIM map and contrast-structure map: two (B,) fp64 tensors (the maps themselves
    are never formed)."""
    _check_pair(y_pred, y, spatial_dims)
    taps = window_taps(spatial_dims, kernel_type, kernel_size, kernel_sigma)
    a, b = _channels_last(y_pred, "compute_ssim_and_cs"), _channels_last(y, "compute_ssim_and_cs")
    st = _pair_stats(a, b, _diagonal_pairs(a.shape[0], a.device), taps, (k1 * data_range) ** 2,
                     (k2 * data_range) ** 2)
    return st[:, 0], st[:, 1]


class _CumulativeMetric:
    """Buffer of per-item values with MONAI's aggregate / reset semantics (NaN items are ignored by the reduction)."""

    def __init__(self, spatial_dims: int, data_range: float, kernel_type: str, kernel_size, kernel_sigma, k1: float,
                 k2: float, reduction: str):
        if spatial_dims not in (2, 3):
            raise ValueError(f"spatial_dims must be 2 or 3, got {spatial_dims}")
        if reduction not in _REDUCTIONS:
            raise ValueError(f"reduction must be one of {_REDUCTIONS}, got {reduction!r}")
        self.spatial_dims, self.data_range, self.kernel_type = spatial_dims, float(data_range), kernel_type
        self.kernel_size = _per_axis(kernel_size, spatial_dims, "kernel_size")
        self.kernel_sigma = _per_axis(kernel_sigma, spatial_dims, "kernel_sigma")
        self.k1, self.k2, self.reduction = float(k1), float(k2), reduction
        self.taps = window_taps(spatial_dims, kernel_type, self.kernel_size, self.kernel_sigma)
        self.c1, self.c2 = (self.k1 * self.data_range) ** 2, (self.k2 * self.data_range) ** 2
        self._buffer: list = []

    def __call__(self, y_pred: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        """(B, 1) fp32 per-item values on the inputs' device; also appended to the buffer."""
        _check_pair(y_pred, y, self.spatial_dims)
        self.check_size(y_pred.shape[2:])
        a, b = _channels_last(y_pred, type(self).__name__), _channels_last(y, type(self).__name__)
        v = self._values(a, b, _diagonal_pairs(a.shape[0], a.device)).float().view(-1, 1)
        self._buffer.append(v)
        return v

    def reset(self) -> None:
        self._buffer = []

    def get_buffer(self) -> Optional[torch.Tensor]:
        return torch.cat(self._buffer) if self._buffer else None

    def aggregate(self, reduction: Optional[str] = None) -> torch.Tensor:
        """'mean' / 'sum' of the buffered values (NaN items ignored) as a 0-d tensor, 'none': the (N, 1) buffer."""
        red = reduction or self.reduction
        if red not in _REDUCTIONS:
            raise ValueError(f"reduction must be one of {_REDUCTIONS}, got {red!r}")
        data = self.get_buffer()
        if data is None:
            raise ValueError(f"{type(self).__name__}.aggregate: no values have been accumulated")
        if red == "none":
            return data
        ok = ~torch.isnan(data)
        total = torch.where(ok, data, torch.zeros_like(data)).sum()
        return total if red == "sum" else total / ok.sum()


class SSIMMetric(_CumulativeMetric):
    """generative.metrics.SSIMMetric: per item, the mean over channels and valid voxels of the SSIM map."""

    def __init__(self, spatial_dims: int, data_range: float = 1.0, kernel_type: str = "gaussian",
                 kernel_size: Union[int, Sequence[int]] = 11, kernel_sigma: Union[float, Sequence[float]] = 1.5,
                 k1: float = 0.01, k2: float = 0.03, reduction: str = "mean"):
        super().__init__(spatial_dims, data_range, kernel_type, kernel_size, kernel_sigma, k1, k2, reduction)

    def check_size(self, spatial_shape) -> None:
        for ax, s in enumerate(spatial_shape):
            if s < self.kernel_size[ax]:
                raise ValueError(f"kernel_size {self.kernel_size[ax]} is larger than spatial axis {ax} ({s})")

    def _values(self, a, b, pairs):
        return _pair_stats(a, b, pairs, self.taps, self.c1, self.c2)[:, 0]


class MultiScaleSSIMMetric(_CumulativeMetric):
    """generative.metrics.MultiScaleSSIMMetric: prod over scales of value_s ** weights[s], value = relu(mean cs) at
    every scale but the last, relu(mean ssim) at the last; each scale is the previous one 2x average-pooled."""

    def __init__(self, spatial_dims: int, data_range: float = 1.0, kernel_type: str = "gaussian",
                 kernel_size: Union[int, Sequence[int]] = 11, kernel_sigma: Union[float, Sequence[float]] = 1.5,
                 k1: float = 0.01, k2: float = 0.03, weights: Sequence[float] = MS_SSIM_WEIGHTS,
                 reduction: str = "mean"):
        super().__init__(spatial_dims, data_range, kernel_type, kernel_size, kernel_sigma, k1, k2, reduction)
        if len(weights) < 1:
            raise ValueError("weights must not be empty")
        self.weights = tuple(float(w) for w in weights)

    def check_size(self, spatial_shape) -> None:
        """ValueError unless every axis still holds the window at the coarsest scale (upstream's check)."""
        div = 2 ** (len(self.weights) - 1)
        for ax, s in enumerate(spatial_shape):
            if s // div <= self.kernel_size[ax] - 1:
                raise ValueError(f"for a kernel size of {self.kernel_size[ax]} and {len(self.weights)} scales, spatial "
                                 f"axis {ax} must be larger than {(self.kernel_size[ax] - 1) * div}, got {s}")

    def _values(self, a, b, pairs):
        return _ms_ssim(a, b, pairs, self.taps, self.weights, self.c1, self.c2)


def pairwise_ms_ssim(samples: torch.Tensor, pairs=None, **ms_ssim_kwargs) -> torch.Tensor:
    """MS-SSIM of pairs of samples (N, C, *spatial): a (P,) fp32 tensor; the sample-diversity score is its mean.

    `pairs`: (P, 2) indices into `samples`, default every i < j. `ms_ssim_kwargs` are MultiScaleSSIMMetric's
    arguments (`spatial_dims` defaults to samples.ndim - 2). Each sample's scale pyramid is built once and every scale is
    one launch over the whole pair table; pair p equals MultiScaleSSIMMetric on (samples[i:i+1], samples[j:j+1])."""
    kw = dict(ms_ssim_kwargs)
    kw.setdefault("spatial_dims", samples.ndim - 2)
    metric = MultiScaleSSIMMetric(**kw)
    if samples.ndim != metric.spatial_dims + 2:
        raise ValueError(f"samples should have {metric.spatial_dims + 2} dimensions, got {samples.ndim}")
    metric.check_size(samples.shape[2:])
    x = _channels_last(samples, "pairwise_ms_ssim")
    N = x.shape[0]
    if pairs is None:
        table = torch.triu_indices(N, N, 1, device=x.device).t().to(torch.int32).contiguous()
    else:
        p = torch.as_tensor(pairs)
        if p.ndim != 2 or p.shape[1] != 2:
            raise ValueError(f"pairs must have shape (P, 2), got {tuple(p.shape)}")
        if not p.is_cuda and p.numel() and (int(p.min()) < 0 or int(p.max()) >= N):
            raise ValueError(f"pair indices must lie in [0, {N}), got {int(p.min())}..{int(p.max())}")
        table = p.to(device=x.device, dtype=torch.int32).contiguous()
    if table.shape[0] == 0:
        return torch.empty(0, dtype=torch.float32, device=x.device)
    return _ms_ssim(x, x, table, metric.taps, metric.weights, metric.c1, metric.c2).float()


__all__ = ["SSIMMetric", "MultiScaleSSIMMetric", "pairwise_ms_ssim", "compute_ssim_and_cs", "window_taps",
           "MS_SSIM_WEIGHTS"]
