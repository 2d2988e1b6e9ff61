"""CPU fp64 restatement of monai-generative's SSIM / MS-SSIM (`generative.metrics.SSIMMetric`, `MultiScaleSSIMMetric`;
their `compute_ssim_and_cs` and `compute_ms_ssim`).

TEST INFRASTRUCTURE (see oracle/__init__.py). PARITY UNPINNED: monai-generative is not installed here and not in the
reference tree, so this file restates its published algorithm from memory of the upstream source. Choices that memory
cannot settle are marked [upstream-memory]. Because parity is unpinned, tests/test_ssim.py anchors the restatement with
identities (SSIM(x, x) = 1, symmetry, the closed form for constant images, MS-SSIM with one weight = relu(SSIM)) and
with an independent scipy.ndimage implementation of the same valid filtering.

The dense path is upstream's: five depthwise `F.conv{2,3}d(..., groups=C)` with the full window, no padding ("valid"):
    mu_x, mu_y, E[x^2], E[y^2], E[xy];  sigma_x = E[x^2] - mu_x^2, sigma_y likewise, sigma_xy = E[xy] - mu_x mu_y
    cs   = (2 sigma_xy + c2) / (sigma_x + sigma_y + c2)
    ssim = (2 mu_x mu_y + c1) / (mu_x^2 + mu_y^2 + c1) * cs,       c1 = (k1 L)^2, c2 = (k2 L)^2, L = data_range
MS-SSIM: per scale relu(mean cs), at the last scale relu(mean ssim), then prod value_s ** w_s; each scale is
avg_pool(kernel_size=2) (floor) of the previous one. `separable=True` filters with the 1-D windows one axis after
another instead (the algorithm of csrc/ssim.cu); in fp64 the two agree to rounding.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

MS_SSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def _rep(v, n):
    return tuple(v) if isinstance(v, (list, tuple)) else (v,) * n


def window_1d(kernel_type: str, k: int, sigma: float = 1.5) -> torch.Tensor:
    """fp32 1-D window as upstream builds it: Gaussian at offsets (1-k)/2 ... (k-1)/2 normalised to sum 1, or 1/k."""
    if kernel_type == "gaussian":
        dist = torch.arange(start=(1 - k) / 2, end=(1 + k) / 2, step=1, dtype=torch.float32)
        gauss = torch.exp(-torch.pow(dist / sigma, 2) / 2)
        return gauss / gauss.sum()
    if kernel_type == "uniform":
        return torch.full((k,), 1.0 / k, dtype=torch.float32)
    raise ValueError(kernel_type)


def windows(spatial_dims, kernel_type, kernel_size, kernel_sigma):
    ks, sig = _rep(kernel_size, spatial_dims), _rep(kernel_sigma, spatial_dims)
    return [window_1d(kernel_type, int(k), float(s)).double() for k, s in zip(ks, sig)]


def dense_window(spatial_dims, kernel_type, kernel_size, kernel_sigma) -> torch.Tensor:
    """The full window, the outer product of the 1-D windows. [upstream-memory] upstream forms the product in fp32
    (`matmul` of the Gaussian rows, then a broadcast multiply for the third axis; `ones / prod(kernel_size)` for the
    uniform window); here it is formed in fp64 from the fp32 1-D windows -- within one fp32 ulp per tap of upstream,
    and exactly the window a separable filter with those taps applies."""
    w = windows(spatial_dims, kernel_type, kernel_size, kernel_sigma)
    out = w[0]
    for v in w[1:]:
        out = out[..., None] * v
    return out


def _filter_dense(x, win):
    Cc = x.shape[1]
    conv = F.conv3d if win.ndim == 3 else F.conv2d
    return conv(x, win.expand(Cc, 1, *win.shape).contiguous(), groups=Cc)


def _filter_separable(x, wins):
    Cc, nd = x.shape[1], len(wins)
    conv = F.conv3d if nd == 3 else F.conv2d
    for ax, w in enumerate(wins):
        shape = [1] * nd
        shape[ax] = w.numel()
        x = conv(x, w.view(1, 1, *shape).expand(Cc, 1, *shape).contiguous(), groups=Cc)
    return x


def ssim_and_cs_maps(y_pred, y, spatial_dims, kernel_type="gaussian", kernel_size=11, kernel_sigma=1.5,
                     data_range=1.0, k1=0.01, k2=0.03, separable=False):
    """(ssim map, cs map) in fp64, valid extent S - k + 1 per axis."""
    if y_pred.shape != y.shape:
        raise ValueError("y_pred and y must have the same shape")
    if y_pred.ndim != spatial_dims + 2:
        raise ValueError("wrong number of dimensions")
    x, y = y_pred.double(), y.double()
    if separable:
        wins = windows(spatial_dims, kernel_type, kernel_size, kernel_sigma)
        filt = lambda t: _filter_separable(t, wins)  # noqa: E731
    else:
        win = dense_window(spatial_dims, kernel_type, kernel_size, kernel_sigma)
        filt = lambda t: _filter_dense(t, win)  # noqa: E731
    c1, c2 = (k1 * data_range) ** 2, (k2 * data_range) ** 2
    mu_x, mu_y = filt(x), filt(y)
    mu_xx, mu_yy, mu_xy = filt(x * x), filt(y * y), filt(x * y)
    sigma_x = mu_xx - mu_x * mu_x
    sigma_y = mu_yy - mu_y * mu_y
    sigma_xy = mu_xy - mu_x * mu_y
    cs = (2 * sigma_xy + c2) / (sigma_x + sigma_y + c2)
    ssim = ((2 * mu_x * mu_y + c1) / (mu_x ** 2 + mu_y ** 2 + c1)) * cs
    return ssim, cs


def ssim(y_pred, y, spatial_dims, **kw) -> torch.Tensor:
    """(B,) fp64: SSIMMetric's per-item value, the mean of the SSIM map over channels and voxels."""
    s, _ = ssim_and_cs_maps(y_pred, y, spatial_dims, **kw)
    return s.reshape(s.shape[0], -1).mean(1)


def ms_ssim(y_pred, y, spatial_dims, weights=MS_SSIM_WEIGHTS, kernel_size=11, **kw) -> torch.Tensor:
    """(B,) fp64: MultiScaleSSIMMetric's per-item value.

    [upstream-memory] upstream's size check is written `S // max(1, len(weights) - 1) ** 2 <= k - 1`, which equals
    `S // 2 ** (len(weights) - 1) <= k - 1` for up to three weights and for the default five; this restatement uses the
    latter, the condition that the coarsest scale still holds the window. Upstream also pools once more after the last
    scale and discards the result; that pool is skipped."""
    if y_pred.shape != y.shape:
        raise ValueError("y_pred and y must have the same shape")
    if y_pred.ndim != spatial_dims + 2:
        raise ValueError("wrong number of dimensions")
    ks = _rep(kernel_size, spatial_dims)
    div = 2 ** (len(weights) - 1)
    for ax, s in enumerate(y_pred.shape[2:]):
        if s // div <= ks[ax] - 1:
            raise ValueError("image too small for the number of scales and the kernel size")
    pool = F.avg_pool3d if spatial_dims == 3 else F.avg_pool2d
    x, y = y_pred.double(), y.double()
    values = []
    for s in range(len(weights)):
        smap, cs = ssim_and_cs_maps(x, y, spatial_dims, kernel_size=kernel_size, **kw)
        values.append(torch.relu(cs.reshape(cs.shape[0], -1).mean(1)))
        if s < len(weights) - 1:
            x, y = pool(x, kernel_size=2), pool(y, kernel_size=2)
    values[-1] = torch.relu(smap.reshape(smap.shape[0], -1).mean(1))
    w = torch.tensor(weights, dtype=torch.float64).view(-1, 1)
    return torch.prod(torch.stack(values) ** w, dim=0)
