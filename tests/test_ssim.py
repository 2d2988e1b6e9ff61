"""CPU: the fp64 SSIM / MS-SSIM oracle (oracle/ssim_oracle.py), which no reference pins, checked against identities and
against an independent scipy.ndimage implementation; the host-side window taps and argument checks of the metrics."""
import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

from medical_image_generation_b200 import metrics
from oracle import ssim_oracle as O


def _smooth(shape, seed, sigma=1.5):
    """Smoothed noise in [0, 1]-ish: structured data whose SSIM spreads over (0, 1)."""
    rng = np.random.default_rng(seed)
    x = ndi.gaussian_filter(rng.standard_normal(shape), sigma=[0, 0] + [sigma] * (len(shape) - 2))
    x = (x - x.min()) / (x.max() - x.min())
    return torch.from_numpy(x)


def _pair(shape, seed, noise=0.05):
    x = _smooth(shape, seed)
    rng = np.random.default_rng(seed + 1000)
    y = 0.8 * x + 0.1 + noise * torch.from_numpy(rng.standard_normal(shape))
    return x, y


WINDOWS = [
    (3, "gaussian", 11, 1.5),
    (3, "gaussian", 4, 1.5),
    (3, "gaussian", (5, 7, 4), (0.8, 1.5, 2.0)),
    (3, "uniform", 7, 1.5),
    (3, "uniform", (3, 4, 6), 1.5),
    (2, "gaussian", 11, 1.5),
    (2, "gaussian", (6, 9), (1.0, 2.5)),
    (2, "uniform", 8, 1.5),
]


@pytest.mark.parametrize("sd,kt,ks,sig", WINDOWS)
def test_separable_equals_dense(sd, kt, ks, sig):
    shape = (2, 2) + ((15, 17, 19) if sd == 3 else (23, 21))
    x, y = _pair(shape, 1)
    kw = dict(kernel_type=kt, kernel_size=ks, kernel_sigma=sig, data_range=1.3, k1=0.02, k2=0.05)
    d = O.ssim_and_cs_maps(x, y, sd, **kw)
    s = O.ssim_and_cs_maps(x, y, sd, separable=True, **kw)
    for a, b in zip(d, s):
        assert a.shape == b.shape
        assert (a - b).abs().max().item() < 1e-12


def _valid_filter_scipy(v: np.ndarray, wins) -> np.ndarray:
    """Valid correlation of one (*spatial) array with 1-D windows along each axis, via ndimage.correlate1d."""
    for ax, w in enumerate(wins):
        k = len(w)
        full = ndi.correlate1d(v, w, axis=ax, mode="constant", cval=0.0)
        # correlate1d centres the window at k // 2: output i reads input i + t - k // 2
        idx = [slice(None)] * v.ndim
        idx[ax] = slice(k // 2, k // 2 + v.shape[ax] - k + 1)
        v = full[tuple(idx)]
    return v


@pytest.mark.parametrize("sd,kt,ks,sig", WINDOWS)
def test_oracle_matches_scipy(sd, kt, ks, sig):
    shape = (2, 2) + ((14, 16, 13) if sd == 3 else (20, 18))
    x, y = _pair(shape, 2)
    kw = dict(kernel_type=kt, kernel_size=ks, kernel_sigma=sig, data_range=1.0, k1=0.01, k2=0.03)
    smap, cmap = O.ssim_and_cs_maps(x, y, sd, **kw)
    wins = [w.numpy() for w in O.windows(sd, kt, ks, sig)]
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    for n in range(shape[0]):
        for c in range(shape[1]):
            xv, yv = x[n, c].numpy(), y[n, c].numpy()
            f = lambda v: _valid_filter_scipy(v, wins)  # noqa: E731
            mx, my, exx, eyy, exy = f(xv), f(yv), f(xv * xv), f(yv * yv), f(xv * yv)
            vx, vy, vxy = exx - mx ** 2, eyy - my ** 2, exy - mx * my
            cs = (2 * vxy + c2) / (vx + vy + c2)
            ss = (2 * mx * my + c1) / (mx ** 2 + my ** 2 + c1) * cs
            assert np.abs(cmap[n, c].numpy() - cs).max() < 1e-12
            assert np.abs(smap[n, c].numpy() - ss).max() < 1e-12


def test_valid_extent():
    x, y = _pair((1, 1, 12, 10, 9), 3)
    s, _ = O.ssim_and_cs_maps(x, y, 3, kernel_size=(4, 3, 9))
    assert s.shape == (1, 1, 9, 8, 1)


def test_identity_and_symmetry():
    x, y = _pair((3, 2, 16, 15, 14), 4)
    assert torch.allclose(O.ssim(x, x, 3), torch.ones(3, dtype=torch.float64), atol=1e-14, rtol=0)
    assert torch.allclose(O.ssim(x, y, 3, kernel_size=5), O.ssim(y, x, 3, kernel_size=5), atol=1e-14, rtol=0)
    v = O.ssim(x, y, 3, kernel_size=5)
    assert ((v > 0.05) & (v < 0.99)).all()


@pytest.mark.parametrize("a,b,L", [(0.3, 0.7, 1.0), (0.0, 0.5, 1.0), (2.0, 3.0, 4.0)])
def test_constant_images(a, b, L):
    """(2ab + c1) / (a^2 + b^2 + c1) for a window summing to 1 (uniform, 4 taps: exactly 1/4 in fp32). The fp32
    Gaussian sums to S = 1 +- 1e-7 instead: mu = aS and sigma_x = a^2 S (1 - S) != 0, which the closed form includes.
    Bar 1e-10: E[x^2] - mu^2 cancels to ~1e-16 in fp64, and cs divides it by c2 ~ 1e-3."""
    x = torch.full((1, 1, 12, 12, 12), a, dtype=torch.float64)
    y = torch.full((1, 1, 12, 12, 12), b, dtype=torch.float64)
    c1, c2 = (0.01 * L) ** 2, (0.03 * L) ** 2
    want = (2 * a * b + c1) / (a * a + b * b + c1)
    for sep in (False, True):
        assert abs(O.ssim(x, y, 3, kernel_type="uniform", kernel_size=4, data_range=L, separable=sep).item()
                   - want) < 1e-10
    S = O.dense_window(3, "gaussian", 5, 1.5).sum().item()
    v = S * (1 - S)
    cs = (2 * a * b * v + c2) / ((a * a + b * b) * v + c2)
    want = (2 * a * b * S * S + c1) / ((a * a + b * b) * S * S + c1) * cs
    assert abs(O.ssim(x, y, 3, kernel_size=5, data_range=L).item() - want) < 1e-10


def test_ms_ssim_one_weight_is_relu_ssim():
    x, y = _pair((2, 1, 20, 20, 18), 5)
    for yy in (y, 1.0 - x):
        want = torch.relu(O.ssim(x, yy, 3, kernel_size=5))
        assert torch.allclose(O.ms_ssim(x, yy, 3, weights=(1.0,), kernel_size=5), want, atol=1e-14, rtol=0)


def test_anticorrelated_pair_gives_zero_ms_ssim():
    """y = c - x: cs < 0 at every scale, the relu makes the product 0."""
    x = _smooth((2, 1, 64, 64, 64), 6)
    v = O.ms_ssim(x, 1.0 - x, 3, kernel_size=4)
    assert (v == 0).all()
    _, cs = O.ssim_and_cs_maps(x, 1.0 - x, 3, kernel_size=4)
    assert cs.reshape(2, -1).mean(1).max() < 0


def test_ms_ssim_of_identical_images_is_one():
    x = _smooth((2, 2, 48, 48), 7)
    assert torch.allclose(O.ms_ssim(x, x, 2, kernel_size=3), torch.ones(2, dtype=torch.float64), atol=1e-13, rtol=0)


@pytest.mark.parametrize("sd,kt,ks,sig", WINDOWS)
def test_host_taps_equal_oracle_window(sd, kt, ks, sig):
    mine = metrics.window_taps(sd, kt, ks, sig)
    ref = O.windows(sd, kt, ks, sig)
    assert len(mine) == sd
    for a, b in zip(mine, ref):
        assert a.dtype == torch.float32
        assert torch.equal(a.double(), b)
        assert abs(a.double().sum().item() - 1.0) < 1e-6


def test_even_window_is_centred_between_voxels():
    w = metrics.window_taps(1, "gaussian", 4, 1.5)[0]
    assert torch.equal(w, w.flip(0))
    assert w[1] > w[0] and w[1] == w[2]


def test_value_errors():
    x = torch.zeros(1, 1, 8, 8, 8)
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3)(x, torch.zeros(1, 1, 8, 8, 7))
    with pytest.raises(ValueError):
        metrics.SSIMMetric(2)(x, x)
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3)(x, x.bfloat16())
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3, kernel_type="box")
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3, kernel_size=17)
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3, kernel_size=(3, 3))
    with pytest.raises(ValueError):
        metrics.SSIMMetric(3, reduction="median")
    with pytest.raises(ValueError):
        metrics.SSIMMetric(4)
    # MS-SSIM: the coarsest of 5 scales (S // 16) must hold the window
    m = metrics.MultiScaleSSIMMetric(3, kernel_size=4)
    m.check_size((128, 128, 64))
    with pytest.raises(ValueError):
        m.check_size((128, 128, 63))
    with pytest.raises(ValueError):
        metrics.MultiScaleSSIMMetric(3)(x, x)
    with pytest.raises(ValueError):
        O.ms_ssim(torch.zeros(1, 1, 128, 128, 63), torch.zeros(1, 1, 128, 128, 63), 3, kernel_size=4)
    with pytest.raises(ValueError):
        O.ssim(x, torch.zeros(1, 1, 8, 8, 7), 3)


def test_cpu_tensors_are_refused():
    x = torch.zeros(1, 1, 16, 16, 16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        metrics.SSIMMetric(3, kernel_size=4)(x, x)
    with pytest.raises(RuntimeError, match="no CPU path"):
        metrics.pairwise_ms_ssim(torch.zeros(3, 1, 64, 64), kernel_size=4)
