"""GPU: the fused SSIM kernel (mig_ssim_pairs, csrc/ssim.cu) and the public metrics (SSIMMetric, MultiScaleSSIMMetric,
pairwise_ms_ssim) against the fp64 oracle (oracle/ssim_oracle.py). Bar: 1e-4 absolute per item, the project's fp32 bar;
bf16 cases give the oracle the same bf16-rounded values."""
import ctypes as C

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

import medical_image_generation_b200 as mig
from medical_image_generation_b200 import _lib, compat, metrics, ops
from oracle import ssim_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4
I3 = C.c_int32 * 3


def _smooth(shape, rng, sigma=1.5):
    x = ndi.gaussian_filter(rng.standard_normal(shape), sigma=[0, 0] + [sigma] * (len(shape) - 2))
    return (x - x.min()) / (x.max() - x.min())


def _structured(shape, seed):
    """x: smoothed noise; y per item: x plus small noise, a contrast change, or a partly independent image, so the
    scores spread over (0, 1)."""
    rng = np.random.default_rng(seed)
    x = _smooth(shape, rng)
    other = _smooth(shape, rng, 2.0)
    y = np.empty_like(x)
    for n in range(shape[0]):
        kind = n % 3
        if kind == 0:
            y[n] = x[n] + 0.03 * rng.standard_normal(x[n].shape)
        elif kind == 1:
            y[n] = 0.6 * x[n] + 0.3 + 0.01 * rng.standard_normal(x[n].shape)
        else:
            y[n] = 0.5 * x[n] + 0.5 * other[n]
    return torch.from_numpy(x), torch.from_numpy(y)


def _device(t, dtype, cl):
    d = t.to(DEV, dtype)
    if cl:
        d = d.contiguous(memory_format=torch.channels_last_3d if t.ndim == 5 else torch.channels_last)
    return d, d.double().cpu()   # the device values, and exactly those values in fp64 for the oracle


# (shape, kwargs, dtype, channels-last)
SSIM_CASES = [
    ((3, 1, 37, 29, 23), dict(kernel_size=7), torch.float32, False),
    ((1, 2, 20, 18, 16), dict(), torch.bfloat16, True),
    ((3, 3, 16, 12, 13), dict(kernel_size=(4, 5, 11), kernel_sigma=(0.8, 1.5, 2.0), data_range=2.0, k1=0.02, k2=0.05),
     torch.float32, True),
    ((2, 1, 11, 11, 11), dict(), torch.float32, False),                       # valid extent 1 on every axis
    ((1, 2, 4, 40, 33), dict(kernel_size=4), torch.bfloat16, False),          # valid extent 1 along D
    ((2, 2, 19, 23, 21), dict(kernel_type="uniform", kernel_size=7), torch.bfloat16, False),
    ((3, 1, 40, 36, 30), dict(kernel_size=4, data_range=0.5), torch.float32, False),
    ((2, 1, 30, 70, 66), dict(kernel_size=16, kernel_sigma=3.0), torch.float32, True),
    ((3, 1, 37, 29), dict(), torch.float32, False),
    ((1, 3, 64, 50), dict(kernel_size=4), torch.bfloat16, True),
    ((2, 2, 30, 30), dict(kernel_type="uniform", kernel_size=8, k1=0.05, k2=0.1), torch.float32, True),
    ((1, 1, 11, 11), dict(), torch.bfloat16, False),
    ((3, 2, 45, 33), dict(kernel_size=(3, 9), kernel_sigma=(0.7, 2.2)), torch.float32, False),
]


@pytest.mark.parametrize("case", range(len(SSIM_CASES)))
def test_ssim_vs_oracle(case):
    shape, kw, dtype, cl = SSIM_CASES[case]
    sd = len(shape) - 2
    x, y = _structured(shape, 100 + case)
    xd, xo = _device(x, dtype, cl)
    yd, yo = _device(y, dtype, cl)
    got = metrics.SSIMMetric(sd, **kw)(xd, yd)
    assert got.shape == (shape[0], 1) and got.dtype == torch.float32 and got.device.type == "cuda"
    s_ref, cs_ref = O.ssim_and_cs_maps(xo, yo, sd, **kw)
    s_ref, cs_ref = s_ref.reshape(shape[0], -1).mean(1), cs_ref.reshape(shape[0], -1).mean(1)
    assert (got.double().cpu().view(-1) - s_ref).abs().max().item() < TOL
    s, cs = metrics.compute_ssim_and_cs(xd, yd, sd, **kw)
    assert (s.cpu() - s_ref).abs().max().item() < TOL
    assert (cs.cpu() - cs_ref).abs().max().item() < TOL


MS_CASES = [
    ((2, 1, 64, 64, 64), dict(kernel_size=4), torch.float32, False),
    ((3, 1, 64, 80, 72), dict(kernel_size=4), torch.bfloat16, True),
    ((3, 2, 96, 80), dict(kernel_size=5, weights=(0.5, 0.3, 0.2)), torch.float32, True),
    ((2, 1, 181, 177), dict(), torch.bfloat16, False),
    ((2, 1, 37, 29, 23), dict(kernel_size=7, weights=(1.0,)), torch.float32, False),
]


@pytest.mark.parametrize("case", range(len(MS_CASES)))
def test_ms_ssim_vs_oracle(case):
    shape, kw, dtype, cl = MS_CASES[case]
    sd = len(shape) - 2
    x, y = _structured(shape, 200 + case)
    xd, xo = _device(x, dtype, cl)
    yd, yo = _device(y, dtype, cl)
    got = metrics.MultiScaleSSIMMetric(sd, **kw)(xd, yd)
    assert got.shape == (shape[0], 1) and got.dtype == torch.float32
    want = O.ms_ssim(xo, yo, sd, **kw)
    assert (got.double().cpu().view(-1) - want).abs().max().item() < TOL
    anti = metrics.MultiScaleSSIMMetric(sd, **kw)(xd, (1.0 - xd.float()).to(dtype))
    assert (anti == 0).all()        # cs < 0 at the finest scale: the relu zeroes the product


def test_identity_symmetry_and_determinism():
    x, y = _structured((3, 2, 33, 31, 29), 7)
    for dtype in (torch.float32, torch.bfloat16):
        xd, yd = x.to(DEV, dtype), y.to(DEV, dtype)
        for m in (metrics.SSIMMetric(3), metrics.MultiScaleSSIMMetric(3, kernel_size=2, weights=(0.6, 0.4))):
            assert (m(xd, xd) - 1).abs().max().item() < 1e-6
            a = m(xd, yd)
            assert torch.equal(a, m(yd, xd))          # symmetric bit for bit
            assert torch.equal(a, m(xd, yd))          # repeatable bit for bit
    # a single pair whose tiles cannot fill the machine: the D axis is split into chunks, the result still repeats
    x, y = _structured((1, 1, 128, 128, 64), 8)
    xd, yd = x.to(DEV, torch.bfloat16), y.to(DEV, torch.bfloat16)
    s1, cs1 = metrics.compute_ssim_and_cs(xd, yd, 3, kernel_size=4)
    s2, cs2 = metrics.compute_ssim_and_cs(xd, yd, 3, kernel_size=4)
    assert torch.equal(s1, s2) and torch.equal(cs1, cs2)
    s_ref = O.ssim(xd.double().cpu(), yd.double().cpu(), 3, kernel_size=4, separable=True)
    assert abs(s1.item() - s_ref.item()) < TOL


def _diverse_samples(n, shape, seed):
    """n volumes sharing structure in varying proportions: pairwise MS-SSIM spreads over (0, 1)."""
    rng = np.random.default_rng(seed)
    base = _smooth((1, 1) + shape, rng, 2.0)
    own = _smooth((n, 1) + shape, rng, 2.0)
    w = np.linspace(0.1, 0.9, n).reshape(-1, 1, 1, 1, 1)
    return torch.from_numpy(w * base + (1 - w) * own)


def test_pairwise_ms_ssim_config4():
    """8 volumes of config-4 size (1x128x128x64, bf16), kernel_size 4: 28 pairs in one launch per scale."""
    x = _diverse_samples(8, (128, 128, 64), 9)
    xd, xo = _device(x, torch.bfloat16, False)
    got = metrics.pairwise_ms_ssim(xd, kernel_size=4)
    assert got.shape == (28,) and got.dtype == torch.float32
    I, J = torch.triu_indices(8, 8, 1)
    m = metrics.MultiScaleSSIMMetric(3, kernel_size=4)
    per_pair = torch.cat([m(xd[i:i + 1], xd[j:j + 1]).view(-1) for i, j in zip(I.tolist(), J.tolist())])
    assert (got - per_pair).abs().max().item() < 1e-6
    want = torch.cat([O.ms_ssim(xo[I[s:s + 7]], xo[J[s:s + 7]], 3, kernel_size=4, separable=True)
                      for s in range(0, 28, 7)])
    assert (got.double().cpu() - want).abs().max().item() < TOL
    assert want.max() > want.min() + 0.1
    sub = metrics.pairwise_ms_ssim(xd, pairs=[[0, 7], [3, 3], [5, 1]], kernel_size=4)
    k = {(i, j): p for p, (i, j) in enumerate(zip(I.tolist(), J.tolist()))}
    assert abs(sub[0].item() - got[k[(0, 7)]].item()) < 1e-6
    assert abs(sub[1].item() - 1.0) < 1e-6
    assert abs(sub[2].item() - got[k[(1, 5)]].item()) < 1e-6
    with pytest.raises(ValueError):
        metrics.pairwise_ms_ssim(xd, pairs=[[0, 8]], kernel_size=4)


def test_ssim_config5_patch():
    x, y = _structured((1, 1, 160, 160, 128), 10)
    xd, xo = _device(x, torch.float32, False)
    yd, yo = _device(y, torch.float32, False)
    got = mig.SSIMMetric(3)(xd, yd)
    want = O.ssim(xo, yo, 3, separable=True)
    assert abs(got.item() - want.item()) < TOL


def test_aggregate_and_reset():
    x, y = _structured((5, 1, 24, 24, 24), 11)
    xd, yd = x.to(DEV, torch.float32), y.to(DEV, torch.float32)
    m = metrics.SSIMMetric(3, kernel_size=5)
    a, b = m(xd[:2], yd[:2]), m(xd[2:], yd[2:])
    allv = torch.cat([a, b])
    assert torch.equal(m.get_buffer(), allv)
    assert torch.allclose(m.aggregate(), allv.mean())
    assert torch.allclose(m.aggregate("sum"), allv.sum())
    assert torch.equal(m.aggregate("none"), allv)
    assert metrics.SSIMMetric(3, kernel_size=5, reduction="sum")(xd, yd).shape == (5, 1)
    m.reset()
    with pytest.raises(ValueError):
        m.aggregate()
    m(xd[:1], yd[:1])
    assert m.aggregate("none").shape == (1, 1)


def _abi_operands():
    x, y = _structured((2, 1, 12, 12, 12), 12)
    a = x.to(DEV, torch.float32).contiguous()
    b = y.to(DEV, torch.float32).contiguous()
    pairs = torch.tensor([[0, 0], [1, 1], [0, 2]], dtype=torch.int32, device=DEV)
    taps = np.concatenate([t.numpy() for t in metrics.window_taps(3, "gaussian", 4, 1.5)]).astype(np.float32)
    return a, b, pairs, taps


def test_ssim_pairs_abi_and_rejections():
    a, b, pairs, taps = _abi_operands()
    lib = _lib.load()
    dims, ks = I3(12, 12, 12), I3(4, 4, 4)
    nbytes = lib.mig_ssim_workspace_bytes(3, 1, dims, ks)
    assert nbytes > 0
    assert lib.mig_ssim_workspace_bytes(3, 1, dims, I3(4, 13, 4)) == -1
    assert lib.mig_ssim_workspace_bytes(3, 0, dims, ks) == -1
    assert lib.mig_ssim_workspace_bytes(3, 1, dims, I3(17, 4, 4)) == -1
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    out = torch.empty(3, 2, dtype=torch.float64, device=DEV)
    tp = taps.ctypes.data_as(C.c_void_p)
    c1, c2 = 1e-4, 9e-4

    def run(**over):
        args = dict(dtype=_lib.F32, a=ops._ptr(a), b=ops._ptr(b), na=2, nb=2, pairs=ops._ptr(pairs), P=3, dims=dims,
                    C=1, ks=ks, taps=tp, out=ops._ptr(out), ws=ops._ptr(ws), nbytes=nbytes)
        args.update(over)
        _lib.call("mig_ssim_pairs", args["dtype"], args["a"], args["b"], args["na"], args["nb"], args["pairs"],
                  args["P"], args["dims"], args["C"], args["ks"], args["taps"], c1, c2, args["out"], args["ws"],
                  args["nbytes"], ops._stream())

    run()
    got = out.cpu()
    want = O.ssim_and_cs_maps(a.double().cpu(), b.double().cpu(), 3, kernel_size=4)
    assert (got[:2, 0] - want[0].reshape(2, -1).mean(1)).abs().max() < TOL
    assert (got[:2, 1] - want[1].reshape(2, -1).mean(1)).abs().max() < TOL
    assert torch.isnan(got[2]).all()          # pair (0, 2): index 2 is outside b
    for over, msg in [(dict(a=None), "must not be NULL"), (dict(pairs=None), "must not be NULL"),
                      (dict(out=None), "must not be NULL"), (dict(taps=None), "must not be NULL"),
                      (dict(C=0), "C must be positive"), (dict(ks=I3(4, 13, 4)), "k <= the extent"),
                      (dict(ks=I3(0, 4, 4)), "1 <= k"), (dict(na=0), "na, nb > 0"),
                      (dict(nbytes=nbytes - 1), "workspace too small"), (dict(ws=None), "workspace too small"),
                      (dict(dtype=7), "unsupported dtype")]:
        with pytest.raises(RuntimeError, match=msg):
            run(**over)
    run(P=0, a=None, b=None, pairs=None, out=None, ws=None, nbytes=0)   # no pairs: nothing to do
    torch.cuda.synchronize()


def test_generative_shim_metrics():
    import importlib.util
    if importlib.util.find_spec("generative") is not None and "shims" not in importlib.util.find_spec(
            "generative").origin:
        pytest.skip("a real monai-generative is installed")
    compat.install()
    try:
        from generative.metrics import FIDMetric, MultiScaleSSIMMetric, SSIMMetric
        assert SSIMMetric is mig.SSIMMetric and MultiScaleSSIMMetric is mig.MultiScaleSSIMMetric
        x, y = _structured((2, 1, 20, 20, 20), 13)
        v = SSIMMetric(spatial_dims=3)(x.to(DEV, torch.float32), y.to(DEV, torch.float32))
        assert v.shape == (2, 1) and v.is_cuda
        with pytest.raises(NotImplementedError):
            FIDMetric()
    finally:
        compat.uninstall()
