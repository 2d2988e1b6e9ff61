"""GPU: every C-ABI operator against a plain PyTorch fp32 CPU reference of the same op.
fp32 path within 1e-4 relative error, bf16 path within 2e-2 (tolerances from BASELINE.json north_star)."""
import math

import pytest
import torch
import torch.nn.functional as F

from util import BF16_TOL, FP32_TOL, bf16_round, rel_err, tol_for

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _ops():
    from medical_image_generation_b200 import ops
    return ops


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last_3d if t.ndim == 5 else torch.channels_last)


# (N, Cin, Cout, spatial, kernel, stride, pad)
CONV_CASES = [
    (2, 16, 32, (6, 6, 6), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 64, (8, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 32, 32, (9, 8, 7), (3, 3, 3), (2, 2, 2), (1, 1, 1)),      # strided Downsample, odd sizes
    (1, 16, 24, (12, 12, 6), (3, 3, 1), (2, 2, 1), (1, 1, 0)),    # anisotropic kernel/stride/pad
    (2, 3, 32, (8, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),       # conv_in: 3 channels (SIMT only)
    (2, 32, 3, (8, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),       # out conv: 3 output channels
    (2, 48, 96, (5, 5, 5), (1, 1, 1), (1, 1, 1), (0, 0, 0)),      # 1x1x1 skip conv
    (1, 128, 256, (6, 6, 6), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # wide: BN=256 tile, K=3456
    (3, 8, 8, (10, 10), (3, 3), (1, 1), (1, 1)),                  # 2-D
    (1, 1, 16, (16, 16), (3, 3), (1, 1), (1, 1)),                 # 2-D, single input channel
    (1, 24, 40, (7, 7, 7), (3, 3, 3), (1, 1, 1), (0, 1, 1)),      # Upsample defect geometry: pad 0 with kernel 3
    # all-TMA kernels (stride 1, Cin/Cout multiples of 64, box-tileable extents)
    (2, 64, 128, (4, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),     # box 1x8x8
    (1, 128, 64, (8, 4, 12), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # box 4x4x4, two channel chunks
    (1, 64, 64, (10, 12, 12), (3, 3, 3), (1, 1, 1), (0, 1, 1)),   # pad 0 on one axis: output smaller than input
    (3, 64, 64, (8, 8, 8), (1, 1, 1), (1, 1, 1), (0, 0, 0)),      # 1x1x1, odd number of boxes (tile tail)
    (2, 64, 64, (16, 16), (3, 3), (1, 1), (1, 1)),                # 2-D
    (1, 192, 320, (4, 4, 8), (3, 3, 1), (1, 1, 1), (1, 1, 0)),    # anisotropic kernel, N tile tail (320 = 256 + 64)
    (1, 64, 24, (8, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),      # narrow output (BN = 32), dgrad falls back (Cout % 64)
    (8, 64, 256, (24, 24, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),  # BASELINE-size level 0: fwd uses the 256x256 CTA tile
    (8, 256, 64, (24, 24, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),  # ... and dgrad / wgrad use it here
    (2, 128, 256, (6, 6, 6), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # 6^3: 3x6x6 boxes in 128-row slots, split-K
    (3, 64, 64, (6, 6, 6), (3, 3, 3), (1, 1, 1), (1, 1, 1)),      # 6^3: 3x6x6 boxes in 128-row slots (108 valid rows), odd box count
    (2, 64, 128, (5, 5, 5), (3, 3, 3), (1, 1, 1), (1, 1, 1)),     # 5^3: one 125-row box per sample
    (1, 64, 3, (8, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),       # out conv of the LDM U-Net: 3 output channels on the TMA kernel
    (1, 96, 32, (16, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # 96 source channels: second 64-channel chunk half out of bounds
    (2, 96, 64, (8, 8, 8), (1, 1, 1), (1, 1, 1), (0, 0, 0)),      # ... 1x1x1 skip conv over a concat input
    (1, 80, 48, (8, 8, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),     # 80 -> 48: both directions use partial chunks
    # strided Downsample convs: dgrad runs as stride-residue classes on the TMA kernel
    (2, 64, 64, (16, 16, 16), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (1, 128, 64, (8, 16, 16), (3, 3, 3), (1, 2, 2), (1, 1, 1)),   # anisotropic stride
    (1, 64, 64, (16, 16, 8), (3, 3, 1), (2, 2, 1), (1, 1, 0)),    # thin axis: kernel 1 / pad 0 / stride 1
    (2, 64, 128, (9, 11, 16), (3, 3, 3), (2, 2, 2), (1, 1, 1)),   # odd extents: classes of different size
    (1, 64, 64, (8, 8, 8), (1, 1, 1), (2, 2, 2), (0, 0, 0)),      # kernel 1 stride 2: most input voxels get zero gradient
    # 32-channel full-resolution layers: smem-resident halo-tile kernel (fwd + dgrad)
    (1, 32, 32, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 32, 32, (12, 40, 44), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # ragged tiles in x and y
    (1, 32, 1, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # out conv of the AE: one output channel (N padded to 16)
    (1, 32, 16, (16, 48, 48), (3, 3, 1), (1, 1, 1), (1, 1, 0)),   # anisotropic kernel
    (4, 32, 32, (96, 96), (3, 3), (1, 1), (1, 1)),                # 2-D
    (1, 32, 64, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # 64 outputs: single staging buffer, N = 64
    (1, 64, 32, (16, 40, 48), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # dgrad produces 64 channels from 32
    (1, 32, 48, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # 48 outputs padded to N = 64
    # thin ends on CUDA cores (conv_in / out conv of the AE and of pixel-space DDPM U-Nets)
    (2, 1, 32, (12, 20, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # conv_in 1 -> 32, ragged tiles
    (1, 2, 32, (16, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # image + label input
    (1, 32, 2, (16, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # out conv 32 -> 2: thin dgrad + wgrad
    (1, 3, 64, (8, 16, 16), (3, 3, 1), (1, 1, 1), (1, 1, 0)),     # 3 -> 64 (wgrad stays on the padded path), flat kernel
    (3, 1, 64, (40, 40), (3, 3), (1, 1), (1, 1)),                 # 2-D
    (2, 64, 1, (40, 40), (3, 3), (1, 1), (1, 1)),                 # 2-D out conv
    # strided 32-channel Downsample: dgrad = stride-residue classes on the halo kernel
    (1, 32, 32, (32, 32, 32), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (1, 32, 32, (33, 35, 37), (3, 3, 3), (2, 2, 2), (1, 1, 1)),   # odd extents: classes of different size
    (2, 32, 32, (8, 64, 64), (3, 3, 1), (2, 2, 1), (1, 1, 0)),    # anisotropic stride / kernel
    (8, 24, 32, (64, 64), (3, 3), (2, 2), (1, 1)),                # 2-D, 24 input channels
    (1, 32, 32, (32, 32, 32), (1, 1, 1), (2, 2, 2), (0, 0, 0)),   # kernel 1 stride 2: most input voxels get zero gradient
]


def _conv_ref(x, w, b, s, p):
    return (F.conv3d if x.ndim == 5 else F.conv2d)(x, w, b, stride=s, padding=p)


@pytest.mark.parametrize("dtype,engine", [(torch.float32, 1), (torch.bfloat16, 1), (torch.bfloat16, 0)])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fwd_bwd(case, dtype, engine):
    ops = _ops()
    N, Cin, Cout, sp, k, s, p = case
    g = torch.Generator().manual_seed(hash(case) % 10000)
    x = torch.randn((N, Cin, *sp), generator=g)
    w = torch.randn((Cout, Cin, *k), generator=g) / math.sqrt(Cin * math.prod(k))
    b = torch.randn(Cout, generator=g) * 0.1
    cb = torch.randn((N, Cout), generator=g) * 0.1
    if dtype == torch.bfloat16:  # the reference sees the same rounded operands
        x, w = bf16_round(x), bf16_round(w)
    xr, wr, br, cbr = (t.clone().requires_grad_(True) for t in (x, w, b, cb))
    y_ref = _conv_ref(xr, wr, br, s, p)
    res = torch.randn(y_ref.shape, generator=g)
    if dtype == torch.bfloat16:
        res = bf16_round(res)
    resr = res.clone().requires_grad_(True)
    y_ref = y_ref + cbr.reshape(N, Cout, *([1] * len(sp))) + resr
    probe = torch.randn(y_ref.shape, generator=g)
    (y_ref * probe).sum().backward()

    ops.set_engine(engine)
    try:
        xd = _cl(x.to(DEV).to(dtype)).requires_grad_(True)
        wd = _cl(w.to(DEV)).requires_grad_(True)
        bd = b.to(DEV).requires_grad_(True)
        cbd = cb.to(DEV).requires_grad_(True)
        resd = _cl(res.to(DEV).to(dtype)).requires_grad_(True)
        y = ops.conv_nd(xd, wd, bd, s, p, chan_bias=cbd, residual=resd)
        assert y.shape == y_ref.shape and y.dtype == dtype
        (y.float() * probe.to(DEV)).sum().backward()
    finally:
        ops.set_engine(0)
    tol = tol_for(dtype)
    assert rel_err(y, y_ref) < tol
    assert rel_err(xd.grad, xr.grad) < tol
    assert rel_err(wd.grad, wr.grad) < tol
    assert rel_err(bd.grad, br.grad) < tol
    assert rel_err(cbd.grad, cbr.grad) < tol
    assert rel_err(resd.grad, resr.grad) < tol
    assert wd.grad.dtype == torch.float32


# BASELINE config 3 layer shapes at FULL size (production engine only; the CPU reference of each takes seconds)
WIDE_CONV_CASES = [
    (2, 1536, 768, (6, 6, 6), (3, 3, 3), (1, 1, 1), (1, 1, 1)),    # first up-block resnet: K = 41 472 over a skip concat
    (2, 1024, 512, (12, 12, 12), (3, 3, 3), (1, 1, 1), (1, 1, 1)),  # 512+512 concat input at the 12^3 level
    (8, 512, 512, (24, 24, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),   # the Upsample conv: the single largest layer
    (8, 512, 512, (12, 12, 12), (3, 3, 3), (2, 2, 2), (1, 1, 1)),   # Downsample 12^3 -> 6^3
    (8, 1536, 768, (6, 6, 6), (1, 1, 1), (1, 1, 1), (0, 0, 0)),     # 1x1x1 skip connection over the widest concat
]


@pytest.mark.parametrize("case", WIDE_CONV_CASES)
def test_conv_fwd_bwd_baseline_width(case):
    ops = _ops()
    N, Cin, Cout, sp, k, s, p = case
    g = torch.Generator().manual_seed(hash(case) % 10000)
    x = bf16_round(torch.randn((N, Cin, *sp), generator=g))
    w = bf16_round(torch.randn((Cout, Cin, *k), generator=g) / math.sqrt(Cin * math.prod(k)))
    b = torch.randn(Cout, generator=g) * 0.1
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    y_ref = _conv_ref(xr, wr, br, s, p)
    probe = torch.randn(y_ref.shape, generator=g)
    (y_ref * probe).sum().backward()
    xd = _cl(x.to(DEV).to(torch.bfloat16)).requires_grad_(True)
    wd = _cl(w.to(DEV)).requires_grad_(True)
    bd = b.to(DEV).requires_grad_(True)
    y = ops.conv_nd(xd, wd, bd, s, p)
    (y.float() * probe.to(DEV)).sum().backward()
    assert rel_err(y, y_ref) < BF16_TOL
    assert rel_err(xd.grad, xr.grad) < BF16_TOL
    assert rel_err(wd.grad, wr.grad) < BF16_TOL
    assert rel_err(bd.grad, br.grad) < BF16_TOL


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,K,O,bias", [(5, 32, 48, True), (300, 64, 64, True), (7, 24, 16, False),
                                            (1000, 256, 512, True), (2, 1024, 768, True)])
def test_linear(rows, K, O, bias, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(rows)
    x, w = torch.randn(rows, K, generator=g), torch.randn(O, K, generator=g) / math.sqrt(K)
    b = torch.randn(O, generator=g) * 0.1 if bias else None
    if dtype == torch.bfloat16:
        x, w = bf16_round(x), bf16_round(w)
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    br = b.clone().requires_grad_(True) if bias else None
    y_ref = F.linear(xr, wr, br)
    probe = torch.randn(y_ref.shape, generator=g)
    (y_ref * probe).sum().backward()
    xd, wd = x.to(DEV).to(dtype).requires_grad_(True), w.to(DEV).requires_grad_(True)
    bd = b.to(DEV).requires_grad_(True) if bias else None
    y = ops.linear(xd, wd, bd)
    (y.float() * probe.to(DEV)).sum().backward()
    tol = tol_for(dtype)
    assert rel_err(y, y_ref) < tol and rel_err(xd.grad, xr.grad) < tol and rel_err(wd.grad, wr.grad) < tol
    if bias:
        assert rel_err(bd.grad, br.grad) < tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("silu", [False, True])
@pytest.mark.parametrize("N,C,G,sp", [(2, 32, 16, (6, 6, 6)), (1, 256, 32, (5, 4, 3)), (2, 16, 16, (9, 9)),
                                      (1, 1536, 32, (3, 3, 3)), (2, 64, 8, (17, 5, 3)), (1, 32, 32, (24, 24, 24)),
                                      # TMA-staged bf16 kernels: groups straddling 256-channel slabs (cpg 24 / 40), groups
                                      # straddling 16-byte vectors (cpg 6), many row chunks, 256-row stages
                                      (8, 768, 32, (6, 6, 6)), (2, 1280, 32, (4, 4, 4)), (2, 96, 16, (8, 8, 8)),
                                      (2, 256, 32, (24, 24, 24)), (1, 32, 16, (40, 40, 40)), (3, 512, 32, (12, 12, 12))])
def test_group_norm(N, C, G, sp, silu, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(C + G)
    x = torch.randn((N, C, *sp), generator=g) * 2 + 0.5
    gamma, beta = 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    if dtype == torch.bfloat16:
        x = bf16_round(x)
    xr, gr, br = (t.clone().requires_grad_(True) for t in (x, gamma, beta))
    y_ref = F.group_norm(xr, G, gr, br, 1e-6)
    if silu:
        y_ref = F.silu(y_ref)
    probe = torch.randn(y_ref.shape, generator=g)
    (y_ref * probe).sum().backward()
    xd = _cl(x.to(DEV).to(dtype)).requires_grad_(True)
    gd, bd = gamma.to(DEV).requires_grad_(True), beta.to(DEV).requires_grad_(True)
    y = ops.group_norm(xd, gd, bd, G, 1e-6, silu=silu)
    pd = _cl(probe.to(DEV).to(dtype)) if dtype == torch.bfloat16 else probe.to(DEV)
    if dtype == torch.bfloat16:  # reference backward must see the same rounded upstream gradient
        xr.grad = None; gr.grad = None; br.grad = None
        y2 = F.group_norm(xr, G, gr, br, 1e-6)
        y2 = F.silu(y2) if silu else y2
        (y2 * bf16_round(probe)).sum().backward()
    y.backward(pd.to(dtype))
    tol = tol_for(dtype)
    assert rel_err(y, y_ref) < tol
    assert rel_err(xd.grad, xr.grad) < tol
    assert rel_err(gd.grad, gr.grad) < tol and rel_err(bd.grad, br.grad) < tol


@pytest.mark.parametrize("C,G,sp", [(64, 16, (8, 8, 8)), (256, 32, (6, 6, 6)), (96, 16, (5, 6, 7))])
def test_group_norm_split_and_colsum(C, G, sp):
    """The two halves of the bf16 forward through their own entry points (statistics as raw fp64 sums -- what a
    convolution epilogue accumulates -- then apply), and the per-(n, c) column sums of dx the backward hands to the
    producing convolution."""
    import ctypes as Cc
    ops = _ops()
    from medical_image_generation_b200 import _lib
    N = 2
    S = math.prod(sp)
    g = torch.Generator().manual_seed(C)
    x = bf16_round(torch.randn((N, C, *sp), generator=g) * 1.5 - 0.3)
    gamma, beta = 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    xd = _cl(x.to(DEV).to(torch.bfloat16))
    assert _lib.load().mig_groupnorm_can_split(1, N, S, C, G) == 1
    sums = torch.empty(N, G, 2, dtype=torch.float64, device=DEV)
    _lib.call("mig_groupnorm_stats", 1, ops._ptr(xd), ops._ptr(sums), N, S, C, G, ops._stream())
    xg = x.reshape(N, G, C // G, -1).double()
    want = torch.stack([xg.sum(dim=(2, 3)), (xg * xg).sum(dim=(2, 3))], dim=-1)
    assert rel_err(sums, want) < 1e-5
    y = torch.empty_like(xd)
    mean, rstd = torch.empty(N, G, device=DEV), torch.empty(N, G, device=DEV)
    gamma_d, beta_d = gamma.to(DEV), beta.to(DEV)         # (named: the raw pointers must outlive the calls)
    _lib.call("mig_groupnorm_apply", 1, ops._ptr(xd), ops._ptr(gamma_d), ops._ptr(beta_d), ops._ptr(sums),
              ops._ptr(y), ops._ptr(mean), ops._ptr(rstd), N, S, C, G, 1e-6, 1, ops._stream())
    assert rel_err(y, F.silu(F.group_norm(x, G, gamma, beta, 1e-6))) < BF16_TOL
    assert rel_err(mean, xg.mean(dim=(2, 3))) < 1e-5
    # backward with the column sums requested
    dy = bf16_round(torch.randn(x.shape, generator=g))
    dyd = _cl(dy.to(DEV).to(torch.bfloat16))
    dx = torch.empty_like(xd)
    dgam, dbet = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    colsum = torch.empty(N, C, device=DEV)
    need = _lib.load().mig_groupnorm_workspace_bytes(N, S, C, G)
    ws = torch.empty(int(need), dtype=torch.uint8, device=DEV)
    _lib.call("mig_groupnorm_bwd", 1, ops._ptr(xd), ops._ptr(dyd), ops._ptr(gamma_d), ops._ptr(beta_d),
              ops._ptr(mean), ops._ptr(rstd), ops._ptr(dx), ops._ptr(dgam), ops._ptr(dbet), ops._ptr(colsum), None, 0, N, S, C, G, 1,
              ops._ptr(ws), ws.numel(), ops._stream())
    xr = x.clone().requires_grad_(True)
    F.silu(F.group_norm(xr, G, gamma, beta, 1e-6)).backward(dy)
    assert rel_err(dx, xr.grad) < BF16_TOL
    # the column sums are computed analytically from the statistics pass (fp32), not from the rounded dx
    assert rel_err(colsum, xr.grad.sum(dim=tuple(range(2, x.ndim)))) < 5e-3


def test_batched_time_embedding_projections():
    """mig_temb_proj_all_fwd / _bwd: time_emb_proj of every ResnetBlock in one launch per pass (unet:691-695) against
    per-layer F.linear with autograd; one layer gets no gradient (null dy), one has no bias."""
    ops = _ops()
    from medical_image_generation_b200 import layers
    g = torch.Generator().manual_seed(11)
    K, rows = 128, 3
    chans = [32, 64, 48, 96, 8]
    lins = [layers.Linear(K, c, bias=(i != 2)) for i, c in enumerate(chans)]
    for m in lins:
        with torch.no_grad():
            for p in m.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)
        m.to(DEV)
    x = torch.randn(rows, K, generator=g)
    xd = x.to(DEV).requires_grad_(True)
    outs = ops.temb_projections(xd, lins)
    assert outs is not None and [tuple(o.shape) for o in outs] == [(rows, c) for c in chans]
    xr = x.clone().requires_grad_(True)
    refs = [F.linear(xr, m.weight.detach().cpu(), None if m.bias is None else m.bias.detach().cpu()) for m in lins]
    wr = []
    for m in lins:
        wr.append((m.weight.detach().cpu().clone().requires_grad_(True),
                   None if m.bias is None else m.bias.detach().cpu().clone().requires_grad_(True)))
    refs = [F.linear(xr, w, b) for w, b in wr]
    for o, r in zip(outs, refs):
        assert rel_err(o, r) < 1e-5
    probes = [torch.randn(rows, c, generator=g) for c in chans]
    used = [0, 1, 2, 4]                                   # layer 3 gets no gradient
    sum((outs[i] * probes[i].to(DEV)).sum() for i in used).backward()
    sum((refs[i] * probes[i]).sum() for i in used).backward()
    assert rel_err(xd.grad, xr.grad) < 1e-5
    for i, m in enumerate(lins):
        if i in used:
            assert rel_err(m.weight.grad, wr[i][0].grad) < 1e-5
            if m.bias is not None:
                assert rel_err(m.bias.grad, wr[i][1].grad) < 1e-5
        else:
            assert m.weight.grad is None


@pytest.mark.parametrize("case", [
    # (N, Cin, Cout, spatial, groups, residual + time embedding, statistics expected from the tcgen05 epilogue)
    (2, 64, 256, (16, 16, 16), 32, True, True),     # 8 channels per group
    (4, 64, 768, (16, 16, 16), 32, False, True),    # 24 channels per group: groups straddle the 32-column reduction units
    (2, 64, 512, (24, 24, 24), 32, True, True),     # 16 channels per group, two N tiles
    (4, 64, 1280, (16, 16, 16), 32, False, True),   # 40 channels per group, five N tiles
    (8, 64, 128, (16, 16, 16), 16, True, True),     # one 128-column tile
    (2, 128, 256, (6, 6, 6), 32, True, False),      # split-K plan: statistics fall back to one pass over y
    (1, 32, 32, (32, 32, 32), 16, False, False),    # halo kernel (2 channels per group): statistics pass
])
def test_conv_epilogue_groupnorm_statistics(case, monkeypatch):
    """mig_conv_fwd_stats: the convolution also delivers (sum y, sum y^2) per (sample, group) of its bf16 output, and
    ops.group_norm on that tensor (apply only) equals GroupNorm computed from scratch."""
    ops = _ops()
    import ctypes as Cc
    from medical_image_generation_b200 import _lib
    N, Cin, Cout, sp, G, extras, in_epilogue = case
    # by default the epilogue delivers the statistics only where it is hidden behind the next tile (narrow layers);
    # "always" exercises it for every group width
    monkeypatch.setenv("MIG_GN_EPILOGUE", "always")
    geom = _lib.conv_geom(N, sp, sp, Cin, Cout, (3, 3, 3), (1, 1, 1), (1, 1, 1))
    need = _lib.load().mig_conv_workspace_bytes(Cc.byref(geom), 1, 0, 0)
    assert bool(_lib.load().mig_conv_fwd_stats_in_epilogue(Cc.byref(geom), 1, G, 0, max(int(need), 1 << 20))) == in_epilogue
    g = torch.Generator().manual_seed(Cout + sp[0])
    x = bf16_round(torch.randn((N, Cin, *sp), generator=g))
    w = bf16_round(torch.randn((Cout, Cin, 3, 3, 3), generator=g) / math.sqrt(Cin * 27))
    b = torch.randn(Cout, generator=g) * 0.1
    xd, wd, bd = _cl(x.to(DEV).to(torch.bfloat16)), _cl(w.to(DEV)), b.to(DEV)
    cb = res = None
    if extras:
        cb = (torch.randn((N, Cout), generator=g) * 0.3).to(DEV)
        res = _cl(bf16_round(torch.randn((N, Cout, *sp), generator=g)).to(DEV).to(torch.bfloat16))
    with torch.no_grad():
        y = ops.conv_nd(xd, wd, bd, 1, 1, chan_bias=cb, residual=res, gn_groups=G)
        y_plain = ops.conv_nd(xd, wd, bd, 1, 1, chan_bias=cb, residual=res)
    if in_epilogue:
        assert torch.equal(y, y_plain)                   # the statistics epilogue must not change the output
    else:
        assert rel_err(y, y_plain) < 4e-3                # (split-K reduces with fp32 atomics: last-bit differences)
    sums, groups = y._mig_gn_sums
    assert groups == G and tuple(sums.shape) == (N, G, 2)
    yg = y.float().cpu().reshape(N, G, Cout // G, -1).double()
    want = torch.stack([yg.sum(dim=(2, 3)), (yg * yg).sum(dim=(2, 3))], dim=-1)
    assert rel_err(sums[..., 1], want[..., 1]) < 1e-5
    assert float((sums[..., 0].cpu() - want[..., 0]).abs().max()) < 1e-4 * float(want[..., 1].sqrt().max()) + 1e-3
    gamma, beta = (1 + 0.2 * torch.randn(Cout, generator=g)).to(DEV), (0.2 * torch.randn(Cout, generator=g)).to(DEV)
    seen = []
    real = ops.call
    ops.call = lambda name, *a: (seen.append(name), real(name, *a))[1]
    try:
        with torch.no_grad():
            z = ops.group_norm(y, gamma, beta, G, 1e-6, silu=True)
    finally:
        ops.call = real
    assert seen == ["mig_groupnorm_apply"], seen
    z_ref = F.silu(F.group_norm(y.float().cpu(), G, gamma.cpu(), beta.cpu(), 1e-6))
    assert rel_err(z, z_ref) < BF16_TOL


def test_resnet_block_backward_uses_groupnorm_column_sums():
    """conv1's bias / time-embedding gradients come from norm2's backward (no mig_chan_bias_bwd / bias column-sum pass
    over dy for conv1) and still match the oracle."""
    from medical_image_generation_b200 import unet as U
    from oracle import torch_oracle as O
    ops = _ops()
    g = torch.Generator().manual_seed(4)
    rb = U.ResnetBlock(3, 64, 32, 64, norm_num_groups=16)
    with torch.no_grad():
        for p in rb.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.1 if p.ndim > 1 else 0.3))
    rb = rb.to(DEV)
    x = torch.randn(2, 64, 8, 8, 8, generator=g)
    emb = torch.randn(2, 32, generator=g)
    sd = {"blk." + k: v.detach().cpu().clone().requires_grad_(True) for k, v in rb.state_dict().items()}
    probe = torch.randn(2, 64, 8, 8, 8, generator=g)
    embr = emb.clone().requires_grad_(True)
    (O.unet_resnet_block(sd, "blk", x, embr, 16, 1e-6) * probe).sum().backward()
    seen = []
    real = ops.call
    ops.call = lambda name, *a: (seen.append(name), real(name, *a))[1]
    try:
        embd = emb.to(DEV).requires_grad_(True)
        y = rb(x.to(DEV).to(torch.bfloat16), embd)
        (y.float() * probe.to(DEV)).sum().backward()
    finally:
        ops.call = real
    assert seen.count("mig_chan_bias_bwd") == 0, seen
    named = dict(rb.named_parameters())
    assert rel_err(named["conv1.conv.bias"].grad, sd["blk.conv1.conv.bias"].grad) < 3e-2
    assert rel_err(named["time_emb_proj.weight"].grad, sd["blk.time_emb_proj.weight"].grad) < 3e-2
    assert rel_err(embd.grad, embr.grad) < 3e-2
    assert rel_err(named["conv1.conv.weight"].grad, sd["blk.conv1.conv.weight"].grad) < 3e-2


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,Lq,Lk,C,heads", [(2, 64, 64, 32, 1), (1, 216, 216, 96, 1), (2, 27, 27, 64, 4),
                                              (2, 30, 3, 32, 2), (1, 130, 130, 256, 1)])
def test_sdpa(B, Lq, Lk, C, heads, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(Lq + C)
    q, k, v = (torch.randn(B, L, C, generator=g) for L in (Lq, Lk, Lk))
    if dtype == torch.bfloat16:
        q, k, v = bf16_round(q), bf16_round(k), bf16_round(v)
    scale = 1 / math.sqrt(C / heads)
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))

    def split(t):
        return t.reshape(B, -1, heads, C // heads).permute(0, 2, 1, 3)

    p = torch.softmax(split(qr) @ split(kr).transpose(-1, -2) * scale, dim=-1)
    o_ref = (p @ split(vr)).permute(0, 2, 1, 3).reshape(B, Lq, C)
    probe = torch.randn(o_ref.shape, generator=g)
    (o_ref * probe).sum().backward()
    qd, kd, vd = (t.to(DEV).to(dtype).requires_grad_(True) for t in (q, k, v))
    o = ops.sdpa(qd, kd, vd, heads, scale)
    (o.float() * probe.to(DEV)).sum().backward()
    tol = tol_for(dtype)
    assert rel_err(o, o_ref) < tol
    assert rel_err(qd.grad, qr.grad) < tol * 1.5 and rel_err(kd.grad, kr.grad) < tol * 1.5
    assert rel_err(vd.grad, vr.grad) < tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_elementwise_family(dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    tol = tol_for(dtype)
    x = torch.randn(2, 24, 5, 6, 7, generator=g)
    x = bf16_round(x) if dtype == torch.bfloat16 else x
    xd = _cl(x.to(DEV).to(dtype)).requires_grad_(True)
    xr = x.clone().requires_grad_(True)
    # silu
    y = ops.silu(xd); y.float().sum().backward()
    F.silu(xr).sum().backward()
    assert rel_err(y, F.silu(x)) < tol and rel_err(xd.grad, xr.grad) < tol
    # concat / split
    a, b = torch.randn(2, 8, 4, 4, 4, generator=g), torch.randn(2, 24, 4, 4, 4, generator=g)
    ad, bd = _cl(a.to(DEV).to(dtype)).requires_grad_(True), _cl(b.to(DEV).to(dtype)).requires_grad_(True)
    c = ops.cat_channels(ad, bd)
    pr = torch.randn(c.shape, generator=g)
    (c.float() * pr.to(DEV)).sum().backward()
    assert rel_err(c, torch.cat([a, b], 1)) < tol
    assert rel_err(ad.grad, pr[:, :8]) < tol and rel_err(bd.grad, pr[:, 8:]) < tol
    # odd channel counts (scalar path)
    a3, b5 = torch.randn(1, 3, 4, 4, generator=g), torch.randn(1, 5, 4, 4, generator=g)
    c2 = ops.cat_channels(_cl(a3.to(DEV).to(dtype)), _cl(b5.to(DEV).to(dtype)))
    assert rel_err(c2, torch.cat([a3, b5], 1)) < tol
    # nearest upsample + adjoint
    for f in [(2, 2, 2), (2, 2, 1), (1, 3, 2)]:
        u = torch.randn(2, 16, 3, 4, 5, generator=g)
        ud = _cl(u.to(DEV).to(dtype)).requires_grad_(True)
        ur = u.clone().requires_grad_(True)
        yu = ops.upsample_nearest(ud, f)
        yr = F.interpolate(ur, scale_factor=tuple(float(v) for v in f), mode="nearest")
        pu = torch.randn(yr.shape, generator=g)
        (yu.float() * pu.to(DEV)).sum().backward(); (yr * pu).sum().backward()
        assert yu.shape == yr.shape and rel_err(yu, yr) < tol and rel_err(ud.grad, ur.grad) < tol
    # layout round trip
    z = torch.randn(2, 5, 3, 4, 6, generator=g)
    zc = ops.to_channels_last(z.to(DEV), dtype)
    assert zc.is_contiguous(memory_format=torch.channels_last_3d) and rel_err(zc, z) < tol
    back = ops.from_channels_last(zc, torch.float32)
    assert back.is_contiguous() and rel_err(back, z) < tol
    # geglu
    h = torch.randn(7, 2 * 24, generator=g)
    hd, hr = h.to(DEV).to(dtype).requires_grad_(True), (bf16_round(h) if dtype == torch.bfloat16 else h).clone().requires_grad_(True)
    yg = ops.geglu(hd); yg.float().sum().backward()
    a_, g_ = hr.chunk(2, -1); (a_ * F.gelu(g_)).sum().backward()
    assert rel_err(yg, a_ * F.gelu(g_)) < tol and rel_err(hd.grad, hr.grad) < tol
    # layer norm
    ln_x = torch.randn(11, 48, generator=g)
    gam, bet = 1 + 0.1 * torch.randn(48, generator=g), 0.1 * torch.randn(48, generator=g)
    lx = (bf16_round(ln_x) if dtype == torch.bfloat16 else ln_x)
    lr, gr_, br_ = lx.clone().requires_grad_(True), gam.clone().requires_grad_(True), bet.clone().requires_grad_(True)
    ld, gd_, bd_ = lx.to(DEV).to(dtype).requires_grad_(True), gam.to(DEV).requires_grad_(True), bet.to(DEV).requires_grad_(True)
    pl = torch.randn(11, 48, generator=g)
    yl = ops.layer_norm(ld, gd_, bd_, 1e-5); (yl.float() * pl.to(DEV)).sum().backward()
    yl_ref = F.layer_norm(lr, (48,), gr_, br_, 1e-5); (yl_ref * pl).sum().backward()
    assert rel_err(yl, yl_ref) < tol and rel_err(ld.grad, lr.grad) < tol * 2
    assert rel_err(gd_.grad, gr_.grad) < tol * 2 and rel_err(bd_.grad, br_.grad) < tol * 2


def test_timestep_embedding_matches_reference_formula():
    ops = _ops()
    from oracle import torch_oracle as O
    for dim in (32, 256, 7):
        t = torch.tensor([0, 1, 17, 500, 999])
        got = ops.timestep_embedding(t.to(DEV), dim)
        assert got.shape == (5, dim)
        assert float((got.cpu() - O.timestep_embedding(t, dim)).abs().max()) < 2e-4  # sin/cos of args up to 999 rad
    with pytest.raises(ValueError):
        ops.timestep_embedding(torch.zeros(2, 2, device=DEV), 8)


def test_losses_and_vae_tail():
    ops = _ops()
    g = torch.Generator().manual_seed(5)
    for shape in [(2, 3, 7, 5, 3), (1, 1, 33)]:
        a, b = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
        for l1 in (False, True):
            ar = a.clone().requires_grad_(True)
            ref = F.l1_loss(ar, b) if l1 else F.mse_loss(ar, b)
            (ref * 3.0).backward()
            ad = a.to(DEV).requires_grad_(True)
            got = (ops.l1_loss if l1 else ops.mse_loss)(ad, b.to(DEV))
            (got * 3.0).backward()
            assert got.dtype == torch.float32 and rel_err(got, ref) < 1e-6 and rel_err(ad.grad, ar.grad) < 1e-6
    mu, lv = torch.randn(2, 3, 4, 4, 4, generator=g), torch.randn(2, 3, 4, 4, 4, generator=g) * 8
    lv[0, 0, 0, 0, 0], lv[0, 0, 0, 0, 1] = -40.0, 30.0   # exercise both clamp sides
    eps = torch.randn(mu.shape, generator=g)
    mr, lr = mu.clone().requires_grad_(True), lv.clone().requires_grad_(True)
    sig_r = torch.exp(torch.clamp(lr, -30.0, 20.0) / 2)
    z_r = mr + eps * sig_r
    kl_r = 0.5 * torch.sum(mr.pow(2) + sig_r.pow(2) - torch.log(sig_r.pow(2)) - 1, dim=[1, 2, 3, 4])
    kl_r = torch.sum(kl_r) / kl_r.shape[0]
    (z_r.sum() + 1e-3 * kl_r).backward()
    md, ld = mu.to(DEV).requires_grad_(True), lv.to(DEV).requires_grad_(True)
    sig = ops.vae_sigma(ld)
    z = ops.vae_reparam(md, sig, eps.to(DEV))
    kl = ops.kl_loss(md, sig)
    (z.sum() + 1e-3 * kl).backward()
    assert rel_err(sig, sig_r) < 1e-6 and rel_err(z, z_r) < 1e-6 and rel_err(kl, kl_r) < 1e-5
    assert rel_err(md.grad, mr.grad) < 1e-5 and rel_err(ld.grad, lr.grad) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scheduler_kernels_vs_oracle(dtype):
    import medical_image_generation_b200 as mig
    from oracle.ddpm_oracle import OracleDDPMScheduler
    kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
    g = torch.Generator().manual_seed(9)
    for pred in ("epsilon", "v_prediction", "sample"):
        s, o = mig.DDPMScheduler(prediction_type=pred, **kw), OracleDDPMScheduler(prediction_type=pred, **kw)
        x0, n = torch.randn(4, 3, 6, 5, 4, generator=g), torch.randn(4, 3, 6, 5, 4, generator=g)
        ts = torch.tensor([0, 1, 500, 999])
        if dtype == torch.bfloat16:
            x0, n = bf16_round(x0), bf16_round(n)
        got = s.add_noise(x0.to(DEV).to(dtype), n.to(DEV).to(dtype), ts.to(DEV))
        want = o.add_noise(x0.to(dtype), n.to(dtype), ts)          # oracle in the same dtype, like upstream
        tol = 1e-6 if dtype == torch.float32 else 8e-3
        assert rel_err(got, want) < tol
        assert rel_err(s.get_velocity(x0.to(DEV).to(dtype), n.to(DEV).to(dtype), ts.to(DEV)),
                       o.get_velocity(x0.to(dtype), n.to(dtype), ts)) < tol
        for t in (999, 500, 1, 0):
            e, x, z = (torch.randn(2, 3, 5, 5, 5, generator=g) for _ in range(3))
            if dtype == torch.bfloat16:
                e, x, z = bf16_round(e), bf16_round(x), bf16_round(z)
            prev, x0h = s.step(e.to(DEV).to(dtype), t, x.to(DEV).to(dtype), noise=z.to(DEV).to(dtype))
            wprev, wx0 = o.step(e, t, x, noise=z)
            tol2 = 2e-6 if dtype == torch.float32 else 8e-3
            assert rel_err(prev, wprev) < tol2 and rel_err(x0h, wx0) < tol2, (pred, t)
    # t == 0 adds no noise; empty batch edge
    prev, _ = s.step(torch.zeros(1, 1, 4, 4, device=DEV), 0, torch.ones(1, 1, 4, 4, device=DEV))
    assert torch.isfinite(prev).all()


def test_adamw_and_clip_match_torch():
    import ctypes as C
    from medical_image_generation_b200 import _lib
    g = torch.Generator().manual_seed(11)
    n = 10007
    p0, grads = torch.randn(n, generator=g), [torch.randn(n, generator=g) * (3.0 if i == 0 else 0.01) for i in range(4)]
    pr = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([pr], lr=2e-5)
    p = p0.clone().to(DEV); m = torch.zeros(n, device=DEV); v = torch.zeros(n, device=DEV)
    shadow = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for step, gr in enumerate(grads, 1):
        pr.grad = gr.clone()
        torch.nn.utils.clip_grad_norm_([pr], max_norm=1.0)
        opt.step()
        gd = gr.to(DEV)
        ss = torch.zeros(1, device=DEV)
        parts = torch.zeros(2048, device=DEV)
        _lib.call("mig_sumsq", C.c_void_p(gd.data_ptr()), C.c_void_p(ss.data_ptr()), C.c_void_p(parts.data_ptr()), n, st)
        ss2 = torch.zeros(1, device=DEV)
        _lib.call("mig_sumsq", C.c_void_p(gd.data_ptr()), C.c_void_p(ss2.data_ptr()), C.c_void_p(parts.data_ptr()), n, st)
        assert torch.equal(ss, ss2)       # deterministic (bit-identical replicas under data parallelism)
        assert rel_err(ss.sqrt(), gr.norm()) < 1e-5
        _lib.call("mig_adamw_step", C.c_void_p(p.data_ptr()), C.c_void_p(gd.data_ptr()), C.c_void_p(m.data_ptr()),
                  C.c_void_p(v.data_ptr()), n, 2e-5, 0.9, 0.999, 1e-8, 0.01, step, C.c_void_p(ss.data_ptr()), 1.0,
                  C.c_void_p(shadow.data_ptr()), None, st)
        assert rel_err(p, pr.detach()) < 1e-6
    assert torch.equal(shadow, p.to(torch.bfloat16))   # the shadow is defined as the round-to-nearest of the master


def test_errors_are_loud():
    ops = _ops()
    x = torch.randn(1, 8, 4, 4, 4, device=DEV)
    w = torch.randn(4, 6, 3, 3, 3, device=DEV)
    with pytest.raises(RuntimeError, match="channels"):
        ops.conv_nd(x, w, None, 1, 1)
    with pytest.raises(RuntimeError, match="match"):
        ops.cat_channels(x, torch.randn(1, 8, 4, 4, 3, device=DEV))
    with pytest.raises(RuntimeError, match="does not fit"):
        ops.conv_nd(torch.randn(1, 8, 1, 1, 1, device=DEV), torch.randn(4, 8, 3, 3, 3, device=DEV), None, 1, 0)
    with pytest.raises(TypeError):
        ops.silu(torch.zeros(4, device=DEV, dtype=torch.float16))


@pytest.mark.parametrize("B,Lq,Lk,C,heads", [(2, 256, 256, 128, 1), (1, 200, 333, 128, 2), (2, 216, 216, 768, 1),
                                              (1, 1728, 1728, 512, 1), (1, 130, 70, 64, 1), (1, 5, 3, 256, 4),
                                              (1, 1024, 4096, 128, 1),
                                              # head dim 128 / 64 through the two-query-tile kernel with ragged tails on both
                                              # sides: second query tile partly / wholly past the end, last key tile ragged
                                              (1, 300, 200, 128, 1), (2, 257, 129, 256, 2), (1, 513, 640, 192, 3),
                                              (1, 100, 1000, 128, 1)])
def test_flash_attention_forward(B, Lq, Lk, C, heads):
    """Fused tcgen05 flash-style attention (forward only) vs fp32 softmax attention on the CPU; includes ragged tails,
    cross-attention lengths, multi-head and the 512/768-channel single heads of the LDM default (value-dim slicing)."""
    ops = _ops()
    g = torch.Generator().manual_seed(Lq + Lk + C)
    q, k, v = (bf16_round(torch.randn(B, L, C, generator=g)) for L in (Lq, Lk, Lk))
    scale = 1 / math.sqrt(C / heads)

    def split(t):
        return t.reshape(B, -1, heads, C // heads).permute(0, 2, 1, 3)

    p = torch.softmax(split(q) @ split(k).transpose(-1, -2) * scale, dim=-1)
    want = (p @ split(v)).permute(0, 2, 1, 3).reshape(B, Lq, C)
    qd, kd, vd = (t.to(DEV).bfloat16() for t in (q, k, v))
    assert ops.flash_attention_usable(qd, kd, vd, heads)
    with torch.no_grad():
        got = ops.sdpa(qd, kd, vd, heads, scale)
    assert got.shape == want.shape and rel_err(got, want) < BF16_TOL
    # and it agrees with the GEMM-composed training path
    ops.set_flash_attention(False)
    try:
        with torch.no_grad():
            ref2 = ops.sdpa(qd, kd, vd, heads, scale)
    finally:
        ops.set_flash_attention(True)
    assert rel_err(got, ref2) < BF16_TOL


@pytest.mark.parametrize("B,Lq,Lk,C,heads", [(2, 256, 256, 128, 1), (1, 200, 333, 128, 2), (2, 216, 216, 768, 1),
                                              (1, 1728, 1728, 512, 1), (1, 130, 70, 64, 1), (1, 5, 3, 256, 4),
                                              (1, 700, 300, 256, 1), (2, 384, 384, 192, 1), (1, 300, 200, 128, 1)])
def test_flash_attention_backward(B, Lq, Lk, C, heads):
    """Training attention through the fused kernels (no L x L tensor): dQ, dK, dV of mig_flash_attention_bwd against fp32
    autograd of softmax attention on the CPU -- ragged tails, cross-attention lengths, multi-head, and the 512 / 768-channel
    single heads of the LDM default (column-sliced accumulators)."""
    ops = _ops()
    g = torch.Generator().manual_seed(Lq * 3 + Lk + C)
    q, k, v = (bf16_round(torch.randn(B, L, C, generator=g)) for L in (Lq, Lk, Lk))
    probe = bf16_round(torch.randn(B, Lq, C, generator=g))
    scale = 1 / math.sqrt(C / heads)

    def split(t):
        return t.reshape(B, -1, heads, C // heads).permute(0, 2, 1, 3)

    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))
    p = torch.softmax(split(qr) @ split(kr).transpose(-1, -2) * scale, dim=-1)
    want = (p @ split(vr)).permute(0, 2, 1, 3).reshape(B, Lq, C)
    (want * probe).sum().backward()
    qd, kd, vd = (t.to(DEV).bfloat16().requires_grad_(True) for t in (q, k, v))
    seen = []
    real = ops.call
    ops.call = lambda name, *a: (seen.append(name), real(name, *a))[1]
    ops.set_flash_attention(True, training=True)     # ("auto" would pick the unfused chain for d = 512 at L = 1728)
    try:
        got = ops.sdpa(qd, kd, vd, heads, scale)
        (got.float() * probe.to(DEV)).sum().backward()
    finally:
        ops.call = real
        ops.set_flash_attention(True, training="auto")
    assert seen == ["mig_flash_attention_fwd_ld", "mig_flash_attention_bwd"], seen
    assert rel_err(got, want) < BF16_TOL
    assert rel_err(qd.grad, qr.grad) < BF16_TOL
    assert rel_err(kd.grad, kr.grad) < BF16_TOL
    assert rel_err(vd.grad, vr.grad) < BF16_TOL
    # and against the unfused GEMM + softmax training chain on the same bf16 inputs
    ops.set_flash_attention(True, training=False)
    try:
        q2, k2, v2 = (t.to(DEV).bfloat16().requires_grad_(True) for t in (q, k, v))
        (ops.sdpa(q2, k2, v2, heads, scale).float() * probe.to(DEV)).sum().backward()
    finally:
        ops.set_flash_attention(True, training="auto")
    assert rel_err(qd.grad, q2.grad) < BF16_TOL and rel_err(kd.grad, k2.grad) < BF16_TOL


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape,k,s", [((2, 16, 8, 8, 4), (2, 2, 1), (2, 2, 1)), ((1, 8, 9, 7, 6), (3, 3, 3), (2, 2, 2)),
                                       ((3, 24, 10, 12), (2, 2), (2, 2)), ((1, 5, 7, 7), (3, 2), (1, 2))])
def test_avg_pool_fwd_bwd(shape, k, s, dtype):
    """nn.AvgPool{2,3}d(kernel, stride) of ResnetBlock(down=True) (unet:517-518), overlapping windows included."""
    ops = _ops()
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(shape, generator=g)
    if dtype == torch.bfloat16:
        x = bf16_round(x)
    xr = x.clone().requires_grad_(True)
    pool = F.avg_pool3d if len(shape) == 5 else F.avg_pool2d
    y_ref = pool(xr, kernel_size=k, stride=s)
    dy = torch.randn(y_ref.shape, generator=g)
    if dtype == torch.bfloat16:
        dy = bf16_round(dy)
    y_ref.backward(dy)
    xd = x.to(DEV).to(dtype).requires_grad_(True)
    y = ops.avg_pool(xd, k, s)
    y.backward(dy.to(DEV).to(dtype))
    tol = 1e-5 if dtype == torch.float32 else BF16_TOL
    assert y.shape == y_ref.shape and rel_err(y, y_ref) < tol and rel_err(xd.grad, xr.grad) < tol


CONVT_CASES = [
    (2, 16, 16, (6, 6, 6), (3, 3, 3), (2, 2, 2), (1, 1, 1)),     # MONAI default output_padding = stride - 1
    (1, 64, 64, (8, 8, 8), (3, 3, 3), (2, 2, 2), (1, 1, 1)),     # tcgen05 stride-residue classes
    (1, 32, 32, (16, 16, 16), (3, 3, 3), (2, 2, 1), (1, 1, 1)),  # anisotropic stride, halo-kernel classes
    (2, 24, 40, (9, 7), (4, 4), (2, 2), (1, 1)),                 # 2-D, kernel 4, different channel counts
]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", CONVT_CASES)
def test_conv_transpose_fwd_bwd(case, dtype):
    """nn.ConvTranspose{2,3}d (ae:66-76) on the convolution data-gradient / forward / wgrad kernels."""
    ops = _ops()
    N, Cin, Cout, sp, k, s, p = case
    op = tuple(si - 1 for si in s)
    g = torch.Generator().manual_seed(hash(case) % 10000)
    x = torch.randn((N, Cin, *sp), generator=g)
    w = torch.randn((Cin, Cout, *k), generator=g) / math.sqrt(Cin * math.prod(k))
    b = torch.randn(Cout, generator=g) * 0.1
    if dtype == torch.bfloat16:
        x, w = bf16_round(x), bf16_round(w)
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    fn = F.conv_transpose3d if len(sp) == 3 else F.conv_transpose2d
    y_ref = fn(xr, wr, br, stride=s, padding=p, output_padding=op)
    dy = torch.randn(y_ref.shape, generator=g)
    if dtype == torch.bfloat16:
        dy = bf16_round(dy)
    y_ref.backward(dy)
    fmt = torch.channels_last_3d if len(sp) == 3 else torch.channels_last
    xd = x.to(DEV).to(dtype).contiguous(memory_format=fmt).requires_grad_(True)
    wd = w.to(DEV).contiguous(memory_format=fmt).requires_grad_(True)
    bd = b.to(DEV).requires_grad_(True)
    y = ops.conv_transpose_nd(xd, wd, bd, s, p, op)
    y.backward(dy.to(DEV).to(dtype))
    tol = 1e-4 if dtype == torch.float32 else BF16_TOL
    assert y.shape == y_ref.shape
    assert rel_err(y, y_ref) < tol
    assert rel_err(xd.grad, xr.grad) < tol
    assert rel_err(wd.grad, wr.grad) < tol
    assert rel_err(bd.grad, br.grad) < tol


@pytest.mark.parametrize("B,L,C,heads", [(2, 300, 128, 1), (1, 200, 128, 2), (1, 1728, 512, 1), (2, 216, 768, 1)])
def test_flash_attention_reads_fused_qkv_in_place(B, L, C, heads):
    """mig_flash_attention_fwd_ld: q / k / v as the column blocks of ONE (B, L, 3C) projection output (row pitch 3C) must
    give bit-identical results to contiguous copies of the same data -- same kernels, same tiles, only the tensor-map
    strides differ. Covers the two-query-tile kernel (head dim 64 / 128) and the two-pass kernels (512 / 768)."""
    ops = _ops()
    g = torch.Generator().manual_seed(L + C)
    qkv = bf16_round(torch.randn(B, L, 3 * C, generator=g)).to(DEV).bfloat16()
    q, k, v = (qkv[:, :, i * C:(i + 1) * C] for i in range(3))
    scale = 1 / math.sqrt(C / heads)
    assert ops._row_pitch(q) == 3 * C and ops._row_pitch(v) == 3 * C
    got, lse = ops._flash_fwd(q, k, v, heads, scale)
    want, lse_w = ops._flash_fwd(q.contiguous(), k.contiguous(), v.contiguous(), heads, scale)
    assert got.is_contiguous() and torch.equal(got, want) and torch.equal(lse, lse_w)
    with torch.no_grad():
        fused = ops.sdpa_qkv(qkv, heads, scale)            # no gradient needed: no copies, strided read
    assert torch.equal(fused, want)


@pytest.mark.parametrize("C,nhc", [(128, 128), (128, 64), (512, 512), (32, 32)])
def test_attention_block_inference_uses_one_projection(C, nhc):
    """SelfAttentionBlock under no_grad in bf16 (the sampling path) projects q, k, v with ONE GEMM on a cached stacked
    weight and lets attention read the column blocks in place; it must match the three-GEMM path that runs when
    gradients are enabled, and follow in-place weight changes (the cache is keyed by the parameters' versions)."""
    from medical_image_generation_b200.layers import SelfAttentionBlock
    torch.manual_seed(C + nhc)
    blk = SelfAttentionBlock(3, C, num_head_channels=nhc, norm_num_groups=32).to(DEV)
    x = torch.randn(2, C, 6, 6, 5, device=DEV).bfloat16()
    with torch.enable_grad():
        ref = blk(x.clone().requires_grad_(True)).detach()
    with torch.no_grad():
        got = blk(x)
    assert "_mig_qkv_eval" in blk.__dict__
    assert rel_err(got, ref) < 5e-3
    with torch.no_grad():
        blk.to_v.weight.mul_(0.5)
        got2 = blk(x)
    with torch.enable_grad():
        ref2 = blk(x.clone().requires_grad_(True)).detach()
    assert rel_err(got2, ref2) < 5e-3 and rel_err(got2, got) > 1e-3


@pytest.mark.parametrize("C,heads", [(128, 1), (256, 2), (512, 1)])
def test_flash_attention_growing_logits(C, heads):
    """Keys whose logits grow tile after tile: every key tile raises the running row maximum by far more than the lazy
    rescale threshold (2^8), so the online-softmax kernel (head dim <= 256) must rescale its tensor-memory accumulator
    each time; a peaked and a flat row distribution are both present. The two-pass kernel (head dim 512) sees the
    same data."""
    ops = _ops()
    B, Lq, Lk = 1, 256, 1024
    g = torch.Generator().manual_seed(7 + C)
    q, k, v = (torch.randn(B, L, C, generator=g) for L in (Lq, Lk, Lk))
    ramp = torch.linspace(0.2, 6.0, Lk).reshape(1, Lk, 1)          # later keys are much "louder"
    k = k * ramp
    q[:, ::2] *= 3.0                                               # half of the rows very peaked
    q, k, v = bf16_round(q), bf16_round(k), bf16_round(v)
    scale = 1 / math.sqrt(C / heads)

    def split(t):
        return t.reshape(B, -1, heads, C // heads).permute(0, 2, 1, 3)

    p = torch.softmax(split(q) @ split(k).transpose(-1, -2) * scale, dim=-1)
    want = (p @ split(v)).permute(0, 2, 1, 3).reshape(B, Lq, C)
    qd, kd, vd = (t.to(DEV).bfloat16() for t in (q, k, v))
    with torch.no_grad():
        got = ops.sdpa(qd, kd, vd, heads, scale)
    assert torch.isfinite(got).all() and rel_err(got, want) < BF16_TOL


# ---- nearest upsample folded into the convolution (ops.upsample_conv_nd, csrc/upconv.cu; unet:576-584, ae:97-106) ----
def _upconv_ref(x, w, b, f, p):
    xu = x
    for i, fi in enumerate(f):
        xu = xu.repeat_interleave(fi, dim=2 + i)          # F.interpolate(mode="nearest") for integer factors
    conv = F.conv3d if x.ndim == 5 else F.conv2d
    return conv(xu, w, b, stride=1, padding=p)


# (N, Cin, Cout, low-resolution spatial, factors)
UPCONV_CASES = [
    (2, 64, 64, (4, 6, 8), (2, 2, 2)),
    (1, 128, 64, (5, 7, 3), (2, 2, 1)),       # anisotropic level (config 4 strides [2, 2, 1]), odd sizes
    (2, 64, 128, (8, 8), (2, 2)),             # 2-D
    (1, 64, 64, (3, 4, 16), (1, 2, 2)),
    (2, 512, 512, (6, 6, 6), (2, 2, 2)),      # LDM width
]


@pytest.mark.parametrize("direct", [True, False])
@pytest.mark.parametrize("case", UPCONV_CASES)
def test_upsample_conv_folded_matches_reference_and_unfolded(case, direct, monkeypatch):
    """Folded path vs (a) torch's interpolate + conv on the same bf16-rounded operands, (b) the two separate operators.
    direct: the forward classes scatter straight into the output (large levels) / go through class buffers + interleave."""
    ops = _ops()
    monkeypatch.setattr(ops, "_UPCONV_DIRECT", direct)
    monkeypatch.setattr(ops, "_UPCONV_MIN_TILES", 0)
    N, Cin, Cout, low, f = case
    nd = len(low)
    k, p = (3,) * nd, (1,) * nd
    g = torch.Generator().manual_seed(sum(low) + Cin)
    x = bf16_round(torch.randn((N, Cin, *low), generator=g))
    w = bf16_round(torch.randn((Cout, Cin, *k), generator=g) / math.sqrt(Cin * math.prod(k)))
    b = torch.randn(Cout, generator=g) * 0.1
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    y_ref = _upconv_ref(xr, wr, br, f, p)
    probe = torch.randn(y_ref.shape, generator=g)
    (y_ref * probe).sum().backward()
    got = {}
    for mode in ("always", "never"):
        ops.set_upconv(mode)
        try:
            xd = _cl(x.to(DEV).to(torch.bfloat16)).requires_grad_(True)
            wd = _cl(w.to(DEV)).requires_grad_(True)
            bd = b.to(DEV).requires_grad_(True)
            assert ops.upconv_usable(xd, wd, f, p) == (mode == "always")
            y = ops.upsample_conv_nd(xd, wd, bd, f, p)
            assert y.shape == y_ref.shape and y.dtype == torch.bfloat16
            (y.float() * probe.to(DEV)).sum().backward()
            got[mode] = (y, xd.grad, wd.grad, bd.grad)
        finally:
            ops.set_upconv("auto")
        assert rel_err(y, y_ref) < BF16_TOL, mode
        assert rel_err(xd.grad, xr.grad) < BF16_TOL, mode
        assert rel_err(wd.grad, wr.grad) < BF16_TOL, mode
        assert rel_err(bd.grad, br.grad) < BF16_TOL, mode
        assert wd.grad.dtype == torch.float32
    # the fold only changes where bf16 rounding happens (summed taps are rounded once more): close to the unfolded path
    for a, c in zip(got["always"], got["never"]):
        assert rel_err(a, c) < BF16_TOL


def test_upconv_fold_tables_match_a_torch_restatement():
    """mig_upconv_fold_filter / _unfold_wgrad / mig_class_interleave against index arithmetic written out in torch."""
    import ctypes as C
    import itertools
    from medical_image_generation_b200 import _lib
    ops = _ops()
    I3 = C.c_int32 * 3
    lib = _lib.load()
    for k3, f3, p3 in [((3, 3, 3), (2, 2, 2), (1, 1, 1)), ((3, 3, 3), (2, 2, 1), (1, 1, 1)), ((1, 3, 3), (1, 2, 2), (0, 1, 1)),
                       ((3, 3, 3), (1, 2, 1), (1, 1, 1))]:
        Cout, Cin = 40, 24
        g = torch.Generator().manual_seed(sum(f3))
        w = bf16_round(torch.randn(Cout, math.prod(k3), Cin, generator=g))
        wd = w.to(DEV).to(torch.bfloat16)
        folds = [ops._axis_fold(k3[i], f3[i], p3[i]) for i in range(3)]
        # forward fold
        n0 = int(lib.mig_upconv_folded_elems(Cout, Cin, I3(*k3), I3(*f3), I3(*p3), 0))
        out = torch.empty(n0, dtype=torch.bfloat16, device=DEV)
        _lib.call("mig_upconv_fold_filter", ops._ptr(wd), ops._ptr(out), Cout, Cin, I3(*k3), I3(*f3), I3(*p3), 0, ops._stream())
        want, dwc_parts, umaps = [], [], []
        for r in itertools.product(*[range(v) for v in f3]):
            base = [folds[i][r[i]][0] for i in range(3)]
            nu = [folds[i][r[i]][1] for i in range(3)]
            wc = torch.zeros(Cout, math.prod(nu), Cin)
            umap = {}
            for t in itertools.product(*[range(v) for v in k3]):
                u = [(r[i] + t[i] - p3[i]) // f3[i] - base[i] for i in range(3)]
                ui = (u[0] * nu[1] + u[1]) * nu[2] + u[2]
                ti = (t[0] * k3[1] + t[1]) * k3[2] + t[2]
                wc[:, ui] += w[:, ti]
                umap[ti] = ui
            want.append(wc.reshape(-1))
            umaps.append((umap, math.prod(nu)))
        want = torch.cat(want)
        assert want.numel() == n0
        assert torch.equal(out.float().cpu(), bf16_round(want))
        # dgrad fold: [Cin][s][Cout]
        K2 = [f3[i] + k3[i] - 1 for i in range(3)]
        pad2 = [k3[i] - 1 - p3[i] for i in range(3)]
        n1 = int(lib.mig_upconv_folded_elems(Cout, Cin, I3(*k3), I3(*f3), I3(*p3), 1))
        assert n1 == Cin * math.prod(K2) * Cout
        outd = torch.empty(n1, dtype=torch.bfloat16, device=DEV)
        _lib.call("mig_upconv_fold_filter", ops._ptr(wd), ops._ptr(outd), Cout, Cin, I3(*k3), I3(*f3), I3(*p3), 1, ops._stream())
        wantd = torch.zeros(Cin, math.prod(K2), Cout)
        for s in itertools.product(*[range(v) for v in K2]):
            si = (s[0] * K2[1] + s[1]) * K2[2] + s[2]
            for t in itertools.product(*[range(v) for v in k3]):
                if all(0 <= (s[i] - pad2[i]) + t[i] - p3[i] < f3[i] for i in range(3)):
                    wantd[:, si] += w[:, (t[0] * k3[1] + t[1]) * k3[2] + t[2]].t()
        assert torch.equal(outd.float().cpu().reshape(wantd.shape), bf16_round(wantd))
        # wgrad unfold (accumulates)
        dwc = torch.randn(n0, generator=g)
        dw0 = torch.randn(Cout, math.prod(k3), Cin, generator=g)
        dwd = dw0.clone().to(DEV)
        _lib.call("mig_upconv_unfold_wgrad", ops._ptr(dwc.to(DEV)), ops._ptr(dwd), Cout, Cin, I3(*k3), I3(*f3), I3(*p3),
                  ops._stream())
        wantw, off = dw0.clone(), 0
        for umap, U in umaps:
            blk = dwc[off:off + Cout * U * Cin].reshape(Cout, U, Cin)
            for ti, ui in umap.items():
                wantw[:, ti] += blk[:, ui]
            off += Cout * U * Cin
        assert torch.allclose(dwd.cpu(), wantw, rtol=1e-6, atol=1e-6)
        # interleave both ways
        N, low, Cc = 2, (3, 2, 5), 24
        full = torch.randn(N, low[0] * f3[0], low[1] * f3[1], low[2] * f3[2], Cc, generator=g).to(torch.bfloat16)
        cls = torch.empty(full.numel(), dtype=torch.bfloat16, device=DEV)
        _lib.call("mig_class_interleave", 1, ops._ptr(full.to(DEV)), ops._ptr(cls), N, I3(*low), I3(*f3), Cc, 1, ops._stream())
        wantc = torch.cat([full[:, r[0]::f3[0], r[1]::f3[1], r[2]::f3[2]].reshape(-1)
                           for r in itertools.product(*[range(v) for v in f3])])
        assert torch.equal(cls.cpu(), wantc)
        back = torch.empty_like(full, device=DEV)
        _lib.call("mig_class_interleave", 1, ops._ptr(cls), ops._ptr(back), N, I3(*low), I3(*f3), Cc, 0, ops._stream())
        assert torch.equal(back.cpu(), full)


def test_upconv_cost_model_and_fallbacks():
    ops = _ops()
    w512 = _cl(torch.zeros(512, 512, 3, 3, 3, device=DEV))
    x24 = _cl(torch.zeros(8, 512, 12, 12, 12, device=DEV, dtype=torch.bfloat16))
    x12 = _cl(torch.zeros(8, 768, 6, 6, 6, device=DEV, dtype=torch.bfloat16))
    w768 = _cl(torch.zeros(768, 768, 3, 3, 3, device=DEV))
    assert ops.upconv_usable(x24, w512, (2, 2, 2), (1, 1, 1))            # the largest layer of the LDM U-Net: folded
    assert not ops.upconv_usable(x12, w768, (2, 2, 2), (1, 1, 1))        # 6^3 level: one class does not fill the GPU
    assert not ops.upconv_usable(x24.float(), w512, (2, 2, 2), (1, 1, 1))   # fp32 parity mode keeps the reference order
    assert not ops.upconv_usable(x24, w512, (2, 2, 2), (1, 1, 0))        # the reference's level-padding defect (unet:557-565)
    assert not ops.upconv_usable(x24, w512, (1, 1, 1), (1, 1, 1))
    w48 = _cl(torch.zeros(48, 48, 3, 3, 3, device=DEV))
    assert not ops.upconv_usable(_cl(torch.zeros(2, 48, 32, 32, 32, device=DEV, dtype=torch.bfloat16)), w48, (2, 2, 2), (1, 1, 1))


@pytest.mark.parametrize("cols", [3, 216, 1728, 2048, 2049, 6400])
@pytest.mark.parametrize("pair", ["f32", "f32->bf16", "bf16"])
def test_softmax_kernels_both_row_layouts(cols, pair):
    """mig_softmax_fwd / _bwd (the unfused training attention, unet:414): rows that fit the registers of one CTA
    (<= 2048 columns: LDM levels) and the three-pass kernel for longer ones (config 5: L = 6400), every dtype pair the
    attention uses (fp32 scores -> bf16 probabilities; bf16 P with fp32 dP)."""
    from medical_image_generation_b200 import _lib
    ops = _ops()
    rows, scale = 37, 0.31
    g = torch.Generator().manual_seed(cols)
    x = torch.randn(rows, cols, generator=g) * 3
    ti, to = {"f32": (torch.float32, torch.float32), "f32->bf16": (torch.float32, torch.bfloat16),
              "bf16": (torch.bfloat16, torch.bfloat16)}[pair]
    code = {torch.float32: 0, torch.bfloat16: 1}
    xd = x.to(DEV).to(ti)
    y = torch.empty(rows, cols, dtype=to, device=DEV)
    _lib.call("mig_softmax_fwd", code[ti], code[to], ops._ptr(xd), ops._ptr(y), rows, cols, scale, ops._stream())
    want = torch.softmax(xd.float().cpu() * scale, dim=-1)
    assert rel_err(y, want) < (1e-5 if to == torch.float32 else 4e-3)
    assert torch.allclose(y.float().sum(-1).cpu(), torch.ones(rows), atol=1e-5 if to == torch.float32 else 2e-2)
    # backward: ds = scale * p * (dp - sum(dp * p)); P in `to`, dP / dS in fp32 unless everything is bf16
    td = torch.float32 if pair != "bf16" else torch.bfloat16
    dp = torch.randn(rows, cols, generator=g).to(DEV).to(td)
    ds = torch.empty(rows, cols, dtype=td, device=DEV)
    _lib.call("mig_softmax_bwd", code[to], code[td], ops._ptr(y), ops._ptr(dp), ops._ptr(ds), rows, cols, scale, ops._stream())
    pf, df = y.float().cpu(), dp.float().cpu()
    want_ds = scale * pf * (df - (df * pf).sum(-1, keepdim=True))
    assert rel_err(ds, want_ds) < (1e-5 if td == torch.float32 else 1e-2)
    if pair == "f32->bf16":      # the bf16 training chain: bf16 P, fp32 dP, bf16 dS in one pass
        dsn = torch.empty(rows, cols, dtype=torch.bfloat16, device=DEV)
        _lib.call("mig_softmax_bwd_narrow", ops._ptr(y), ops._ptr(dp), ops._ptr(dsn), rows, cols, scale, ops._stream())
        assert torch.equal(dsn, ds.to(torch.bfloat16))
