"""GPU: every entry of the convolution variant table (conv_plan.py) through the C ABI, against an fp32 CPU reference.

Each case names the kernels its plan launches; the test records the launched kernels with torch.profiler and requires
exactly the variants the restated plan names for this device's SM count. Outputs start as NaN (y, dx, C) so an element
no kernel writes fails; dw, dbias and accumulated GEMM outputs start from random values, since the C ABI accumulates
into them, and the test checks the increment. Results are compared per voxel and per channel as well as globally
(util.local_errors), with the bars of callcheck.BARS; the worst value of each kind is printed at the end of the module.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

import callcheck
import conv_plan as cp
from util import bf16_round, rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _lib():
    from medical_image_generation_b200 import _lib as L
    return L


def _ptr(t, offset=0):
    return None if t is None else C.c_void_p(t.data_ptr() + offset)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _launched(fn):
    """The normalised names of the variant kernels `fn` launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return cp.variant_kernels({cp.normalise(e.name) for e in prof.events()})


def _cl(t):
    """(N, C, *sp) -> contiguous (N, *sp, C)"""
    return t.permute(0, *range(2, t.ndim), 1).contiguous()


def _nc(t):
    """(N, *sp, C) -> (N, C, *sp)"""
    return t.permute(0, t.ndim - 1, *range(1, t.ndim - 1))


@pytest.fixture(scope="module")
def total():
    rep = callcheck._Report("conv variants")
    yield rep
    print(f"\n{torch.cuda.get_device_name(0)}, {_sms()} SMs")
    failures, rep.failures = rep.failures, []
    rep.finish()                    # prints the worst values; the cases have asserted their own failures
    rep.failures = failures


@pytest.fixture(autouse=True)
def _fp32_reference():
    tf = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf


class _Both:
    """Records every check in the case's report and in the module's."""

    def __init__(self, title, total):
        self.rep, self.total = callcheck._Report(title), total

    def local(self, kind, got, want, what):
        for r in (self.rep, self.total):
            r.local(kind, got, want, what)

    def value(self, kind, err, bar, what):
        for r in (self.rep, self.total):
            r.value(kind, err, bar, what)

    def require(self, ok, what):
        self.rep.require(ok, what)

    def written(self, t, what):
        bad = int((~torch.isfinite(t)).sum())
        self.require(bad == 0, f"{what}: {bad} of {t.numel()} elements not written (still NaN) or not finite")

    def kernels(self, got, want, what):
        self.require(got == want, f"{what}: launched {sorted(got)}, the restated plan names {sorted(want)}")


@pytest.mark.parametrize("case", cp.CASES, ids=lambda c: c.id)
def test_conv_variant(case, monkeypatch, total):
    L = _lib()
    lib = L.load()
    g = case.geom
    sms = _sms()
    if case.gn_groups:
        monkeypatch.setenv("MIG_GN_EPILOGUE", "always")      # read on every call
    geom = L.conv_geom(g.N, g.in_dims, g.out_dims, g.Cin, g.Cout, g.ksize, g.stride, g.pad)
    gen = torch.Generator().manual_seed(sum(map(ord, case.id)))
    x = bf16_round(torch.randn((g.N, g.Cin, *g.in_dims), generator=gen))
    w = bf16_round(torch.randn((g.Cout, g.Cin, *g.ksize), generator=gen) / math.sqrt(g.Cin * g.taps))
    b = torch.randn(g.Cout, generator=gen) * 0.1
    cb = torch.randn((g.N, g.Cout), generator=gen) * 0.1 if case.extras else None
    res = bf16_round(torch.randn((g.N, g.Cout, *g.out_dims), generator=gen)) if case.extras else None
    dy = bf16_round(torch.randn((g.N, g.Cout, *g.out_dims), generator=gen))
    xd, wd = _cl(x).to(DEV, torch.bfloat16), _cl(w).to(DEV, torch.bfloat16)
    dyd = _cl(dy).to(DEV, torch.bfloat16)
    shift = 4 if case.bias_shift else 0                   # bias pointer 4 bytes past a 16-byte boundary
    bbuf = torch.zeros(g.Cout + 4, device=DEV)
    bbuf[shift // 4:shift // 4 + g.Cout] = b.to(DEV)
    cbd = cb.to(DEV) if cb is not None else None
    resd = _cl(res).to(DEV, torch.bfloat16) if res is not None else None
    rep = _Both(case.id, total)

    def workspace(which):
        want = case.ws_bytes(which)
        if case.ws == "full":
            got = int(lib.mig_conv_workspace_bytes(C.byref(geom), 1, which, 0))
            rep.require(got == want, f"{cp.PASS_NAMES[which]} workspace: library {got}, restatement {want}")
        return (torch.empty(max(want, 1), dtype=torch.uint8, device=DEV), want) if want else (None, 0)

    def expected(which):
        return cp.conv_kernels(g, which, case.ws_bytes(which), sms=sms, chan_bias=case.extras, residual=case.extras,
                               finish_aligned=not case.bias_shift)

    s, p = tuple(g.stride), tuple(g.pad)
    if "fwd" in case.kernels:
        ws, wsb = workspace(cp.FWD)
        y = torch.full((g.N, *g.out_dims, g.Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
        G = case.gn_groups
        sums = torch.full((g.N, G, 2), float("nan"), device=DEV, dtype=torch.float64) if G else None
        if G:
            rep.require(lib.mig_conv_fwd_stats_in_epilogue(C.byref(geom), 1, G, 0, wsb) == 1,
                        "GroupNorm sums not taken from the epilogue")
            run = lambda: L.call("mig_conv_fwd_stats", C.byref(geom), 1, _ptr(xd), _ptr(wd), _ptr(bbuf, shift),  # noqa
                                 _ptr(cbd), _ptr(resd), _ptr(y), _ptr(sums), G, 0, _ptr(ws), wsb, _stream())
        else:
            run = lambda: L.call("mig_conv_fwd", C.byref(geom), 1, _ptr(xd), _ptr(wd), _ptr(bbuf, shift), _ptr(cbd),  # noqa
                                 _ptr(resd), _ptr(y), 0, _ptr(ws), wsb, _stream())
        rep.kernels(_launched(run), expected(cp.FWD), "fwd")
        want = callcheck._conv_ref(x, w, b, s, p, cb, res)
        rep.written(y, "fwd y")
        rep.local("bf16", _nc(y).cpu(), want, f"fwd {case.id}")
        if G:
            yg = _nc(y).double().cpu().reshape(g.N, G, g.Cout // G, -1)
            s1, s2 = yg.sum(dim=(2, 3)), (yg * yg).sum(dim=(2, 3))
            sums = sums.cpu()
            rep.value("gn_sums_sq", rel_err(sums[..., 1], s2), callcheck.GN_SUMS_BAR, f"epilogue sum y^2 {case.id}")
            rep.value("gn_sums", float((sums[..., 0] - s1).abs().max() / s2.sqrt().max()), callcheck.GN_SUMS_BAR,
                      f"epilogue sum y {case.id} (abs / sqrt(max sum y^2))")
    if "dgrad" in case.kernels:
        ws, wsb = workspace(cp.DGRAD)
        dx = torch.full((g.N, *g.in_dims, g.Cin), float("nan"), device=DEV, dtype=torch.bfloat16)
        run = lambda: L.call("mig_conv_dgrad", C.byref(geom), 1, _ptr(dyd), _ptr(wd), _ptr(dx), 0, _ptr(ws), wsb,  # noqa
                             _stream())
        rep.kernels(_launched(run), expected(cp.DGRAD), "dgrad")
        want = torch.nn.grad.conv3d_input(x.shape, w, dy, s, p)
        rep.written(dx, "dgrad dx")
        rep.local("bf16", _nc(dx).cpu(), want, f"dgrad {case.id}")
    if "wgrad" in case.kernels:
        ws, wsb = workspace(cp.WGRAD)
        # mig_conv_wgrad ACCUMULATES into dw and dbias (include/medimgen_b200.h): start from random values
        dw0 = torch.randn((g.Cout, *g.ksize, g.Cin), generator=gen) * 0.5
        db0 = torch.randn(g.Cout, generator=gen)
        dw, db = dw0.to(DEV), db0.to(DEV)
        run = lambda: L.call("mig_conv_wgrad", C.byref(geom), 1, _ptr(xd), _ptr(dyd), _ptr(dw), _ptr(db), 0, _ptr(ws),  # noqa
                             wsb, _stream())
        rep.kernels(_launched(run), expected(cp.WGRAD), "wgrad")
        want_w = torch.nn.grad.conv3d_weight(x, w.shape, dy, s, p)
        rep.written(dw, "wgrad dw")
        rep.local("fp32", _nc(dw.cpu() - dw0), want_w, f"wgrad dw {case.id}")
        rep.local("fp32", db.cpu() - db0, dy.sum(dim=(0, 2, 3, 4)), f"wgrad dbias {case.id}")
    rep.rep.finish()


@pytest.mark.parametrize("case", cp.GEMM_CASES, ids=lambda c: c.id)
def test_gemm_variant(case, total):
    L = _lib()
    Bo, Bi, M, N, K = case.batch_outer, case.batch_inner, case.M, case.N, case.K
    gen = torch.Generator().manual_seed(M + N + K)
    a = bf16_round(torch.randn((Bo * Bi, M, K), generator=gen))
    bmat = bf16_round(torch.randn((Bo * Bi, N, K), generator=gen) / math.sqrt(K))      # B[b][n][k]
    alpha = 0.5
    ad = a.to(DEV, torch.bfloat16)
    bd = (bmat.transpose(1, 2) if case.b_mn else bmat).contiguous().to(DEV, torch.bfloat16)
    c0 = torch.randn((Bo * Bi, M, N), generator=gen)
    if case.accumulate:
        cd = c0.to(DEV)
    else:
        cd = torch.full((Bo * Bi, M, N), float("nan"), device=DEV, dtype=torch.float32 if case.c_f32 else torch.bfloat16)
    d = L.GemmDesc()
    d.M, d.N, d.K, d.batch_outer, d.batch_inner = M, N, K, Bo, Bi
    d.a_m, d.a_k, d.a_inner, d.a_outer = K, 1, M * K, Bi * M * K
    d.b_k, d.b_n = (N, 1) if case.b_mn else (1, K)
    d.b_inner, d.b_outer = N * K, Bi * N * K
    d.c_m, d.c_n, d.c_inner, d.c_outer = N, 1, M * N, Bi * M * N
    d.alpha, d.accumulate = alpha, int(case.accumulate)
    run = lambda: L.call("mig_gemm_strided", C.byref(d), 1, 0 if case.c_f32 else 1, _ptr(ad), _ptr(bd), _ptr(cd), 0,  # noqa
                         _stream())
    rep = _Both(case.id, total)
    rep.kernels(_launched(run), cp.gemm_kernels(M, N, K), "gemm")
    want = alpha * torch.bmm(a, bmat.transpose(1, 2))
    got = cd.float().cpu() - (c0 if case.accumulate else 0)
    rep.written(cd, "gemm C")
    rep.local("fp32" if case.c_f32 else "bf16", got.transpose(1, 2), want.transpose(1, 2), f"gemm {case.id}")
    rep.rep.finish()


@pytest.mark.parametrize("case", cp.UPCONV_CASES, ids=lambda c: c.id)
def test_upconv_variant(case, total):
    L = _lib()
    lib = L.load()
    I3 = C.c_int32 * 3
    N, low, Cin, Cout = case.N, case.low, case.Cin, case.Cout
    kk, ff, pp = I3(*case.k), I3(*case.f), I3(*case.p)
    assert lib.mig_upconv_fwd_direct_ok(N, I3(*low), Cin, Cout) == 1
    gen = torch.Generator().manual_seed(Cin * Cout + sum(low))
    x = bf16_round(torch.randn((N, Cin, *low), generator=gen))
    w = bf16_round(torch.randn((Cout, Cin, *case.k), generator=gen) / math.sqrt(Cin * math.prod(case.k)))
    b = torch.randn(Cout, generator=gen) * 0.1
    xd, wd, bd = _cl(x).to(DEV, torch.bfloat16), _cl(w).to(DEV, torch.bfloat16), b.to(DEV)
    folded = torch.empty(int(lib.mig_upconv_folded_elems(Cout, Cin, kk, ff, pp, 0)), device=DEV, dtype=torch.bfloat16)
    L.call("mig_upconv_fold_filter", _ptr(wd), _ptr(folded), Cout, Cin, kk, ff, pp, 0, _stream())
    out = tuple(low[i] * case.f[i] for i in range(3))
    y = torch.full((N, *out, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    run = lambda: L.call("mig_upconv_fwd", _ptr(xd), _ptr(folded), _ptr(bd), _ptr(y), N, I3(*low), Cin, Cout, kk, ff,  # noqa
                         pp, _stream())
    rep = _Both(case.id, total)
    rep.kernels(_launched(run), cp.upconv_kernels(N, low, Cin, Cout, case.k, case.f, case.p, sms=_sms()), "upconv")
    want = F.conv3d(callcheck._nearest(x, case.f), w, b, padding=case.p)
    rep.written(y, "upconv y")
    rep.local("bf16", _nc(y).cpu(), want, f"upconv {case.id}")
    rep.rep.finish()
