"""The convolution dispatcher's host plan, restated in Python (TEST CODE, not collected).

Given a convolution geometry, a pass (fwd, dgrad or wgrad), the workspace the call gets and an SM count, `conv_kernels`
returns the names of the variant kernels the C entry points launch (e.g. {"conv_tma_kernel<128,2,1>"} or
{"conv_tma_kernel<256,1,0>", "tma_splitk_finish8"}); `gemm_kernels` and `upconv_kernels` do the same for
mig_gemm_strided and mig_upconv_fwd. Each function restates one C++ function line for line and names it, so that a
change to the tile plan shows up here as a disagreement with the kernels the profiler records.

Names are normalised (`normalise`): no namespace, no spaces, booleans as 0 / 1, and conv_tma_kernel always with its
third (BMN) argument. The cached A/B environment switches (MIG_DISABLE_*, MIG_DGRAD_TRANSPOSE, MIG_CONV_SCHED, ...) are
taken at their defaults.

`CASES`, `GEMM_CASES` and `UPCONV_CASES` are the variant table: each entry says which plan it exists to reach, and
tests/test_conv_variants.py checks that the restatement agrees with that claim.
"""
from __future__ import annotations

import math
import re
from dataclasses import dataclass, field

SMS_B200 = 148
FWD, DGRAD, WGRAD = 0, 1, 2
PASS_NAMES = ("fwd", "dgrad", "wgrad")

TBM, TBK = 128, 64                 # conv_tma.cu / gemm_tc.cu
HT_X, HT_Y, H_C = 8, 16, 32        # conv_halo.cu
BF16_T = "__nv_bfloat16"


# ------------------------------------------------------------------------------------------------------------------
# kernel names
# ------------------------------------------------------------------------------------------------------------------
def normalise(name: str) -> str:
    """A profiler kernel name ("void mig::conv_tma_kernel<256, 2, false>(CUtensorMap, ...)") in the form used here."""
    n = name.strip()
    if n.startswith("void "):
        n = n[5:]
    depth, cut = 0, len(n)
    for i, ch in enumerate(n):          # the argument list starts at the first "(" outside the template brackets
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            cut = i
            break
    n = n[:cut]
    n = re.sub(r"\b(?:mig|tc)::", "", n).replace(" ", "")
    n = re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", n))
    m = re.fullmatch(r"conv_tma_kernel<(\d+),(\d+)>", n)
    if m:                               # BMN defaults to false
        n = f"conv_tma_kernel<{m.group(1)},{m.group(2)},0>"
    return n


def conv_tma(bn, mt, bmn):
    return f"conv_tma_kernel<{bn},{mt},{int(bmn)}>"


# every family of kernels a convolution / strided GEMM call may launch as its main work; tests compare the launched
# kernels of these families with the restatement (helper kernels such as filter transposes and memsets are not listed)
VARIANT_FAMILIES = ("conv_tma_kernel", "wgrad_tma_kernel", "tma_splitk_finish", "tma_splitk_finish8", "conv_tc_kernel",
                    "splitk_finish_kernel", "wgrad_tc_kernel", "gemm_tc_kernel", "thin_conv_kernel", "thin_wgrad_kernel",
                    "thin_wgrad_k3_kernel", "conv_halo_kernel", "wgrad_halo_kernel", "skinny_fwd_kernel",
                    "skinny_dgrad_kernel", "skinny_wgrad_kernel", "pad_channels_kernel", "unpad_add_kernel",
                    "conv_igemm_kernel", "conv_wgrad_kernel", "gemm_strided_kernel")


def family(name: str) -> str:
    return name.split("<", 1)[0]


def variant_kernels(names) -> set:
    return {n for n in names if family(n) in VARIANT_FAMILIES}


# ------------------------------------------------------------------------------------------------------------------
# geometry
# ------------------------------------------------------------------------------------------------------------------
def cdiv(a, b):
    """C integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


@dataclass(frozen=True)
class Geom:
    """mig_conv_geom; out_dims follow from the others."""
    N: int
    in_dims: tuple
    Cin: int
    Cout: int
    ksize: tuple = (3, 3, 3)
    stride: tuple = (1, 1, 1)
    pad: tuple = (1, 1, 1)

    @property
    def out_dims(self):
        return tuple((self.in_dims[i] + 2 * self.pad[i] - self.ksize[i]) // self.stride[i] + 1 for i in range(3))

    @property
    def taps(self):
        return math.prod(self.ksize)

    def in_vox(self):
        return self.N * math.prod(self.in_dims)

    def out_vox(self):
        return self.N * math.prod(self.out_dims)

    def replace(self, **kw):
        d = dict(N=self.N, in_dims=self.in_dims, Cin=self.Cin, Cout=self.Cout, ksize=self.ksize, stride=self.stride,
                 pad=self.pad)
        d.update(kw)
        return Geom(**d)


def pick_bn(cdst):
    """tc_host.cuh: pick_bn."""
    return 256 if cdst > 128 else (128 if cdst > 64 else (64 if cdst > 32 else 32))


# ------------------------------------------------------------------------------------------------------------------
# TMA box engine (conv_tma.cu)
# ------------------------------------------------------------------------------------------------------------------
_BOX_CAND = ((1, 8, 8), (2, 4, 8), (4, 2, 8), (8, 1, 8), (1, 4, 16), (2, 2, 16), (4, 1, 16), (4, 4, 4), (2, 8, 4),
             (8, 2, 4), (1, 16, 4), (16, 1, 4), (1, 2, 32), (2, 1, 32), (1, 1, 64), (8, 4, 2), (4, 8, 2), (16, 2, 2),
             (2, 16, 2), (8, 8, 1), (16, 4, 1), (4, 16, 1))


def _cover(D, H, W, box):
    return float((D + box[0] - 1) // box[0] * box[0]) * ((H + box[1] - 1) // box[1] * box[1]) * \
        ((W + box[2] - 1) // box[2] * box[2])


def pick_box(D, H, W):
    """conv_tma.cu: pick_box. Returns (ok, (bd, bh, bw)); the box is None when no candidate improved on 0."""
    best, box = 0.0, None
    for c in _BOX_CAND:
        eff = float(D * H * W) / _cover(D, H, W, c)
        if eff > best + 1e-9:
            best, box = eff, c
    return best >= 0.5, box


def pick_box_k(D, H, W):
    """conv_tma.cu: pick_box_k (wgrad: a box is one K stage, any multiple of 16 voxels up to 64)."""
    ok, box = pick_box(D, H, W)
    best = 0.0
    if ok:
        best = float(D * H * W) / _cover(D, H, W, box)
    if best >= 0.8:
        return True, box
    best_s = best * 64.0 / 72.0
    d = 1
    while d <= D and d <= 64:
        h = 1
        while h <= H and d * h <= 64:
            w = 1
            while w <= W and d * h * w <= 64:
                nb = d * h * w
                if nb % 16 == 0:
                    boxes = float((D + d - 1) // d) * ((H + h - 1) // h) * ((W + w - 1) // w)
                    sc = float(D * H * W) / (boxes * nb) * nb / (nb + 8.0)
                    if sc > best_s + 0.05:
                        best_s, box, ok = sc, (d, h, w), True
                w += 1
            h += 1
        d += 1
    return ok and best_s * 72.0 / 64.0 >= 0.5, box


def pick_box_rows(D, H, W):
    """conv_tma.cu: pick_box_rows (fwd / dgrad: a box may fill a whole 128-row slot). Returns (ok, box, rb)."""
    best = 0.0
    ok, box = pick_box(D, H, W)
    if ok:
        best = float(D * H * W) / _cover(D, H, W, box)
    if best >= 0.8:
        return True, box, 64
    best128, c = 0.0, (0, 0, 0)
    d = 1
    while d <= D and d <= 128:
        h = 1
        while h <= H and d * h <= 128:
            w = 1
            while w <= W and d * h * w <= 128:
                boxes = float((D + d - 1) // d) * ((H + h - 1) // h) * ((W + w - 1) // w)
                eff = float(D * H * W) / (boxes * 128.0)
                if eff > best128 + 1e-9 or (eff > best128 - 1e-9 and w > c[2]):
                    best128, c = eff, (d, h, w)
                w += 1
            h += 1
        d += 1
    if best128 > best + 0.1:
        return best128 >= 0.5, c, 128
    return ok, box, 64


@dataclass
class BoxGeom:
    """conv_tma.cu: BoxGeom, the fields the plan reads."""
    N: int
    ext: tuple
    box: tuple
    rb: int
    ks: tuple
    Csrc: int
    Cdst: int
    ok: bool = True
    nb: int = field(init=False)
    num_boxes: int = field(init=False)
    K: int = field(init=False)
    cchunks: int = field(init=False)

    def __post_init__(self):
        self.nb = math.prod(self.box)
        self.num_boxes = self.N * math.prod((self.ext[i] + self.box[i] - 1) // self.box[i] for i in range(3))
        self.K = math.prod(self.ks) * self.Csrc
        self.cchunks = (self.Csrc + 63) // 64


def box_geom(pick, N, ext, ks, Csrc, Cdst):
    """conv_tma.cu: box_geom (pick: "box64", "rows" or "stage")."""
    if pick == "rows":
        ok, box, rb = pick_box_rows(*ext)
    elif pick == "stage":
        (ok, box), rb = pick_box_k(*ext), 64
    else:
        (ok, box), rb = pick_box(*ext), 64
    return BoxGeom(N, tuple(ext), box, rb, tuple(ks), Csrc, Cdst, ok)


def make_box_geom(g: Geom, which):
    """conv_tma.cu: make_box_geom."""
    rows = g.in_dims if which == DGRAD else g.out_dims
    return box_geom("stage" if which == WGRAD else "rows", g.N, rows, g.ksize, g.Cout if which == DGRAD else g.Cin,
                    g.Cin if which == DGRAD else g.Cout)


@dataclass
class BoxPlan:
    bn: int
    mt: int
    num_kb: int
    splits: int
    kb_per_split: int
    mtiles: int = 0
    ntiles: int = 0

    @property
    def tiles(self):
        return self.mtiles * self.ntiles * self.splits

    def ctas(self, sms):
        """launch_box_conv: persistent grid, one CTA per SM once there are more tiles than SMs."""
        return min(self.tiles, sms)


def plan_box(b: BoxGeom, ws_bytes, sms) -> BoxPlan:
    """conv_tma.cu: plan_box (plus the tile counts launch_box_conv derives from it)."""
    bn = pick_bn(b.Cdst)
    num_kb = (b.K // b.Csrc) * b.cchunks
    ntiles = (b.Cdst + bn - 1) // bn
    M = b.N * math.prod(b.ext)
    ws_ok = ws_bytes >= M * b.Cdst * 4
    best, mt, splits = 1e30, 1, 1
    for m_ in (1, 2):
        nslot_ = m_ * (TBM // b.rb)
        mtiles_ = (b.num_boxes + nslot_ - 1) // nslot_
        t_stage = max(512.0 * m_ * bn / 256.0, (float(nslot_) * b.nb + bn) * 128.0 / 70.0)
        for s_ in (1, 2, 3, 4, 6, 8, 12, 16):
            if s_ > 1 and (not ws_ok or num_kb // s_ < 4):
                continue
            waves = float((mtiles_ * ntiles * s_ + sms - 1) // sms)
            kb = float((num_kb + s_ - 1) // s_)
            t_epi = 2500.0 + m_ * (bn // 16) * (160.0 if s_ > 1 else 110.0)
            t = waves * (kb * t_stage + t_epi + 9000.0)
            if s_ > 1:
                t += float(M) * b.Cdst * 14.0 / 3000.0 + 8000.0
            if t < best:
                best, mt, splits = t, m_, s_
    kb_per_split = (num_kb + splits - 1) // splits
    splits = (num_kb + kb_per_split - 1) // kb_per_split
    nslot = mt * (TBM // b.rb)
    return BoxPlan(bn, mt, num_kb, splits, kb_per_split, (b.num_boxes + nslot - 1) // nslot, ntiles)


def epilogue_stats_ok(b: BoxGeom, pl: BoxPlan, groups, mode=None):
    """conv_tma.cu: epilogue_stats_ok; `mode` is MIG_GN_EPILOGUE ("always", "never" or None for the default)."""
    if not (pl.splits == 1 and pl.bn >= 64 and b.Cdst % 16 == 0 and groups > 0 and b.Cdst % groups == 0
            and (b.Cdst // groups) % 8 == 0):
        return False
    if mode and mode[0] == "a":
        return True
    if mode and mode[0] == "n":
        return False
    return 2 * pl.mt * pl.bn <= 512


def box_kernels(b: BoxGeom, ws_bytes, sms, bmn=False, finish_aligned=True):
    """conv_tma.cu: launch_box_conv -- the conv kernel of the plan, and the split-K finish pass."""
    pl = plan_box(b, ws_bytes, sms)
    assert not bmn or pl.bn >= 64, "conv_tma: the MN-major filter operand needs at least 64 output channels"
    out = {conv_tma(pl.bn, pl.mt, bmn)}
    if pl.splits > 1:
        out.add("tma_splitk_finish8" if b.Cdst % 8 == 0 and finish_aligned else "tma_splitk_finish")
    return out


def tma_conv_eligible(g: Geom, which):
    """conv_tma.cu: tma_conv_eligible."""
    strided = False
    for i in range(3):
        if g.stride[i] < 1 or g.stride[i] > 2:
            return False
        strided = strided or g.stride[i] != 1
    if strided and which == DGRAD:
        return False
    csrc = g.Cout if which == DGRAD else g.Cin
    if (csrc % 64 != 0) if which == WGRAD else (csrc % 8 != 0 or csrc < (32 if strided else 48)):
        return False
    if which == WGRAD and g.Cout % 8 != 0:
        return False
    dims = g.in_dims if which == DGRAD else g.out_dims
    if float(g.N) * math.prod(dims) > 16.0 * 2147483647.0:
        return False
    if which != WGRAD:
        return pick_box_rows(*dims)[0]
    return pick_box_k(*dims)[0]


def tma_dgrad_bmn(g: Geom):
    """conv_tma.cu: tma_conv_dgrad -- dgrad reads the forward filter as an MN-major operand when Cin % 64 == 0."""
    return g.Cin % 64 == 0


def tma_dgrad_ws(g: Geom, ws_bytes):
    """The workspace the box plan of tma_conv_dgrad sees (the transposed filter copy comes first)."""
    if tma_dgrad_bmn(g):
        return ws_bytes
    wt = (g.Cin * g.taps * g.Cout * 2 + 255) // 256 * 256
    assert ws_bytes >= wt, "conv_dgrad(tma): workspace too small"
    return ws_bytes - wt


def tma_wgrad_plan(g: Geom, sms):
    """conv_tma.cu: tma_conv_wgrad's tile / split plan. Returns (bn, mt, splits, boxes_per_split)."""
    b = make_box_geom(g, WGRAD)
    bn, mt, splits = 64, 1, 1
    best = 1e30
    for bn_, mt_ in ((256, 2), (256, 1), (128, 1), (64, 1)):
        if bn_ > 64 and b.K <= bn_ // 2:
            continue
        if mt_ == 2 and g.Cout <= 128:
            continue
        tiles = ((g.Cout + TBM * mt_ - 1) // (TBM * mt_)) * ((b.K + bn_ - 1) // bn_)
        t_stage = max(512.0 * mt_ * bn_ / 256.0 * b.nb / 64.0, b.nb * 3.5 * (2 * mt_ + bn_ // 64))
        t_epi = 2500.0 + mt_ * 128.0 * bn_ / 5.0
        s_ = 1
        while s_ <= b.num_boxes and s_ <= 4096:
            waves = float((tiles * s_ + sms - 1) // sms)
            st = float((b.num_boxes + s_ - 1) // s_)
            t = waves * (st * t_stage + t_epi + 2500.0)
            if t < best:
                best, bn, mt, splits = t, bn_, mt_, s_
            s_ = s_ + 1 if s_ < 8 else s_ + s_ // 4
    splits = min(splits, 65535)
    per = (b.num_boxes + splits - 1) // splits
    splits = (b.num_boxes + per - 1) // per
    return bn, mt, splits, per


def tma_wgrad_kernel(g: Geom, sms):
    bn, mt, _, _ = tma_wgrad_plan(g, sms)
    return f"wgrad_tma_kernel<{256 if mt == 2 else bn},{mt}>"


# ---- stride-residue classes (residue_classes.cuh) ----
@dataclass
class AxisClass:
    rho: int
    o: int
    ext: int
    nu: int
    base: int


def axis_class(n_in, k, s, p, rho):
    """residue_classes.cuh: axis_class."""
    o = ((rho - p) % s + s) % s
    ext = (n_in - o + s - 1) // s if n_in > o else 0
    nu = (k - rho + s - 1) // s if rho < k else 0
    return AxisClass(rho, o, ext, nu, cdiv(o + p - rho, s))


def residue_classes(g: Geom):
    """residue_classes.cuh: residue_classes -- the classes holding at least one input voxel, as (axes, ntaps)."""
    out = []
    for r0 in range(g.stride[0]):
        for r1 in range(g.stride[1]):
            for r2 in range(g.stride[2]):
                a = [axis_class(g.in_dims[i], g.ksize[i], g.stride[i], g.pad[i], r) for i, r in enumerate((r0, r1, r2))]
                if any(x.ext == 0 for x in a):
                    continue
                out.append((a, a[0].nu * a[1].nu * a[2].nu))
    return out


def tma_dgrad_strided_eligible(g: Geom):
    """conv_tma.cu: tma_dgrad_strided_eligible."""
    anyst = False
    for i in range(3):
        if g.stride[i] < 1 or g.stride[i] > 2:
            return False
        anyst = anyst or g.stride[i] == 2
    if not anyst or g.Cout % 64 != 0 or g.Cin < 8:
        return False
    for a, ntaps in residue_classes(g):
        if ntaps > 32 or not pick_box(a[0].ext, a[1].ext, a[2].ext)[0]:
            return False
    return True


def tma_dgrad_strided_kernels(g: Geom, sms):
    """conv_tma.cu: tma_conv_dgrad_strided -- every class with taps is a box problem without workspace."""
    out = set()
    for a, ntaps in residue_classes(g):
        if ntaps == 0:
            continue
        b = box_geom("box64", g.N, tuple(x.ext for x in a), tuple(x.nu for x in a), g.Cout, g.Cin)
        out |= box_kernels(b, 0, sms)
    return out


# ---- folded upsample convolution (upconv.cu) ----
def upconv_classes(k, f, p):
    """upconv.cu: make_plan and mig_upconv_fwd -- per class (r, nu, base)."""
    out = []
    for r0 in range(f[0]):
        for r1 in range(f[1]):
            for r2 in range(f[2]):
                r = (r0, r1, r2)
                nu, base = [], []
                for i in range(3):
                    ds = [(r[i] + t - p[i]) // f[i] for t in range(k[i])]     # floordiv
                    nu.append(max(ds) - min(ds) + 1)
                    base.append((r[i] - p[i]) // f[i])
                out.append((r, tuple(nu), tuple(base)))
    return out


def upconv_direct_ok(N, low, Cin, Cout):
    """conv_tma.cu: tma_upconv_class_eligible (mig_upconv_fwd_direct_ok on an sm_100 device)."""
    if Cin % 8 != 0 or Cin < 48 or Cout % 8 != 0:
        return False
    if float(N) * math.prod(low) > 16.0 * 2147483647.0:
        return False
    return pick_box(*low)[0]


def upconv_kernels(N, low, Cin, Cout, k, f, p, sms=SMS_B200):
    """mig_upconv_fwd: one box launch per class (tma_upconv_class_fwd), rows scattered to f*j + r."""
    assert upconv_direct_ok(N, low, Cin, Cout), "upconv_fwd: shape not eligible for the tcgen05 box kernel"
    out = set()
    for _, nu, _ in upconv_classes(k, f, p):
        out |= box_kernels(box_geom("box64", N, low, nu, Cin, Cout), 0, sms)
    return out


# ------------------------------------------------------------------------------------------------------------------
# gather engine (gemm_tc.cu, gemm_tc2.cu)
# ------------------------------------------------------------------------------------------------------------------
def gather(g: Geom, which):
    """gemm_simt.cu: make_gather_fwd / make_gather_dgrad -- (M, K, Csrc, Cdst)."""
    if which == DGRAD:
        return g.in_vox(), g.taps * g.Cout, g.Cout, g.Cin
    return g.out_vox(), g.taps * g.Cin, g.Cin, g.Cout


def split_plan(M, K, Cdst, bn, sms):
    """gemm_tc.cu: split_plan. Returns (num_kb, splits, kb_per_split)."""
    num_kb = (K + TBK - 1) // TBK
    tiles = ((M + TBM - 1) // TBM) * ((Cdst + bn - 1) // bn)
    s = 1
    if tiles * 2 <= sms:
        s = sms // tiles
        if s > num_kb // 8:
            s = num_kb // 8
        if s < 1:
            s = 1
    per = (num_kb + s - 1) // s
    s = (num_kb + per - 1) // per
    return num_kb, s, per


def tc_conv_kernels(g: Geom, which, ws_bytes, sms):
    """gemm_tc.cu: tc_conv_fwd / tc_conv_dgrad -> run_conv_tc."""
    M, K, Csrc, Cdst = gather(g, which)
    assert Csrc % 8 == 0 and K % 8 == 0 and M > 0, "conv_tc: shape not eligible"
    if which == DGRAD:
        wt = (g.Cin * g.taps * g.Cout * 2 + 255) // 256 * 256
        assert ws_bytes >= wt, "conv_dgrad(tc): workspace too small"
        ws_bytes -= wt
    bn = pick_bn(Cdst)
    _, splits, _ = split_plan(M, K, Cdst, bn, sms)
    if splits > 1 and ws_bytes < M * Cdst * 4:
        splits = 1
    out = {f"conv_tc_kernel<{bn}>"}
    if splits > 1:
        out.add("splitk_finish_kernel")
    return out


def tc_conv_splits(g: Geom, which, ws_bytes, sms):
    M, K, _, Cdst = gather(g, which)
    if which == DGRAD:
        ws_bytes -= (g.Cin * g.taps * g.Cout * 2 + 255) // 256 * 256
    _, splits, per = split_plan(M, K, Cdst, pick_bn(Cdst), sms)
    return (splits, per) if splits == 1 or ws_bytes >= M * Cdst * 4 else (1, (K + TBK - 1) // TBK)


def tc_wgrad_eligible(g: Geom):
    """gemm_tc2.cu: tc_wgrad_eligible."""
    return g.Cin % 8 == 0 and g.Cout % 8 == 0 and g.out_vox() < (1 << 31)


def tc_wgrad_plan(g: Geom, sms):
    """gemm_tc2.cu: tc_conv_wgrad's tile / split plan. Returns (bn, splits, vox_per_split)."""
    M, K = g.out_vox(), g.taps * g.Cin
    bn = 256 if K > 128 else (128 if K > 64 else 64)
    tiles = ((g.Cout + TBM - 1) // TBM) * ((K + bn - 1) // bn)
    total_st = (M + TBK - 1) // TBK
    splits = (sms * 3 + tiles - 1) // tiles
    if splits > total_st // 4:
        splits = total_st // 4
    splits = max(1, min(splits, 65535))
    per = ((total_st + splits - 1) // splits) * TBK
    return bn, (M + per - 1) // per, per


def tc_gemm_bn(N):
    """gemm_tc2.cu: tc_gemm_strided's output tile."""
    return 256 if N > 128 else (128 if N > 64 else 64)


def gemm_kernels(M, N, K):
    return {f"gemm_tc_kernel<{tc_gemm_bn(N)}>"}


# ------------------------------------------------------------------------------------------------------------------
# halo, thin and skinny kernels
# ------------------------------------------------------------------------------------------------------------------
def halo_conv_eligible(g: Geom, which):
    """conv_halo.cu: halo_conv_eligible."""
    csrc, cdst = (g.Cout, g.Cin) if which == DGRAD else (g.Cin, g.Cout)
    if csrc != H_C or cdst < 1 or cdst > 64:
        return False
    if any(g.stride[i] != 1 or g.ksize[i] > 3 for i in range(3)):
        return False
    od = g.in_dims if which == DGRAD else g.out_dims
    return g.out_vox() >= 32768 and od[2] >= HT_X and od[1] >= HT_Y // 2


def halo_dgrad_strided_eligible(g: Geom):
    """conv_halo.cu: halo_dgrad_strided_eligible."""
    if g.Cout != H_C or g.Cin < 1 or g.Cin > 64:
        return False
    anyst = False
    for i in range(3):
        if g.stride[i] < 1 or g.stride[i] > 2 or g.ksize[i] > 3:
            return False
        anyst = anyst or g.stride[i] == 2
    if not anyst or g.in_vox() < 32768:
        return False
    if any(axis_class(g.in_dims[1], g.ksize[1], g.stride[1], g.pad[1], r).ext < HT_Y // 2 for r in range(g.stride[1])):
        return False
    return all(axis_class(g.in_dims[2], g.ksize[2], g.stride[2], g.pad[2], r).ext >= HT_X for r in range(g.stride[2]))


def halo_wgrad_eligible(g: Geom):
    """conv_halo.cu: halo_wgrad_eligible."""
    if g.Cin != H_C or g.Cout > 32 or g.Cout < 8 or g.Cout % 8 != 0:
        return False
    if any(g.stride[i] != 1 or g.ksize[i] > 3 for i in range(3)):
        return False
    if (g.taps + 1) // 2 * 32 > 512:
        return False
    return g.out_vox() >= 32768 and g.out_dims[2] >= HT_X and g.out_dims[1] >= HT_Y // 2


def thin_conv_eligible(g: Geom, which):
    """conv_thin.cu: thin_conv_eligible."""
    if any(g.stride[i] != 1 or g.ksize[i] > 3 or g.ksize[i] < 1 for i in range(3)):
        return False
    in_thin = g.Cin <= 4 and g.Cout in (32, 64)
    out_thin = g.Cout <= 4 and g.Cin in (32, 64)
    if which == FWD:
        return in_thin
    if which == DGRAD:
        return out_thin
    return (in_thin and g.Cin <= 2) or (out_thin and g.Cout <= 2)


def thin_tile_z(od0):
    """conv_thin.cu: thin_tiles -- the z extent of a tile."""
    return 1 if od0 == 1 else (2 if od0 < 4 else 4)


def thin_wgrad_kernel(g: Geom):
    """conv_thin.cu: thin_conv_wgrad -> launch_thin_wgrad."""
    in_thin = g.Cin <= 2 and g.Cout in (32, 64)
    od = g.out_dims if in_thin else g.in_dims
    CS, CD = (g.Cin, g.Cout) if in_thin else (g.Cout, g.Cin)
    if (CD, CS) not in ((32, 1), (32, 2), (64, 1)):
        CD, CS = 64, 2
    k3 = tuple(g.ksize) == (3, 3, 3) and thin_tile_z(od[0]) == 4
    return f"thin_wgrad{'_k3' if k3 else ''}_kernel<{CD},{CS}>"


def skinny_eligible(g: Geom):
    """small_ops.cu: skinny_eligible."""
    return (g.N * math.prod(g.in_dims) <= 32 and tuple(g.ksize) == (1, 1, 1) and tuple(g.stride) == (1, 1, 1)
            and tuple(g.pad) == (0, 0, 0))


# ------------------------------------------------------------------------------------------------------------------
# the dispatcher (conv.cu), bf16 on a tcgen05 device, engine 0 (auto), 16-byte aligned activations
# ------------------------------------------------------------------------------------------------------------------
def tc_conv_eligible(g: Geom, which):
    """gemm_tc.cu: tc_conv_eligible (bf16)."""
    if which == FWD:
        return g.Cin % 8 == 0
    if which == DGRAD:
        return g.Cout % 8 == 0
    return tc_wgrad_eligible(g)


def pad8(c):
    return (c + 7) // 8 * 8


def up256(v):
    return (v + 255) // 256 * 256


def want_pad(g: Geom, which):
    """conv.cu: want_pad."""
    if tc_conv_eligible(g, which) or g.out_vox() < 4096:
        return False
    if which == FWD:
        return g.Cin % 8 != 0
    if which == DGRAD:
        return g.Cout % 8 != 0
    return g.Cin % 8 != 0 or g.Cout % 8 != 0


def tc_conv_workspace(g: Geom, which):
    """gemm_tc.cu: tc_conv_workspace."""
    wt = up256(g.Cin * g.taps * g.Cout * 2 if which == DGRAD else 0)
    M, _, _, Cdst = gather(g, which)
    return wt + (M * Cdst * 4 if which <= DGRAD else 0)


def pad_workspace(g: Geom, which):
    """conv.cu: pad_workspace."""
    cin, cout, T = pad8(g.Cin), pad8(g.Cout), g.taps
    if which == FWD:
        return up256(g.in_vox() * cin * 2) + up256(g.Cout * T * cin * 2)
    if which == DGRAD:
        return up256(g.out_vox() * cout * 2) + up256(cout * T * g.Cin * 2)
    return up256(g.in_vox() * cin * 2) + up256(g.out_vox() * cout * 2) + up256(cout * T * cin * 4)


def padded_geom(g: Geom, pin, pout):
    return g.replace(Cin=pad8(g.Cin) if pin else g.Cin, Cout=pad8(g.Cout) if pout else g.Cout)


def workspace_bytes(g: Geom, which):
    """conv.cu: mig_conv_workspace_bytes (bf16, engine 0, tcgen05 device)."""
    simt = g.Cin * g.taps * g.Cout * 2 if which == DGRAD else 0
    tc = tc_conv_workspace(g, which)
    if want_pad(g, which):
        tc = pad_workspace(g, which) + tc_conv_workspace(padded_geom(g, which != DGRAD, which != FWD), which)
    return max(simt, tc)


def _run_fwd(g, ws, sms, finish_aligned):
    """conv.cu: run_fwd."""
    if halo_conv_eligible(g, FWD):
        return {"conv_halo_kernel"}
    if tma_conv_eligible(g, FWD):
        return box_kernels(make_box_geom(g, FWD), ws, sms, finish_aligned=finish_aligned)
    return tc_conv_kernels(g, FWD, ws, sms)


def _run_dgrad(g, ws, sms):
    """conv.cu: run_dgrad."""
    if halo_conv_eligible(g, DGRAD):
        assert ws >= g.Cin * g.taps * g.Cout * 2, "conv_dgrad(halo): workspace too small"
        return {"conv_halo_kernel"}
    if halo_dgrad_strided_eligible(g):
        return {"conv_halo_kernel"}
    if tma_conv_eligible(g, DGRAD):
        return box_kernels(make_box_geom(g, DGRAD), tma_dgrad_ws(g, ws), sms, bmn=tma_dgrad_bmn(g))
    if tma_dgrad_strided_eligible(g):
        return tma_dgrad_strided_kernels(g, sms)
    return tc_conv_kernels(g, DGRAD, ws, sms)


def _run_wgrad(g, sms):
    """conv.cu: run_wgrad."""
    if halo_wgrad_eligible(g):
        return {"wgrad_halo_kernel"}
    if tma_conv_eligible(g, WGRAD):
        return {tma_wgrad_kernel(g, sms)}
    bn, _, _ = tc_wgrad_plan(g, sms)
    return {f"wgrad_tc_kernel<{bn}>"}


def engine(g: Geom, which, chan_bias=False, residual=False):
    """Which engine conv.cu picks: skinny, thin, halo, halo-strided, tma, tma-strided, gather, pad (the padded-channel
    route) or simt."""
    if skinny_eligible(g) and not (which == FWD and (chan_bias or residual)):
        return "skinny"
    if thin_conv_eligible(g, which):
        return "thin"
    if tc_conv_eligible(g, which):
        if which == FWD:
            return "halo" if halo_conv_eligible(g, FWD) else ("tma" if tma_conv_eligible(g, FWD) else "gather")
        if which == DGRAD:
            if halo_conv_eligible(g, DGRAD):
                return "halo"
            if halo_dgrad_strided_eligible(g):
                return "halo-strided"
            if tma_conv_eligible(g, DGRAD):
                return "tma"
            return "tma-strided" if tma_dgrad_strided_eligible(g) else "gather"
        return "halo" if halo_wgrad_eligible(g) else ("tma" if tma_conv_eligible(g, WGRAD) else "gather")
    return "pad" if want_pad(g, which) else "simt"


def conv_kernels(g: Geom, which, ws_bytes, sms=SMS_B200, chan_bias=False, residual=False, finish_aligned=True):
    """The variant kernels mig_conv_fwd / mig_conv_dgrad / mig_conv_wgrad launch (conv.cu: conv_fwd_impl,
    mig_conv_dgrad, mig_conv_wgrad). `finish_aligned`: bias, chan_bias, residual and output are 16-byte aligned."""
    if which == FWD:
        if skinny_eligible(g) and not chan_bias and not residual:
            return {f"skinny_fwd_kernel<{BF16_T},8>"}
        if thin_conv_eligible(g, FWD):
            return {f"thin_conv_kernel<{g.Cout}>"}
        if tc_conv_eligible(g, FWD):
            return _run_fwd(g, ws_bytes, sms, finish_aligned)
        if want_pad(g, FWD) and ws_bytes >= workspace_bytes(g, FWD):
            inner = ws_bytes - up256(g.in_vox() * pad8(g.Cin) * 2) - up256(g.Cout * g.taps * pad8(g.Cin) * 2)
            return {f"pad_channels_kernel<{BF16_T}>"} | _run_fwd(padded_geom(g, True, False), inner, sms, finish_aligned)
        return {f"conv_igemm_kernel<{BF16_T}>"}
    if which == DGRAD:
        if skinny_eligible(g):
            return {f"skinny_dgrad_kernel<{BF16_T},8>"}
        if thin_conv_eligible(g, DGRAD):
            return {f"thin_conv_kernel<{g.Cin}>"}
        if tc_conv_eligible(g, DGRAD):
            return _run_dgrad(g, ws_bytes, sms)
        if want_pad(g, DGRAD) and ws_bytes >= workspace_bytes(g, DGRAD):
            cp = pad8(g.Cout)
            inner = ws_bytes - up256(g.out_vox() * cp * 2) - up256(cp * g.taps * g.Cin * 2)
            return {f"pad_channels_kernel<{BF16_T}>"} | _run_dgrad(padded_geom(g, False, True), inner, sms)
        return {f"conv_igemm_kernel<{BF16_T}>"}
    if skinny_eligible(g):
        return {f"skinny_wgrad_kernel<{BF16_T}>"}
    if thin_conv_eligible(g, WGRAD):
        return {thin_wgrad_kernel(g)}
    if tc_conv_eligible(g, WGRAD):
        return _run_wgrad(g, sms)
    if want_pad(g, WGRAD) and ws_bytes >= workspace_bytes(g, WGRAD):
        return {f"pad_channels_kernel<{BF16_T}>", "unpad_add_kernel"} | _run_wgrad(padded_geom(g, True, True), sms)
    return {f"conv_wgrad_kernel<{BF16_T}>"}


def box_plan_of(g: Geom, which, ws_bytes, sms=SMS_B200):
    """The BoxPlan of a pass that runs on the TMA box engine without classes (for the table's claims)."""
    b = make_box_geom(g, which)
    return b, plan_box(b, tma_dgrad_ws(g, ws_bytes) if which == DGRAD else ws_bytes, sms)


def plan_facts(g: Geom, which, ws_bytes, sms=SMS_B200):
    """What a table entry may claim about the box plan of a pass on the TMA engine."""
    b, pl = box_plan_of(g, which, ws_bytes, sms)
    return dict(bn=pl.bn, mt=pl.mt, splits=pl.splits, tiles=pl.tiles, rb=b.rb, box=b.box, valid_rows=b.nb,
                short_last_split=pl.splits > 1 and pl.num_kb % pl.kb_per_split != 0, n_tail=b.Cdst % pl.bn != 0,
                persistent=pl.tiles > sms, last_cta_fewer=pl.tiles > sms and pl.tiles % sms != 0)


# ------------------------------------------------------------------------------------------------------------------
# the variant table
# ------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    """One convolution geometry and the variant kernels each of its passes launches at 148 SMs.

    ws: "full" passes mig_conv_workspace_bytes of the pass, "none" no workspace (split-K impossible);
    bias_shift: the bias pointer sits 4 bytes past a 16-byte boundary (the scalar split-K finish);
    gn_groups: the forward runs as mig_conv_fwd_stats with MIG_GN_EPILOGUE=always;
    extras: the forward also adds a per-sample channel bias and a residual (the skinny kernels take neither);
    plan: pass -> facts of the box plan (`plan_facts`) the entry exists to reach."""
    id: str
    geom: Geom
    why: str
    kernels: dict
    ws: str = "full"
    bias_shift: bool = False
    gn_groups: int = 0
    extras: bool = True
    plan: dict = field(default_factory=dict)

    def ws_bytes(self, which):
        return workspace_bytes(self.geom, which) if self.ws == "full" else 0


K1 = dict(ksize=(1, 1, 1), pad=(0, 0, 0))
S2 = dict(stride=(2, 2, 2))
_F8, _F1 = "tma_splitk_finish8", "tma_splitk_finish"
_PAD = f"pad_channels_kernel<{BF16_T}>"


def _c(id, geom, why, ws="full", bias_shift=False, gn_groups=0, extras=True, plan=None, **kernels):
    return Case(id, geom, why, {k: set(v) for k, v in kernels.items()}, ws, bias_shift, gn_groups, extras, plan or {})


CASES = [
    # ---- TMA box engine, forward: the eight conv_tma_kernel<BN, MT, false> ----
    _c("tma32x1_split", Geom(1, (4, 4, 4), 96, 24), "BN 32, MT 1; split-K 11 x 5 k-blocks of 54: short last slice",
       plan={"fwd": dict(bn=32, mt=1, splits=11, short_last_split=True)},
       fwd=[conv_tma(32, 1, 0), _F8], dgrad=["conv_tc_kernel<128>"], wgrad=["wgrad_tc_kernel<256>"]),
    _c("tma32x1_nows", Geom(1, (4, 4, 4), 96, 24), "the same shape without workspace: one split, no finish pass",
       ws="none", plan={"fwd": dict(bn=32, mt=1, splits=1)}, fwd=[conv_tma(32, 1, 0)]),
    _c("tma32x2_eq_sms", Geom(1, (37, 32, 32), 48, 3, **K1), "BN 32, MT 2; exactly 148 tiles = one per SM; 3 outputs",
       plan={"fwd": dict(bn=32, mt=2, tiles=148, splits=1)},
       fwd=[conv_tma(32, 2, 0)], dgrad=["conv_tc_kernel<64>", _PAD],
       wgrad=[_PAD, "unpad_add_kernel", "wgrad_tc_kernel<64>"]),
    _c("tma32x2_sms_plus1", Geom(2, (33, 24, 24), 48, 3, **K1), "149 tiles: CTA 0 walks a second tile",
       plan={"fwd": dict(bn=32, mt=2, tiles=149, persistent=True)}, fwd=[conv_tma(32, 2, 0)]),
    _c("tma32x2_persist_split", Geom(4, (16, 16, 24), 320, 24),
       "persistence AND split-K: 288 tiles (96 m-tiles x 3 splits) on 148 CTAs",
       plan={"fwd": dict(bn=32, mt=2, splits=3, tiles=288, persistent=True, last_cta_fewer=True)},
       fwd=[conv_tma(32, 2, 0), _F8]),
    _c("tma32x2_rows128", Geom(3, (5, 5, 24), 256, 16),
       "1x5x24 boxes in 128-row slots (120 valid rows) with MT 2, split-K 16 with a short last slice",
       plan={"fwd": dict(bn=32, mt=2, rb=128, valid_rows=120, splits=16, short_last_split=True)},
       fwd=[conv_tma(32, 2, 0), _F8]),
    _c("tma64x1_split", Geom(1, (4, 4, 4), 96, 40), "BN 64, MT 1 with an N tail (40 of 64); split-K short last slice",
       plan={"fwd": dict(bn=64, mt=1, splits=11, short_last_split=True, n_tail=True)},
       fwd=[conv_tma(64, 1, 0), _F8], dgrad=["conv_tc_kernel<128>", "splitk_finish_kernel"],
       wgrad=["wgrad_tc_kernel<256>"]),
    _c("tma64x1_split_unaligned_bias", Geom(1, (4, 4, 4), 96, 40), "bias 4 bytes off: the scalar split-K finish",
       bias_shift=True, plan={"fwd": dict(bn=64, mt=1, splits=11)}, fwd=[conv_tma(64, 1, 0), _F1]),
    _c("tma128x1_split_c100", Geom(1, (4, 4, 4), 48, 100), "split-K with Cdst % 8 != 0: the scalar split-K finish",
       plan={"fwd": dict(bn=128, mt=1, splits=6, short_last_split=True, n_tail=True)},
       fwd=[conv_tma(128, 1, 0), _F1]),
    _c("tma64x2_gn", Geom(4, (16, 16, 24), 48, 64, **K1), "BN 64, MT 2; GroupNorm sums from the epilogue (8 groups)",
       gn_groups=8, plan={"fwd": dict(bn=64, mt=2, splits=1), "dgrad": dict(bn=64, mt=2)},
       fwd=[conv_tma(64, 2, 0)], dgrad=[conv_tma(64, 2, 0)], wgrad=["wgrad_tc_kernel<64>"]),
    _c("tma128x2_gn", Geom(4, (16, 16, 24), 48, 96, **K1), "BN 128, MT 2, N tail; GroupNorm sums, 12 groups of 8",
       gn_groups=12, plan={"fwd": dict(bn=128, mt=2, splits=1, n_tail=True)}, fwd=[conv_tma(128, 2, 0)]),
    _c("tma256x2_persist", Geom(4, (16, 16, 24), 48, 320, **K1),
       "BN 256, MT 2: 192 tiles on 148 CTAs (the last CTAs walk one tile fewer); N tail 320 = 256 + 64",
       plan={"fwd": dict(bn=256, mt=2, tiles=192, persistent=True, last_cta_fewer=True, n_tail=True)},
       fwd=[conv_tma(256, 2, 0)], dgrad=[conv_tma(64, 2, 0)], wgrad=["wgrad_tc_kernel<64>"]),
    _c("tma256x2_gn", Geom(3, (12, 12, 24), 48, 320, **K1), "BN 256, MT 2 with GroupNorm sums (40 groups), two N tiles",
       gn_groups=40, plan={"fwd": dict(bn=256, mt=2, splits=1, n_tail=True)}, fwd=[conv_tma(256, 2, 0)]),
    _c("tma256x1_split", Geom(1, (4, 4, 4), 48, 192), "BN 256, MT 1, split-K 6 x 5 of 27 k-blocks",
       plan={"fwd": dict(bn=256, mt=1, splits=6, short_last_split=True)},
       fwd=[conv_tma(256, 1, 0), _F8], dgrad=[conv_tma(64, 1, 0), _F8], wgrad=["wgrad_tc_kernel<256>"]),
    _c("gn64x1", Geom(1, (3, 4, 4), 48, 64, **K1), "GroupNorm sums from the BN 64, MT 1 epilogue (one 3x4x4 box)",
       gn_groups=8, plan={"fwd": dict(bn=64, mt=1, splits=1)}, fwd=[conv_tma(64, 1, 0)]),
    _c("gn128x1", Geom(1, (3, 4, 4), 48, 96, **K1), "GroupNorm sums from the BN 128, MT 1 epilogue, 24 channels a group",
       gn_groups=4, plan={"fwd": dict(bn=128, mt=1, splits=1)}, fwd=[conv_tma(128, 1, 0)]),
    _c("gn256x1", Geom(1, (3, 4, 4), 48, 192, **K1), "GroupNorm sums from the BN 256, MT 1 epilogue",
       gn_groups=24, plan={"fwd": dict(bn=256, mt=1, splits=1)}, fwd=[conv_tma(256, 1, 0)]),
    # ---- TMA box engine, dgrad on the MN-major filter: the six conv_tma_kernel<BN, MT, true> ----
    _c("bmn64x1_split", Geom(1, (3, 4, 4), 64, 96), "dgrad BN 64, MT 1 on the forward filter; split-K short slice",
       plan={"dgrad": dict(bn=64, mt=1, splits=11, short_last_split=True)},
       fwd=[conv_tma(128, 1, 0), _F8], dgrad=[conv_tma(64, 1, 1), _F8], wgrad=["wgrad_tma_kernel<64,1>"]),
    _c("bmn64x2", Geom(4, (16, 16, 24), 64, 48, **K1), "dgrad BN 64, MT 2 on the forward filter",
       plan={"dgrad": dict(bn=64, mt=2, splits=1)}, dgrad=[conv_tma(64, 2, 1)], wgrad=["wgrad_tma_kernel<64,1>"]),
    _c("bmn128x1_split", Geom(1, (3, 4, 4), 128, 48), "dgrad BN 128, MT 1 on the forward filter, split-K",
       plan={"dgrad": dict(bn=128, mt=1, splits=6)}, dgrad=[conv_tma(128, 1, 1), _F8]),
    _c("bmn128x2", Geom(4, (16, 16, 24), 128, 48, **K1), "dgrad BN 128, MT 2 on the forward filter",
       plan={"dgrad": dict(bn=128, mt=2, splits=1)}, fwd=[conv_tma(64, 2, 0)], dgrad=[conv_tma(128, 2, 1)]),
    _c("bmn256x1_split", Geom(1, (3, 4, 4), 192, 48), "dgrad BN 256, MT 1 on the forward filter, split-K",
       plan={"dgrad": dict(bn=256, mt=1, splits=6)}, dgrad=[conv_tma(256, 1, 1), _F8]),
    _c("bmn256x2_ntail", Geom(3, (12, 12, 24), 320, 48, **K1), "dgrad BN 256, MT 2 on the forward filter, N tail 320",
       plan={"dgrad": dict(bn=256, mt=2, splits=1, n_tail=True)}, dgrad=[conv_tma(256, 2, 1)]),
    _c("bmn64x1_nows", Geom(1, (3, 4, 4), 64, 96), "the MN-major dgrad without workspace: no split",
       ws="none", plan={"dgrad": dict(bn=64, mt=1, splits=1)}, fwd=[conv_tma(128, 1, 0)], dgrad=[conv_tma(64, 1, 1)]),
    # ---- TMA dgrad through the transposed filter copy (Cin % 64 != 0) ----
    _c("dgradT64", Geom(1, (3, 4, 4), 48, 96), "dgrad Cin 48: transposed filter copy, BN 64, split-K",
       plan={"dgrad": dict(bn=64, mt=1, splits=11)}, dgrad=[conv_tma(64, 1, 0), _F8]),
    _c("dgradT128", Geom(1, (3, 4, 4), 96, 48), "dgrad Cin 96: transposed filter copy, BN 128, split-K",
       plan={"dgrad": dict(bn=128, mt=1, splits=6)}, dgrad=[conv_tma(128, 1, 0), _F8]),
    # ---- TMA wgrad: the four wgrad_tma_kernel<BN, MT> ----
    _c("wgrad64x1", Geom(1, (3, 4, 4), 64, 16, **K1), "wgrad BN 64 (K = 64), a 48-voxel box",
       wgrad=["wgrad_tma_kernel<64,1>"]),
    _c("wgrad128x1", Geom(1, (5, 5, 6), 192, 16), "wgrad BN 128 over 2x4x6 boxes", wgrad=["wgrad_tma_kernel<128,1>"]),
    _c("wgrad256x1", Geom(4, (5, 5, 7), 256, 16), "wgrad BN 256, MT 1", wgrad=["wgrad_tma_kernel<256,1>"]),
    _c("wgrad256x2", Geom(4, (5, 5, 6), 256, 320), "wgrad BN 256, MT 2 (Cout > 128), 320 rows: M tail",
       wgrad=["wgrad_tma_kernel<256,2>"]),
    # ---- stride-2: forward through element-strided tensor maps, dgrad by stride-residue classes ----
    _c("strided_classes_odd", Geom(2, (9, 11, 16), 64, 128, **S2),
       "stride 2 with odd extents: residue classes of different sizes on the box kernel",
       fwd=[conv_tma(128, 1, 0), _F8], dgrad=[conv_tma(64, 1, 0)], wgrad=["wgrad_tma_kernel<64,1>"]),
    _c("strided_k1", Geom(1, (8, 8, 8), 64, 64, **S2, **K1), "kernel 1 stride 2: seven classes get no tap (dx zeroed)",
       fwd=[conv_tma(64, 1, 0)], dgrad=[conv_tma(64, 1, 0)], wgrad=["wgrad_tma_kernel<64,1>"]),
    # ---- gather engine: conv_tc_kernel<32/64/128/256> with and without split-K, wgrad_tc_kernel<64/128/256> ----
    _c("gather32_split", Geom(2, (6, 6, 6), 40, 24), "Cin 40 (< 48: no box), BN 32, split-K 2",
       fwd=["conv_tc_kernel<32>", "splitk_finish_kernel"], dgrad=["conv_tc_kernel<64>"],
       wgrad=["wgrad_tc_kernel<256>"]),
    _c("gather32_nows", Geom(2, (6, 6, 6), 40, 24), "the same without workspace: no split", ws="none",
       fwd=["conv_tc_kernel<32>"]),
    _c("gather64_split", Geom(2, (6, 6, 6), 40, 64), "BN 64, split-K 2",
       fwd=["conv_tc_kernel<64>", "splitk_finish_kernel"], dgrad=[conv_tma(64, 1, 0)]),
    _c("gather64_nows", Geom(2, (6, 6, 6), 40, 64), "BN 64 without workspace", ws="none", fwd=["conv_tc_kernel<64>"]),
    _c("gather128_split", Geom(2, (6, 6, 6), 40, 96), "BN 128 with an N tail, split-K 2",
       fwd=["conv_tc_kernel<128>", "splitk_finish_kernel"], dgrad=[conv_tma(64, 1, 0), _F8]),
    _c("gather128_nows", Geom(2, (6, 6, 6), 40, 96), "BN 128 without workspace", ws="none",
       fwd=["conv_tc_kernel<128>"]),
    _c("gather256_split", Geom(2, (6, 6, 6), 40, 192), "BN 256 with an N tail, split-K 2",
       fwd=["conv_tc_kernel<256>", "splitk_finish_kernel"], dgrad=[conv_tma(64, 1, 0), _F8]),
    _c("gather256_nows", Geom(2, (6, 6, 6), 40, 192), "BN 256 without workspace", ws="none",
       fwd=["conv_tc_kernel<256>"]),
    _c("gather_wgrad128", Geom(2, (6, 6, 6), 96, 40, **K1), "wgrad K = 96 (Cin % 64 != 0): BN 128",
       fwd=[conv_tma(64, 1, 0)], dgrad=["conv_tc_kernel<128>"], wgrad=["wgrad_tc_kernel<128>"]),
    _c("gather_wgrad64", Geom(2, (6, 6, 6), 40, 40, **K1), "wgrad K = 40: BN 64",
       fwd=["conv_tc_kernel<64>"], dgrad=["conv_tc_kernel<64>"], wgrad=["wgrad_tc_kernel<64>"]),
    # ---- thin kernels (1- and 2-channel ends on CUDA cores) ----
    _c("thin32_c1", Geom(1, (12, 20, 24), 1, 32), "conv_in 1 -> 32; wgrad <32, 1> on the 3x3x3 kernel",
       fwd=["thin_conv_kernel<32>"], dgrad=["conv_tc_kernel<32>"], wgrad=["thin_wgrad_k3_kernel<32,1>"]),
    _c("thin32_c1_flat", Geom(1, (3, 20, 24), 1, 32), "3 planes: z tiles of 2, the general wgrad <32, 1>",
       fwd=["thin_conv_kernel<32>"], wgrad=["thin_wgrad_kernel<32,1>"]),
    _c("thin32_c2", Geom(1, (8, 16, 16), 2, 32), "2 -> 32: wgrad <32, 2> on the 3x3x3 kernel",
       fwd=["thin_conv_kernel<32>"], wgrad=["thin_wgrad_k3_kernel<32,2>"]),
    _c("thin32_c2_k331", Geom(1, (8, 16, 16), 2, 32, ksize=(3, 3, 1), pad=(1, 1, 0)), "3x3x1 kernel: general wgrad",
       fwd=["thin_conv_kernel<32>"], wgrad=["thin_wgrad_kernel<32,2>"]),
    _c("thin64_c1", Geom(1, (8, 16, 16), 1, 64), "1 -> 64: thin_conv_kernel<64>, wgrad <64, 1> (3x3x3)",
       fwd=["thin_conv_kernel<64>"], dgrad=[conv_tma(32, 1, 0)], wgrad=["thin_wgrad_k3_kernel<64,1>"]),
    _c("thin64_c1_2d", Geom(1, (1, 40, 40), 1, 64, ksize=(1, 3, 3), pad=(0, 1, 1)), "2-D: general wgrad <64, 1>",
       fwd=["thin_conv_kernel<64>"], wgrad=["thin_wgrad_kernel<64,1>"]),
    _c("thin_out64_c2", Geom(1, (16, 16, 16), 64, 2), "out conv 64 -> 2: thin dgrad, wgrad <64, 2> (3x3x3)",
       fwd=[conv_tma(32, 1, 0)], dgrad=["thin_conv_kernel<64>"], wgrad=["thin_wgrad_k3_kernel<64,2>"]),
    _c("thin_out64_c2_flat", Geom(1, (2, 16, 16), 64, 2), "2 planes: general wgrad <64, 2>",
       dgrad=["thin_conv_kernel<64>"], wgrad=["thin_wgrad_kernel<64,2>"]),
    # ---- halo kernels (32 source channels at full resolution) ----
    _c("halo_ragged", Geom(2, (12, 40, 44), 32, 32), "halo fwd / dgrad / wgrad; 40 x 44 leaves ragged y and x tiles",
       fwd=["conv_halo_kernel"], dgrad=["conv_halo_kernel"], wgrad=["wgrad_halo_kernel"]),
    _c("halo_strided_odd", Geom(1, (33, 35, 37), 32, 32, **S2), "strided dgrad classes on the halo kernel, odd extents",
       fwd=[conv_tma(32, 1, 0)], dgrad=["conv_halo_kernel"], wgrad=["wgrad_tc_kernel<256>"]),
    # ---- skinny kernels (<= 32 rows, 1x1x1: the time-embedding linears) ----
    _c("skinny", Geom(4, (1, 1, 1), 64, 96, **K1), "4 rows: skinny fwd / dgrad / wgrad", extras=False,
       fwd=[f"skinny_fwd_kernel<{BF16_T},8>"], dgrad=[f"skinny_dgrad_kernel<{BF16_T},8>"],
       wgrad=[f"skinny_wgrad_kernel<{BF16_T}>"]),
    # ---- channel padding (want_pad) ----
    _c("pad_in3", Geom(1, (16, 16, 16), 3, 48), "3 input channels, 48 outputs (not thin): fwd and wgrad pad to 8",
       fwd=[_PAD, "conv_tc_kernel<64>"], dgrad=[conv_tma(32, 1, 0)],
       wgrad=[_PAD, "unpad_add_kernel", "wgrad_tc_kernel<256>"]),
]


@dataclass(frozen=True)
class GemmCase:
    """C[b] = alpha A[b] B[b] through mig_gemm_strided: A [M][K]; B [N][K] (b_mn False) or [K][N]; C [M][N]."""
    id: str
    M: int
    N: int
    K: int
    batch_outer: int
    batch_inner: int
    b_mn: bool
    c_f32: bool
    accumulate: bool
    kernels: tuple
    why: str


GEMM_CASES = [
    GemmCase("gemm64_bf16", 200, 40, 72, 1, 1, False, False, False, ("gemm_tc_kernel<64>",),
             "BN 64, M tail (200), N tail (40), K tail (72)"),
    GemmCase("gemm128_f32_mn", 130, 96, 200, 1, 1, True, True, False, ("gemm_tc_kernel<128>",),
             "BN 128 with an MN-major B and fp32 C"),
    GemmCase("gemm256_bf16_batched", 96, 320, 64, 2, 3, False, False, False, ("gemm_tc_kernel<256>",),
             "BN 256, N tail 320, 2 x 3 batches"),
    GemmCase("gemm256_f32_acc", 64, 136, 128, 1, 2, True, True, True, ("gemm_tc_kernel<256>",),
             "fp32 C accumulated into (C += alpha A B), ragged 136 columns"),
]


@dataclass(frozen=True)
class UpconvCase:
    """y = conv(nearest_upsample(x, f), w, b, padding p) through mig_upconv_fold_filter + mig_upconv_fwd."""
    id: str
    N: int
    low: tuple
    Cin: int
    Cout: int
    k: tuple
    f: tuple
    p: tuple
    kernels: tuple
    why: str


UPCONV_CASES = [
    UpconvCase("upconv_odd", 1, (5, 6, 7), 64, 64, (3, 3, 3), (2, 2, 2), (1, 1, 1), (conv_tma(64, 1, 0),),
               "eight classes of 2x2x2 taps over odd extents, rows scattered to 2j + r"),
    UpconvCase("upconv_ntail", 1, (5, 6, 7), 64, 320, (3, 3, 3), (2, 2, 2), (1, 1, 1), (conv_tma(256, 1, 0),),
               "the same with 320 outputs: BN 256 with an N tail"),
    UpconvCase("upconv_aniso", 2, (4, 6, 5), 48, 128, (3, 3, 1), (2, 2, 1), (1, 1, 0), (conv_tma(128, 1, 0),),
               "anisotropic: factor 1 and kernel 1 on the last axis, four classes"),
]
