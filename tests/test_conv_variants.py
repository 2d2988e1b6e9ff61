"""CPU: the restated convolution plan (conv_plan.py) against the worked examples of the sources, every explicit kernel
instantiation in csrc/ against the variant table, and every table entry against the plan it claims to reach.

A kernel variant added to csrc/ without a table entry that reaches it fails `test_every_instantiation_is_reached`
here, before the GPU tests run."""
import os
import re

import pytest

import conv_plan as cp

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "medical_image_generation_b200",
                    "csrc")

# instantiations no table entry reaches, with the reason (empty: every variant is reached at 148 SMs)
UNREACHED = {}


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return re.sub(r"//[^\n]*", "", f.read())


def _ints(args):
    vals = [a.strip() for a in args.split(",")]
    return [{"true": "1", "false": "0"}.get(v, v) for v in vals]


def instantiated_kernels() -> set:
    """The variant kernels csrc/ can launch, from the explicit template arguments of the launch helpers and the
    direct launches (the skinny kernels are named by their bf16 instantiation: the table covers the bf16 path)."""
    out = set()
    for fname in sorted(os.listdir(CSRC)):
        if not fname.endswith(".cu"):
            continue
        src = _source(fname)
        for m in re.finditer(r"\blaunch_conv_tma<([^<>]*)>", src):
            a = _ints(m.group(1))
            if all(v.isdigit() for v in a):
                out.add(cp.conv_tma(a[0], a[1], a[2] if len(a) > 2 else 0))
        for helper, kernel in (("launch_wgrad_tma", "wgrad_tma_kernel"), ("launch_conv_tc", "conv_tc_kernel"),
                               ("launch_wgrad", "wgrad_tc_kernel"), ("launch_gemm", "gemm_tc_kernel"),
                               ("thin_conv_kernel", "thin_conv_kernel")):
            for m in re.finditer(rf"\b{helper}<([^<>]*)>", src):
                a = _ints(m.group(1))
                if all(v.isdigit() for v in a):      # the SIMT launch_wgrad<T> is a dtype template: not a variant
                    out.add(f"{kernel}<{','.join(a)}>")
        for m in re.finditer(r"\blaunch_thin_wgrad<([^<>]*)>", src):
            a = _ints(m.group(1))
            if all(v.isdigit() for v in a):          # each (CD, CS) launches the 3x3x3 or the general kernel
                out.add(f"thin_wgrad_kernel<{','.join(a)}>")
                out.add(f"thin_wgrad_k3_kernel<{','.join(a)}>")
        for k in ("tma_splitk_finish8", "tma_splitk_finish", "splitk_finish_kernel", "conv_halo_kernel",
                  "wgrad_halo_kernel"):
            if re.search(rf"\b{k}<<<", src):
                out.add(k)
        for m in re.finditer(r"\b(skinny_[a-z]+_kernel)<T(?:,\s*(\d+))?>\s*<<<", src):
            out.add(f"{m.group(1)}<{cp.BF16_T}{',' + m.group(2) if m.group(2) else ''}>")
    return out


def test_instantiation_parser_sees_every_family():
    got = instantiated_kernels()
    counts = {f: sum(cp.family(k) == f for k in got) for f in
              ("conv_tma_kernel", "wgrad_tma_kernel", "conv_tc_kernel", "wgrad_tc_kernel", "gemm_tc_kernel",
               "thin_conv_kernel", "thin_wgrad_kernel", "thin_wgrad_k3_kernel", "skinny_fwd_kernel",
               "skinny_dgrad_kernel", "skinny_wgrad_kernel", "tma_splitk_finish", "tma_splitk_finish8",
               "splitk_finish_kernel", "conv_halo_kernel", "wgrad_halo_kernel")}
    assert counts == {"conv_tma_kernel": 14, "wgrad_tma_kernel": 4, "conv_tc_kernel": 4, "wgrad_tc_kernel": 3,
                      "gemm_tc_kernel": 3, "thin_conv_kernel": 2, "thin_wgrad_kernel": 4, "thin_wgrad_k3_kernel": 4,
                      "skinny_fwd_kernel": 1, "skinny_dgrad_kernel": 1, "skinny_wgrad_kernel": 1,
                      "tma_splitk_finish": 1, "tma_splitk_finish8": 1, "splitk_finish_kernel": 1,
                      "conv_halo_kernel": 1, "wgrad_halo_kernel": 1}


def _table_kernels() -> dict:
    """kernel -> ids of the table entries expected to launch it (at 148 SMs)."""
    seen = {}
    for c in cp.CASES:
        for p in c.kernels:
            w = cp.PASS_NAMES.index(p)
            for k in cp.conv_kernels(c.geom, w, c.ws_bytes(w), chan_bias=c.extras, residual=c.extras,
                                     finish_aligned=not c.bias_shift):
                seen.setdefault(k, []).append(f"{c.id}:{p}")
    for c in cp.GEMM_CASES:
        for k in cp.gemm_kernels(c.M, c.N, c.K):
            seen.setdefault(k, []).append(c.id)
    for c in cp.UPCONV_CASES:
        for k in cp.upconv_kernels(c.N, c.low, c.Cin, c.Cout, c.k, c.f, c.p):
            seen.setdefault(k, []).append(c.id)
    return seen


def test_every_instantiation_is_reached():
    seen = _table_kernels()
    missing = sorted(k for k in instantiated_kernels() if k not in seen and k not in UNREACHED)
    assert not missing, f"instantiated in csrc/ but reached by no entry of the variant table: {missing}"
    stale = sorted(k for k in UNREACHED if k in seen)
    assert not stale, f"allow-listed as unreachable but reached: {stale}"
    print("\n".join(f"{k:45s} {', '.join(v[:4])}" for k, v in sorted(seen.items())))


def test_table_kernels_are_instantiated():
    """The restatement names no kernel that csrc/ does not instantiate (the helper kernels aside)."""
    helpers = {f"pad_channels_kernel<{cp.BF16_T}>", "unpad_add_kernel"}
    unknown = sorted(set(_table_kernels()) - instantiated_kernels() - helpers)
    assert not unknown, unknown


@pytest.mark.parametrize("case", cp.CASES, ids=lambda c: c.id)
def test_table_entry_reaches_its_claimed_plan(case):
    assert case.why and case.kernels
    for p, want in case.kernels.items():
        w = cp.PASS_NAMES.index(p)
        got = cp.conv_kernels(case.geom, w, case.ws_bytes(w), chan_bias=case.extras, residual=case.extras,
                              finish_aligned=not case.bias_shift)
        assert got == want, f"{case.id} {p}: the restated plan launches {sorted(got)}, the table claims {sorted(want)}"
    for p, claims in case.plan.items():
        w = cp.PASS_NAMES.index(p)
        facts = cp.plan_facts(case.geom, w, case.ws_bytes(w))
        for key, v in claims.items():
            assert facts[key] == v, f"{case.id} {p}: {key} is {facts[key]}, the table claims {v}"
    if case.gn_groups:
        b, pl = cp.box_plan_of(case.geom, cp.FWD, case.ws_bytes(cp.FWD))
        assert cp.epilogue_stats_ok(b, pl, case.gn_groups, "always"), "the GroupNorm sums would not come from the epilogue"


@pytest.mark.parametrize("case", cp.GEMM_CASES, ids=lambda c: c.id)
def test_gemm_entry_reaches_its_claimed_tile(case):
    assert set(case.kernels) == cp.gemm_kernels(case.M, case.N, case.K) and case.why


@pytest.mark.parametrize("case", cp.UPCONV_CASES, ids=lambda c: c.id)
def test_upconv_entry_reaches_its_claimed_plan(case):
    assert cp.upconv_direct_ok(case.N, case.low, case.Cin, case.Cout)
    assert set(case.kernels) == cp.upconv_kernels(case.N, case.low, case.Cin, case.Cout, case.k, case.f, case.p)


def test_table_reaches_every_schedule_shape():
    """The schedules the issue of tile coverage is about, each reached by at least one entry."""
    facts = []
    for c in cp.CASES:
        for p in c.kernels:
            w = cp.PASS_NAMES.index(p)
            if p != "wgrad" and cp.engine(c.geom, w, c.extras, c.extras) == "tma":
                facts.append((c.id, p, cp.plan_facts(c.geom, w, c.ws_bytes(w))))
    have = lambda pred: [f"{i}:{p}" for i, p, f in facts if pred(f)]   # noqa: E731
    assert have(lambda f: f["tiles"] < cp.SMS_B200)
    assert have(lambda f: f["tiles"] == cp.SMS_B200)
    assert have(lambda f: f["tiles"] > cp.SMS_B200 and f["tiles"] % cp.SMS_B200 == 1)
    assert have(lambda f: f["last_cta_fewer"])
    assert have(lambda f: f["persistent"] and f["splits"] > 1), "persistence with split-K is reachable at 148 SMs"
    assert have(lambda f: f["n_tail"] and f["bn"] == 256)
    assert have(lambda f: f["rb"] == 128 and f["valid_rows"] < 128 and f["mt"] == 2)
    assert have(lambda f: f["short_last_split"])
    gn = {(c.id, *[(f["bn"], f["mt"]) for i, p, f in facts if i == c.id and p == "fwd"]) for c in cp.CASES if c.gn_groups}
    assert {t[1] for t in gn} == {(64, 1), (64, 2), (128, 1), (128, 2), (256, 1), (256, 2)}


# ---- the restatement against the examples worked out in the source comments ----
def test_pick_box_examples():
    assert cp.pick_box(24, 24, 24) == (True, (1, 8, 8))      # exact tiling
    assert cp.pick_box(12, 12, 12) == (True, (4, 4, 4))      # exact tiling
    # 6^3: no exact tiling; 1x8x8 and 2x4x8 tie at 56 % useful rows and the first candidate wins
    assert cp.pick_box(6, 6, 6) == (True, (1, 8, 8))
    assert cp.pick_box(6, 6, 6)[1] == (1, 8, 8) and 216 / cp._cover(6, 6, 6, (2, 4, 8)) == 216 / cp._cover(6, 6, 6, (1, 8, 8))


def test_pick_box_rows_example():
    # 6^3 forward: two 3x6x6 boxes per sample in 128-row slots (84 % useful rows instead of 56 %)
    ok, box, rb = cp.pick_box_rows(6, 6, 6)
    assert ok and box == (3, 6, 6) and rb == 128
    assert cp.make_box_geom(cp.Geom(1, (6, 6, 6), 64, 64), cp.FWD).num_boxes == 2


def test_pick_box_k_example():
    # 6^3 wgrad: 48-voxel boxes (75 % useful rows instead of 56 %); 2x4x6 and 4x2x6 tie and the first one found wins
    ok, box = cp.pick_box_k(6, 6, 6)
    assert ok and box == (2, 4, 6)
    assert cp.make_box_geom(cp.Geom(1, (6, 6, 6), 64, 64, (3, 3, 3)), cp.WGRAD).num_boxes == 6


def test_plan_box_settles_split_and_persistence():
    # the 6^3 level of the LDM U-Net (128 -> 256) splits K; the 24^3 level (64 -> 256, N = 8) runs the 256 x 256 tile
    b, pl = cp.box_plan_of(cp.Geom(2, (6, 6, 6), 128, 256), cp.FWD, cp.workspace_bytes(cp.Geom(2, (6, 6, 6), 128, 256), 0))
    assert pl.splits > 1 and pl.bn == 256
    b, pl = cp.box_plan_of(cp.Geom(8, (24, 24, 24), 64, 256), cp.FWD, 1 << 40)
    assert (pl.bn, pl.mt, pl.splits) == (256, 2, 1) and pl.tiles > cp.SMS_B200
    # fewer SMs: the same shape's plan is a function of the SM count
    assert cp.plan_box(b, 0, 132).bn == 256


def test_epilogue_stats_default_branch():
    g = cp.Geom(2, (16, 16, 16), 64, 256)
    b, pl = cp.box_plan_of(g, cp.FWD, cp.workspace_bytes(g, 0))
    assert cp.epilogue_stats_ok(b, pl, 32) == (2 * pl.mt * pl.bn <= 512)
    assert cp.epilogue_stats_ok(b, pl, 32, "always") and not cp.epilogue_stats_ok(b, pl, 32, "never")
    b, pl = cp.box_plan_of(cp.Geom(2, (6, 6, 6), 128, 256), cp.FWD, cp.workspace_bytes(cp.Geom(2, (6, 6, 6), 128, 256), 0))
    assert pl.splits > 1 and not cp.epilogue_stats_ok(b, pl, 32, "always")   # split-K: statistics pass over y


def test_residue_classes_of_an_odd_volume():
    g = cp.Geom(2, (9, 11, 16), 64, 128, stride=(2, 2, 2))
    cls = cp.residue_classes(g)
    assert len(cls) == 8
    assert sorted({a[0].ext for a, _ in cls}) == [4, 5] and sorted({a[1].ext for a, _ in cls}) == [5, 6]
    assert sum(n for _, n in cls) == 27                  # every tap lands in exactly one class
    assert sum(a[0].ext * a[1].ext * a[2].ext for a, _ in cls) == 9 * 11 * 16


def test_engine_order():
    G = cp.Geom
    assert cp.engine(G(4, (1, 1, 1), 64, 96, (1, 1, 1), pad=(0, 0, 0)), 0) == "skinny"
    assert cp.engine(G(1, (12, 20, 24), 1, 32), 0) == "thin"
    assert cp.engine(G(1, (32, 32, 32), 32, 32), 0) == "halo"
    assert cp.engine(G(1, (33, 35, 37), 32, 32, stride=(2, 2, 2)), 1) == "halo-strided"
    assert cp.engine(G(1, (8, 8, 8), 64, 64), 0) == "tma"
    assert cp.engine(G(2, (9, 11, 16), 64, 128, stride=(2, 2, 2)), 1) == "tma-strided"
    assert cp.engine(G(2, (6, 6, 6), 40, 24), 0) == "gather"
    assert cp.engine(G(1, (16, 16, 16), 3, 48), 0) == "pad"
    assert cp.engine(G(1, (8, 8, 8), 3, 48), 0) == "simt"           # 512 voxels: not worth padding


def test_normalise_profiler_names():
    for raw in ("void mig::conv_tma_kernel<256, 2, false>(CUtensorMap, CUtensorMap, mig::ConvTmaParams)",
                "mig::conv_tma_kernel<256, 2, 0>", "conv_tma_kernel<256, 2>"):
        assert cp.normalise(raw) == "conv_tma_kernel<256,2,0>"
    assert cp.normalise("void mig::conv_tma_kernel<64, 1, true>(CUtensorMap, CUtensorMap, mig::ConvTmaParams)") == \
        "conv_tma_kernel<64,1,1>"
    assert cp.normalise("void mig::skinny_fwd_kernel<__nv_bfloat16, 8>(__nv_bfloat16 const*, int)") == \
        "skinny_fwd_kernel<__nv_bfloat16,8>"
    assert cp.normalise("mig::tma_splitk_finish8(float const*, float const*)") == "tma_splitk_finish8"
