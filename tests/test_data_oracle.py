"""CPU: pin oracle/data_oracle.py (numpy restatement of medimgen/data_processing.py's sampling / crop path) to the goldens
produced by the UNMODIFIED reference (oracle/gen_golden_data.py), to the reference live when it is present, and check the
host half of medical_image_generation_b200/data.py (same np.random consumption order => same batches and boxes)."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import data_oracle as D
from oracle import reference_loader as ref
from oracle.gen_golden_checks import BBOX_PATCH, fake_task, normalized_split, random_boxes
from oracle.gen_golden_data import DATASETS, make_case


def test_crop_and_pad_matches_reference_golden(golden):
    g = golden("data_path")
    assert len(g["crop"]) >= 8
    for case in g["crop"]:
        got = D.crop_and_pad_nd(case["image"].numpy(), case["bbox"], case["pad"])
        assert got.shape == tuple(case["out"].shape)
        assert np.array_equal(got, case["out"].numpy()), case["bbox"]
        assert np.array_equal(got, case["out_torch"].numpy()), case["bbox"]   # the reference's torch branch agrees


def test_sampler_matches_reference_golden(golden):
    for rec in golden("data_path")["sampler"]:
        np.random.seed(99)
        indices = list(range(rec["n"]))
        epochs = [D.sampler_batches_from(indices, rec["batch_size"], rec["steps"], rec["shuffle"]) for _ in range(2)]
        assert epochs == rec["epochs"], rec


@pytest.mark.parametrize("name", sorted(DATASETS))
@pytest.mark.parametrize("section", ["training", "validation"])
def test_getitem_matches_reference_golden(golden, name, section):
    rec = golden("data_path")["datasets"][name]
    want = rec[section]
    cases = [make_case(seed, shape) for seed, shape in zip(rec["seeds"], rec["shapes"])]
    patch = rec["patch"]
    patch3 = (1, *patch) if len(patch) == 2 else tuple(patch)
    assert tuple(want["initial_patch_size"]) == patch3 and want["need_to_pad"] == [0] * len(patch3)
    np.random.seed(2024)
    batches = D.sampler_batches(len(cases), rec["batch_size"], 3, shuffle=section == "training")
    assert batches == want["batches"]
    k = 0
    for batch in batches:
        for pos, idx in batch:
            image, locs = cases[idx]
            # the box alone (replayed on a copy of the RNG state), then the whole __getitem__
            state = np.random.get_state()
            force = D.oversample_last_xx_percent(pos, rec["batch_size"], rec["oversample"])
            lbs, ubs = D.get_bbox(image.shape[1:], force, locs, patch3, [0] * len(patch3), is_2d=patch3[0] == 1)
            assert (list(map(int, lbs)), list(map(int, ubs))) == tuple(list(map(int, b)) for b in want["bboxes"][k]), k
            np.random.set_state(state)
            got = D.getitem_untransformed(image, locs, pos, rec["batch_size"], patch, rec["oversample"],
                                          rec["channel_ids"])
            assert got.shape == tuple(want["shape"])
            assert hashlib.sha256(got.tobytes()).hexdigest() == want["sha256"][k], (name, section, k)
            if k < rec["batch_size"]:
                assert np.array_equal(got, want["images"][k].numpy())
            k += 1
    assert k == len(want["sha256"])


def test_soft_augmentation_params_match_reference_golden(golden):
    for patch, want in golden("data_path")["aug_params"].items():
        got = D.soft_augmentation_params(patch)
        assert tuple(got["mirror_axes"]) == tuple(want["mirror_axes"])
        init = tuple(got["initial_patch_size"])      # the dataset makes a 2-D size pseudo-3-D (data_processing.py:301-302)
        assert ((1, *init) if len(init) == 2 else init) == tuple(want["initial_patch_size"])
        assert got["scale_range"] == want["scaling_range"]
        for key in ("brightness_range", "contrast_range", "gamma_range"):
            assert got[key] == want[key]
        assert bool(got["do_dummy_2d"]) == bool(want["dummy_2d"])
        axis, lo, hi = got["rot_for_da"]
        np.random.seed(5)
        for draws in want["rot_draws"]:
            mine = [np.random.uniform(lo, hi) if a == axis else 0 for a in range(3)]
            assert mine == draws


def test_oracle_matches_live_reference_random_boxes(golden):
    """Random boxes through crop_and_pad_nd and get_bbox against the unmodified functions' results: stored in
    tests/golden/reference_checks.pt, and computed live as well when the reference is present."""
    stored = golden("reference_checks")
    crops, trials = random_boxes()
    fn = ref.data_functions() if ref.available() else None
    assert len(crops) == len(stored["crops"]) == 60 and len(trials) == len(stored["bboxes"]) == 40
    for (img, bbox), want in zip(crops, stored["crops"]):
        assert (img.shape, bbox) == (want["shape"], want["bbox"])      # the seeded inputs are the recorded ones
        got = D.crop_and_pad_nd(img, bbox, 0)
        assert got.shape == want["out_shape"], bbox
        assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == want["sha256"], bbox
        if fn is not None:
            assert np.array_equal(got, fn["crop_and_pad_nd"](img, bbox, 0)), (img.shape, bbox)
    if fn is not None:
        ds = fn["MedicalDataset"]("/nonexistent/", [], 4, "training", {"patch_size": list(BBOX_PATCH), **_OFF}, 0.5)
    for (trial, shape, force, locs), want in zip(trials, stored["bboxes"]):
        np.random.seed(trial)
        got = D.get_bbox(shape, force, locs, BBOX_PATCH, [0, 0, 0])
        assert [list(map(int, v)) for v in got] == want, (shape, force)
        if fn is not None:
            np.random.seed(trial)
            assert [list(map(int, v)) for v in ds.get_bbox(shape, force, locs)] == want, (shape, force)


def test_affine_identity_and_transform_algebra():
    """Closed-form checks of the unpinned (third-party) transform restatements."""
    rs = np.random.RandomState(3)
    x = rs.rand(2, 6, 7, 8).astype(np.float32)
    eye = D.rotation_scale_matrix((0, 0, 0), (1, 1, 1))
    assert np.allclose(D.affine_resample(x, eye), x, atol=1e-6)
    # contrast keeps the mean (before clamping) and the range; gamma with retain_stats keeps mean and std
    c = D.contrast(x, [0.9, 1.1])
    assert c[0].min() >= x[0].min() - 1e-7 and c[1].max() <= x[1].max() + 1e-7
    gm = D.gamma(x, [0.9, 1.1])
    for ch in range(2):
        assert abs(float(gm[ch].mean()) - float(x[ch].mean())) < 1e-5
        assert abs(float(torch.as_tensor(gm[ch]).std()) - float(torch.as_tensor(x[ch]).std())) < 1e-5
    assert np.array_equal(D.mirror(x, (2,)), x[:, :, :, ::-1])
    # a 90 degree rotation about the slice axis on a square patch is an exact permutation of the voxels
    sq = rs.rand(1, 3, 8, 8).astype(np.float32)
    rot = D.affine_resample(sq, D.rotation_scale_matrix((np.pi / 2, 0, 0), (1, 1, 1)))
    assert np.allclose(rot[0], np.rot90(sq[0], k=1, axes=(1, 2)), atol=1e-5) or \
        np.allclose(rot[0], np.rot90(sq[0], k=-1, axes=(1, 2)), atol=1e-5)


# ------------------------------------------------------------------ host half of the package (no GPU, no compute calls)
from medical_image_generation_b200 import data as pkg   # noqa: E402

_OFF = {"scaling": False, "rotation": False, "gaussian_noise": False, "gaussian_blur": False, "low_resolution": False,
        "brightness": False, "contrast": False, "gamma": False, "mirror": False, "dummy_2d": False}


@pytest.mark.parametrize("name", sorted(DATASETS))
@pytest.mark.parametrize("section", ["training", "validation"])
def test_package_sampler_and_boxes_match_reference_golden(golden, name, section):
    """CustomBatchSampler + PatchSampler.get_bbox of the PACKAGE replay the reference's batches and boxes bit for bit."""
    rec = golden("data_path")["datasets"][name]
    want = rec[section]
    ps = pkg.PatchSampler(rec["batch_size"], section, dict(_OFF, patch_size=list(rec["patch"])), rec["oversample"])
    assert tuple(ps.initial_patch_size) == tuple(want["initial_patch_size"])
    assert ps.need_to_pad.tolist() == want["need_to_pad"]
    cases = [make_case(seed, shape) for seed, shape in zip(rec["seeds"], rec["shapes"])]
    sampler = pkg.CustomBatchSampler(range(len(cases)), rec["batch_size"], number_of_steps=3,
                                     shuffle=section == "training")
    np.random.seed(2024)
    k = 0
    for step, batch in enumerate(sampler):
        assert batch == want["batches"][step]
        for pos, idx in batch:
            image, locs = cases[idx]
            lbs, ubs = ps.get_bbox(image.shape[1:], ps.oversampling_method(pos), locs, is_2d=ps.patch_size[0] == 1)
            assert (list(map(int, lbs)), list(map(int, ubs))) == tuple(list(map(int, b)) for b in want["bboxes"][k])
            assert ps._draw_augmentation(image.shape[0])["mat"] is None   # everything off: no RNG consumed
            k += 1


def test_package_sampler_epochs_match_reference_golden(golden):
    for rec in golden("data_path")["sampler"]:
        np.random.seed(99)
        s = pkg.CustomBatchSampler(range(rec["n"]), rec["batch_size"], rec["steps"], rec["shuffle"])
        assert [list(s), list(s)] == rec["epochs"] and len(s) == rec["steps"]


def test_package_augmentation_params_match_reference_golden(golden):
    for patch, want in golden("data_path")["aug_params"].items():
        ps = pkg.PatchSampler(2, "training", dict(_OFF, patch_size=list(patch), rotation=True, scaling=True, mirror=True,
                                                  brightness=True, contrast=True, gamma=True), 0.0)
        ta = ps.transformation_args
        assert tuple(ta["mirror_axes"]) == tuple(want["mirror_axes"]) and ta["scaling_range"] == want["scaling_range"]
        for key in ("brightness_range", "contrast_range", "gamma_range"):
            assert ta[key] == want[key]
        assert tuple(ps.initial_patch_size) == tuple(want["initial_patch_size"])
        np.random.seed(5)
        assert [[ta["rot_for_da"](None, a) for a in range(3)] for _ in range(4)] == want["rot_draws"]
    with pytest.raises(NotImplementedError):
        pkg.PatchSampler(2, "training", dict(_OFF, patch_size=[8, 8, 8], gaussian_blur=True), 0.0)


def test_package_oversampling_rule():
    ps = pkg.PatchSampler(4, "training", dict(_OFF, patch_size=[8, 8, 8]), 0.33)
    assert [ps.oversampling_method(i) for i in range(4)] == [D.oversample_last_xx_percent(i, 4, 0.33) for i in range(4)]
    assert [ps.oversampling_method(i) for i in range(4)] == [False, False, False, True]


def _write_zarr(path, array, chunks, compressor, sep="."):
    """A zarr v2 directory store written by hand (the zarr package is not installed)."""
    import json
    import math
    import os
    import zlib
    os.makedirs(path)
    meta = {"zarr_format": 2, "shape": list(array.shape), "chunks": list(chunks), "dtype": array.dtype.str,
            "compressor": compressor, "fill_value": 0, "order": "C", "filters": None}
    if sep != ".":
        meta["dimension_separator"] = sep
    with open(os.path.join(path, ".zarray"), "w") as f:
        json.dump(meta, f)
    grid = [math.ceil(s / c) for s, c in zip(array.shape, chunks)]
    for n, idx in enumerate(np.ndindex(*grid)):
        if n == 1:
            continue    # a missing chunk reads as fill_value
        block = np.zeros(chunks, dtype=array.dtype)
        sel = tuple(slice(i * c, min((i + 1) * c, s)) for i, c, s in zip(idx, chunks, array.shape))
        block[tuple(slice(0, s.stop - s.start) for s in sel)] = array[sel]
        raw = block.tobytes()
        if compressor is not None:
            raw = zlib.compress(raw, compressor.get("level", 1))
        name = os.path.join(path, sep.join(map(str, idx)))
        os.makedirs(os.path.dirname(name), exist_ok=True)
        with open(name, "wb") as f:
            f.write(raw)


@pytest.mark.parametrize("compressor,sep", [(None, "."), ({"id": "zlib", "level": 1}, "."), ({"id": "zlib", "level": 3}, "/")])
def test_zarr_v2_reader(tmp_path, compressor, sep):
    """The layout the reference's preprocessing writes (configuration.py:1404-1410: chunks (1, 1, Y, X)) with the
    codecs this image has; Blosc is refused with a clear message."""
    import json
    import os
    import pickle
    rs = np.random.RandomState(0)
    arr = rs.rand(2, 5, 7, 9).astype(np.float32)
    _write_zarr(str(tmp_path / "case.zarr" / "image"), arr, (1, 2, 7, 9), compressor, sep)
    with open(tmp_path / "case.pkl", "wb") as f:
        pickle.dump({"class_locations": {1: [(0, 1, 2)]}}, f)
    want = arr.copy()
    want[0, 2:4] = 0                      # the chunk the writer skipped
    got, props = pkg.load_case(str(tmp_path), "case")
    assert got.dtype == np.float32 and np.array_equal(got, want) and props["class_locations"][1] == [(0, 1, 2)]
    meta_path = tmp_path / "case.zarr" / "image" / ".zarray"
    meta = json.loads(meta_path.read_text())
    meta["compressor"] = {"id": "blosc", "cname": "zstd", "clevel": 5, "shuffle": 2, "blocksize": 0}
    meta_path.write_text(json.dumps(meta))
    try:
        import numcodecs  # noqa: F401
    except ImportError:
        with pytest.raises(RuntimeError, match="numcodecs"):
            pkg.load_case(str(tmp_path), "case")
    np.save(tmp_path / "other.npy", arr)
    with open(tmp_path / "other.pkl", "wb") as f:
        pickle.dump({"class_locations": {}}, f)
    assert np.array_equal(pkg.load_case(str(tmp_path), "other")[0], arr)
    with pytest.raises(FileNotFoundError):
        pkg.load_case(str(tmp_path), "missing")


def test_data_path_refuses_cpu():
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.crop_and_pad_nd(torch.zeros(1, 4, 4, 4), [[0, 2], [0, 2], [0, 2]])
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.ResidentVolumes("cpu")
    assert pkg._DESC.itemsize == 152


@pytest.mark.parametrize("splitting", ["train-val-test", "5-fold"])
def test_split_files_like_reference(golden, tmp_path, monkeypatch, splitting):
    """create_split_files / get_data_ids (data_processing.py:34-116): 70 / 10 / 20 split or 5 folds with seed 12345, file
    reused when present; identical to the unmodified reference functions' split, stored in
    tests/golden/reference_checks.pt and computed live as well when the reference is present."""
    import json
    import os
    mine_root = tmp_path / "mine"
    mine_root.mkdir()
    task = fake_task(str(mine_root))
    monkeypatch.setenv("medimgen_preprocessed", str(mine_root))
    path = pkg.create_split_files("007", splitting, "3d")
    assert os.path.dirname(path) == task
    split = json.load(open(path))
    want = golden("reference_checks")["splits"][splitting]
    assert normalized_split(split) == want
    names = sorted(f"pat{i:03d}" for i in range(20))
    if splitting == "train-val-test":
        assert os.path.basename(path) == "splits_train_val_test.json"
        assert (len(split["train"]), len(split["val"]), len(split["test"])) == (14, 2, 4)
        assert sorted(split["train"] + split["val"] + split["test"]) == names
        ids = pkg.get_data_ids(path)
    else:
        assert os.path.basename(path) == "splits_final.json" and len(split) == 5
        assert all(sorted(f["train"] + f["val"]) == names and len(f["val"]) == 4 for f in split)
        ids = pkg.get_data_ids(path, fold=2)
        assert ids["val"] == split[2]["val"]
    assert set(ids) == {"train", "val"}
    # an existing split file is reused, not regenerated
    with open(path, "w") as f:
        json.dump({"train": ["a"], "val": ["b"], "test": []} if splitting == "train-val-test" else [{"train": ["a"], "val": ["b"]}] * 5, f)
    assert pkg.create_split_files("007", splitting, "3d") == path
    assert pkg.get_data_ids(path, fold=None if splitting == "train-val-test" else 0) == {"train": ["a"], "val": ["b"]}
    with pytest.raises(ValueError):
        os.remove(path)
        pkg.create_split_files("007", "leave-one-out", "3d")
    if ref.available():
        ref_root = tmp_path / "ref"
        ref_root.mkdir()
        fake_task(str(ref_root))
        monkeypatch.setenv("medimgen_preprocessed", str(ref_root))
        fn = ref.data_functions()
        assert normalized_split(json.load(open(fn["create_split_files"]("007", splitting, "3d")))) == want
        monkeypatch.setenv("medimgen_preprocessed", str(mine_root))
        assert normalized_split(json.load(open(pkg.create_split_files("007", splitting, "3d")))) == want


def test_npz_cases_are_found_when_there_is_no_zarr(tmp_path, monkeypatch):
    mine_root = tmp_path / "npz"
    mine_root.mkdir()
    fake_task(str(mine_root), n=10, ext=".npz")
    monkeypatch.setenv("medimgen_preprocessed", str(mine_root))
    import json
    split = json.load(open(pkg.create_split_files("007", "train-val-test", "3d")))
    assert len(split["train"]) + len(split["val"]) + len(split["test"]) == 10
    assert all(not n.endswith(".npz") for n in split["train"])
