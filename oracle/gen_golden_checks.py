"""Stored expectations of the checks that compare the package and the oracle with the unmodified reference functions,
so that these checks also run where the reference sources are absent.

    python -m oracle.gen_golden_checks        -> tests/golden/reference_checks.pt

Holds the kwargs of `create_autoencoder_dict` / `create_ddpm_dict` (configuration.py:821-902) for four patch sizes,
`crop_and_pad_nd` / `get_bbox` (data_processing.py:150-225, 463-527) on seeded random boxes, the split files of
`create_split_files` (data_processing.py:34-116) for a 20-case fake task, and the constructor / zero-output quirks.
The values are recorded from the package planner, the package split files and oracle/data_oracle.py. With the
reference present, the tests that read this file assert exact equality between these restatements and the reference
on the same inputs, and between the reference and the stored values. Regenerate only in such a run: recording
after a change to the restatements would pin the change instead of the reference. The quirk outcomes are the
reference probes of SURVEY.md section 0.6."""
from __future__ import annotations

import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "reference_checks.pt")

PLANNER_PATCHES = (([96, 96, 96], 1), ([160, 160, 128], 2), ([448, 512, 512], 1), ([64, 64], 1))
BBOX_PATCH = (16, 24, 24)
SPLITTINGS = ("train-val-test", "5-fold")
QUIRKS = {"DiffusionModelUNet(spatial_dims=3, in_channels=1, out_channels=1)": "IndexError",
          "AutoencoderKL(spatial_dims=3)": "IndexError",
          "fresh U-Net output max |y|": 0.0}


def planner_ds_cfg(patch):
    """The dataset-config fields create_autoencoder_dict / create_ddpm_dict read, for a dataset whose median and
    maximum shape are `patch`."""
    return {"median_shape": patch, "max_shape": patch if len(patch) == 3 else [1] + patch}


def random_boxes():
    """Seeded inputs: 60 (image, bbox) pairs for crop_and_pad_nd, then 40 (seed, shape, force_fg, class_locations)
    for get_bbox with patch BBOX_PATCH."""
    rs = np.random.RandomState(11)
    crops = []
    for _ in range(60):
        shape = tuple(int(v) for v in rs.randint(1, 12, size=4))
        img = rs.rand(*shape).astype(np.float32)
        bbox = [[int(lo), int(lo + rs.randint(1, 14))] for lo in rs.randint(-8, 12, size=3)]
        crops.append((img, bbox))
    trials = []
    for trial in range(40):
        shape = tuple(int(v) for v in rs.randint(6, 60, size=3))
        locs = {1: [tuple(int(rs.randint(s)) for s in shape) for _ in range(3)], 2: []}
        trials.append((trial, shape, bool(trial % 2), locs))
    return crops, trials


def fake_task(root, n=20, ext=".zarr"):
    """A preprocessed task directory with `n` empty cases pat000..; returns the task path."""
    images = os.path.join(root, "Task007_Fake", "imagesTr")
    os.makedirs(images)
    for i in range(n):
        path = os.path.join(images, f"pat{i:03d}{ext}")
        if ext == ".zarr":
            os.makedirs(path)
        else:
            open(path, "wb").close()
    return os.path.join(root, "Task007_Fake")


def normalized_split(split):
    """Split-file contents with every id list sorted (the comparison ignores order within a list)."""
    if isinstance(split, dict):
        return {k: sorted(v) for k, v in split.items()}
    return [{k: sorted(v) for k, v in fold.items()} for fold in split]


def main():
    import hashlib
    from medical_image_generation_b200 import data as pkg, planner
    from oracle import data_oracle as D
    g = {"planner_dicts": {}, "crops": [], "bboxes": [], "splits": {}, "quirks": dict(QUIRKS)}
    for patch, in_ch in PLANNER_PATCHES:
        vae = planner.autoencoder_kwargs(patch, in_channels=in_ch)
        latent = planner.compute_output_size(patch, vae["downsample_parameters"])
        g["planner_dicts"][(tuple(patch), in_ch)] = {"vae": vae, "ddpm": planner.ddpm_kwargs(latent, latent_channels=8)}
    crops, trials = random_boxes()
    for img, bbox in crops:
        out = D.crop_and_pad_nd(img, bbox, 0)
        g["crops"].append({"shape": img.shape, "bbox": bbox, "out_shape": out.shape,
                           "sha256": hashlib.sha256(np.ascontiguousarray(out).tobytes()).hexdigest()})
    for trial, shape, force, locs in trials:
        np.random.seed(trial)
        g["bboxes"].append([list(map(int, v)) for v in D.get_bbox(shape, force, locs, BBOX_PATCH, [0, 0, 0])])
    saved = os.environ.get("medimgen_preprocessed")
    try:
        for splitting in SPLITTINGS:
            with tempfile.TemporaryDirectory() as d:
                fake_task(d)
                os.environ["medimgen_preprocessed"] = d
                with open(pkg.create_split_files("007", splitting, "3d")) as f:
                    g["splits"][splitting] = normalized_split(json.load(f))
    finally:
        if saved is None:
            os.environ.pop("medimgen_preprocessed", None)
        else:
            os.environ["medimgen_preprocessed"] = saved
    torch.save(g, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
