"""Shared helpers for tests that read tests/golden/*.npz (fixtures minted from the unmodified reference by
tests/golden/make_golden.py)."""
import ast
import glob
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def raw_golden_names():
    """Fixtures of the un-guided DepthAnythingV2 (tests/golden/raw/, make_golden.py:main_raw)."""
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "raw", "*.npz")))


def load_golden(name, sub=""):
    """(meta, {key: array}). A fixture may hold its float32 output as the four little-endian byte planes
    `output_planes` [4, *shape] (make_golden.py:byte_planes) instead of `output`; it is returned as `output`."""
    with np.load(os.path.join(GOLDEN_DIR, sub, name + ".npz")) as f:
        z = {k: f[k] for k in f.files}
    if "output_planes" in z:
        z["output"] = np.ascontiguousarray(np.moveaxis(z.pop("output_planes"), 0, -1)).view("<f4")[..., 0]
    meta = ast.literal_eval(str(z["meta"]))
    return meta, z


def sample(t, n=4096):
    """Must match tests/golden/make_golden.py:sample."""
    f = t.detach().float().flatten().cpu()
    step = max(f.numel() // n, 1)
    return f[::step][:n].numpy()
