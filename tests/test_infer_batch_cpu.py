"""Pins tests/resize_ref.py, the numpy restatement of cv2.resize's uint8 INTER_LINEAR (the host resize of the reference's
infer.py:17, done on the device by AmodalInference.batch), against the digests cv2.resize itself produced
(tests/golden/resize/, make_golden_resize.py) and, where OpenCV imports, against cv2.resize on a sweep of sizes. Two
plausible restatement bugs (the y border handled like x, float interpolation) must each fail a fixture. A third
candidate, leaving out OpenCV's INTER_AREA path for exact 2x downscales, is no bug: the linear arithmetic gives the same
bits there, which test_area_2x_path_equals_linear_path shows for every input."""
import glob
import hashlib
import os

import numpy as np
import pytest

from tests import resize_ref as R

RESIZE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resize")
FIXTURES = sorted(glob.glob(os.path.join(RESIZE, "*.npz")))


def load_case(path):
    z = np.load(path)
    img = R.synth_image(int(z["h0"]), int(z["w0"]), str(z["kind"]), int(z["seed"]))
    return img, int(z["H"]), int(z["W"]), str(z["sha256"]), z["sample"]


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_fixtures_cover_the_cases():
    names = {os.path.basename(p)[:-4] for p in FIXTURES}
    assert names == {c[0] for c in R.cases()} and len(names) == 58


@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: os.path.basename(p)[:-4])
def test_resize_ref_reproduces_cv2_digest(path):
    img, H, W, sha, sample = load_case(path)
    out = R.resize_linear_u8(img, H, W)
    assert out.shape == (H, W, 3) and np.array_equal(out[::37, ::41], sample)
    assert digest(out) == sha


def test_resize_ref_matches_cv2_sweep():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(77)
    for _ in range(200):
        h0, w0 = (int(v) for v in rng.integers(2, 2501, 2))
        H, W = (518, 518) if rng.random() < 0.5 else (int(v) for v in rng.integers(2, 1000, 2))
        img = rng.integers(0, 256, size=(h0, w0, 3), dtype=np.uint8)
        assert np.array_equal(R.resize_linear_u8(img, H, W), cv2.resize(img, (W, H))), (h0, w0, H, W)


def _resize_with_bug(img, H, W, bug):
    """resize_ref.resize_linear_u8 with one deliberate deviation from OpenCV."""
    H0, W0 = img.shape[:2]
    p = img.astype(np.int64)
    sx, a0, a1 = R.linear_coeffs(W, W0)
    edge = (sx < 0) | (sx >= W0 - 1)
    sx = np.clip(sx, 0, W0 - 1)
    a0, a1 = np.where(edge, 2048, a0), np.where(edge, 0, a1)
    sx1 = np.minimum(sx + 1, W0 - 1)
    sy, b0, b1 = R.linear_coeffs(H, H0)
    if bug == "fy_reset":
        yedge = (sy < 0) | (sy >= H0 - 1)
        sy = np.clip(sy, 0, H0 - 1)
        b0, b1 = np.where(yedge, 2048, b0), np.where(yedge, 0, b1)
    y0, y1 = np.clip(sy, 0, H0 - 1), np.clip(sy + 1, 0, H0 - 1)
    if bug == "float_interp":
        fx, fy = a1 / 2048.0, b1 / 2048.0
        rows = p[:, sx] * (1 - fx)[None, :, None] + p[:, sx1] * fx[None, :, None]
        out = rows[y0] * (1 - fy)[:, None, None] + rows[y1] * fy[:, None, None]
        return np.clip(np.rint(out), 0, 255).astype(np.uint8)
    rows = p[:, sx] * a0[None, :, None] + p[:, sx1] * a1[None, :, None]
    out = (((b0[:, None, None] * (rows[y0] >> 4)) >> 16) + ((b1[:, None, None] * (rows[y1] >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


@pytest.mark.parametrize("bug", ["fy_reset", "float_interp"])
def test_fixtures_catch_simulated_bugs(bug):
    failed = []
    for path in FIXTURES:
        img, H, W, sha, _ = load_case(path)
        if img.size > 4_000_000:
            continue   # the smaller sources are enough to tell, and keep this quick
        if digest(_resize_with_bug(img, H, W, bug)) != sha:
            failed.append(os.path.basename(path))
    assert failed, f"no fixture catches {bug}"


def test_area_2x_path_equals_linear_path():
    """OpenCV's INTER_AREA fast path for exactly 2H x 2W, (a + b + c + d + 2) >> 2, against the linear arithmetic. At 2x
    every source coordinate is 2d + 0.5: both coefficients are 1024 and no index reaches the border, so each vertical term
    (1024 * ((1024 * s) >> 4)) >> 16 is exactly the column sum s = a + b. Checked in closed form for every s and size up
    to 2500, and on the 2x fixtures (cv2's own output)."""
    s = np.arange(0, 511, dtype=np.int64)
    assert np.array_equal((1024 * ((1024 * s) >> 4)) >> 16, s)
    for n in range(1, 1251):
        src, a0, a1 = R.linear_coeffs(n, 2 * n)
        assert (a0 == 1024).all() and (a1 == 1024).all() and np.array_equal(src, 2 * np.arange(n))
    n2x = 0
    for path in FIXTURES:
        img, H, W, sha, _ = load_case(path)
        if img.shape[:2] == (2 * H, 2 * W):
            p = img.astype(np.int64)
            area = ((p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2] + 2) >> 2).astype(np.uint8)
            assert digest(area) == sha == digest(R.resize_linear_u8(img, H, W))
            n2x += 1
    assert n2x == 4   # 1036x1036 -> 518x518 and 1036x1372 -> 518x686, random and smooth
