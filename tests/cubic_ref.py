"""Numpy restatement of DepthAnythingV2.image2tensor (depth_anything_v2_raw/dpt.py:186-222): cvtColor(BGR -> RGB) / 255.0,
cv2.resize(..., INTER_CUBIC) of that float64 image, ImageNet (x - mean) / std in float64, astype(float32), bit-exact, so
the device kernel (csrc/postproc.cuh, resize_cubic_normalize_kernel) can be checked on a machine without OpenCV. Pinned
against cv2.resize itself by tests/golden/cubic/*.npz (make_golden_cubic.py).

OpenCV's float64 INTER_CUBIC arithmetic, restated:
  * per axis f = float((d + 0.5) * (1 / (dst / src)) - 0.5) (double, rounded to float), s = floor(f), f -= s in float;
  * four coefficients in float, A = -0.75, each operation rounded on its own:
    c0 = ((A(f+1) - 5A)(f+1) + 8A)(f+1) - 4A, c1 = ((A+2)f - (A+3))f f + 1, c2 = the same at 1 - f, c3 = 1 - c0 - c1 - c2;
  * taps s - 1 .. s + 2, clamped into the image along both axes (replicated border, not reflect-101);
  * horizontal pass ((p0 c0 + p1 c1) + p2 c2) + p3 c3 in double with the float coefficients widened, then the same
    left-to-right sum of the four row values with the y coefficients.
"""
from __future__ import annotations

import numpy as np

from tests.resize_ref import synth_image  # noqa: F401  (the fixtures' inputs)

MEAN = np.array([0.485, 0.456, 0.406])
STD = np.array([0.229, 0.224, 0.225])


def input_size(h: int, w: int, target: int = 518, multiple: int = 14):
    """DepthAnythingV2._input_size: Resize(keep_aspect_ratio, lower_bound, ensure_multiple_of=14)."""
    from amodal_depth_anything_b200 import DepthAnythingV2
    return DepthAnythingV2._input_size(h, w, target, multiple)


def cubic_coeffs(dst: int, src: int, dtype=np.float32):
    """Per output index: first source tap s - 1 (unclamped, int64) and the four coefficients [dst, 4] in `dtype` (OpenCV:
    float32)."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(dtype)
    A, one = dtype(-0.75), dtype(1)
    f1, g = f + one, one - f
    c0 = ((A * f1 - dtype(5) * A) * f1 + dtype(8) * A) * f1 - dtype(4) * A
    c1 = ((A + dtype(2)) * f - (A + dtype(3))) * f * f + one
    c2 = ((A + dtype(2)) * g - (A + dtype(3))) * g * g + one
    c3 = one - c0 - c1 - c2
    return s.astype(np.int64) - 1, np.stack([c0, c1, c2, c3], -1)


def taps(dst: int, src: int):
    """(source indices [dst, 4] clamped into [0, src - 1], float64 coefficients [dst, 4])."""
    s, c = cubic_coeffs(dst, src)
    return np.clip(s[:, None] + np.arange(4), 0, src - 1), c.astype(np.float64)


def resize_cubic_rgb(img: np.ndarray, H: int, W: int) -> np.ndarray:
    """cv2.resize(cv2.cvtColor(img, BGR2RGB) / 255.0, (W, H), interpolation=INTER_CUBIC) for a uint8 [h0, w0, 3] BGR image
    -> float64 [H, W, 3]."""
    img = np.asarray(img)
    assert img.dtype == np.uint8 and img.ndim == 3 and img.shape[2] == 3
    x = img[..., ::-1] / 255.0
    cols, cx = taps(W, img.shape[1])
    rows, cy = taps(H, img.shape[0])
    h = x[:, cols[:, 0]] * cx[None, :, 0, None]
    for k in range(1, 4):
        h = h + x[:, cols[:, k]] * cx[None, :, k, None]
    v = h[rows[:, 0]] * cy[:, 0, None, None]
    for k in range(1, 4):
        v = v + h[rows[:, k]] * cy[:, k, None, None]
    return v


def normalize_chw(rgb64: np.ndarray) -> np.ndarray:
    """image2tensor's tail: (x - mean) / std in float64, HWC -> CHW, astype(float32)."""
    return np.ascontiguousarray(np.transpose((rgb64 - MEAN) / STD, (2, 0, 1))).astype(np.float32)


def image2tensor(img: np.ndarray, size: int = 518) -> np.ndarray:
    """DepthAnythingV2.image2tensor(img, size)[0][0] as numpy: fp32 [3, H, W]."""
    H, W = input_size(img.shape[0], img.shape[1], size)
    return normalize_chw(resize_cubic_rgb(img, H, W))


def sample(x: np.ndarray) -> np.ndarray:
    """The strided sample of a [3, H, W] tensor a fixture keeps: about 12 x 16 points per channel."""
    return x[:, ::max(x.shape[1] // 12, 1), ::max(x.shape[2] // 16, 1)]


# ---- inputs of the fixtures in tests/golden/cubic/ (make_golden_cubic.py): regenerated from the seed by the tests
SOURCES = [(1080, 1920), (1920, 1080), (576, 768), (768, 576), (13, 7), (100, 80), (300, 401), (777, 518), (2000, 3000),
           (37, 1000), (518, 686)]
INPUT_SIZES = [518, 98]


def cases():
    """(name, h0, w0, input_size, kind, seed) of every fixture: each source at each input_size, random and smooth images.
    518x686 at input_size 518 is an identity resize."""
    out = []
    for i, (h0, w0) in enumerate(SOURCES):
        for size in INPUT_SIZES:
            for kind in ("rand", "grad"):
                seed = 2000 + 10 * i + (kind == "grad")
                out.append((f"{h0}x{w0}_at_{size}_{kind}", h0, w0, size, kind, seed))
    return out
