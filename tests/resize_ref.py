"""Numpy restatement of cv2.resize(img, (W, H)) with the default INTER_LINEAR on uint8 HWC images (the host resize of the
reference's infer.py:17), bit-exact, so the device kernel (csrc/postproc.cuh, resize_linear_kernel) can be checked on a
machine without OpenCV. Pinned against cv2.resize itself by tests/golden/resize/*.npz (make_golden_resize.py).

OpenCV's arithmetic, restated:
  * per axis f = float((d + 0.5) * (1 / (dst / src)) - 0.5) (double, rounded to float), s = floor(f), f -= s,
    coefficients rint((1 - f) * 2048) and rint(f * 2048) (half to even, each on its own);
  * x borders: s < 0 -> (s, f) = (0, 0); s >= W0 - 1 -> (W0 - 1, 0). y borders: f is kept, only the rows s and s + 1
    are clamped into [0, H0 - 1] when read;
  * fixed point: S = p[sx] * a0 + p[sx + 1] * a1 per row, then
    dst = (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
OpenCV switches an exact 2x downscale in both axes to its INTER_AREA fast path, (a + b + c + d + 2) >> 2 over each 2x2
block. The linear path computes the same there (every coefficient is 1024, so each vertical term is exactly a + b), so
it needs no case of its own; tests/test_infer_batch_cpu.py checks the identity.
"""
from __future__ import annotations

import numpy as np


def linear_coeffs(dst: int, src: int):
    """Per output index: source index s (unclamped), coefficients (a0, a1) of s and s + 1 (int64)."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    a0 = np.rint((np.float32(1) - f) * np.float32(2048)).astype(np.int64)
    a1 = np.rint(f * np.float32(2048)).astype(np.int64)
    return s.astype(np.int64), a0, a1


def resize_linear_u8(img: np.ndarray, H: int, W: int) -> np.ndarray:
    """cv2.resize(img, (W, H)) for a uint8 [H0, W0, C] image (INTER_LINEAR) -> uint8 [H, W, C]."""
    img = np.asarray(img)
    assert img.dtype == np.uint8 and img.ndim == 3
    H0, W0 = img.shape[:2]
    sx, a0, a1 = linear_coeffs(W, W0)
    edge = (sx < 0) | (sx >= W0 - 1)
    sx = np.clip(sx, 0, W0 - 1)
    a0 = np.where(edge, 2048, a0)[None, :, None]
    a1 = np.where(edge, 0, a1)[None, :, None]
    sx1 = np.minimum(sx + 1, W0 - 1)
    sy, b0, b1 = linear_coeffs(H, H0)

    def row_sums(rows):   # horizontal pass over the source rows one output row reads
        r = img[rows]
        return r[:, sx].astype(np.int64) * a0 + r[:, sx1].astype(np.int64) * a1

    S0 = row_sums(np.clip(sy, 0, H0 - 1))
    S1 = row_sums(np.clip(sy + 1, 0, H0 - 1))
    out = (((b0[:, None, None] * (S0 >> 4)) >> 16) + ((b1[:, None, None] * (S1 >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


# ---- inputs of the fixtures in tests/golden/resize/ (make_golden_resize.py): regenerated from the seed by the tests
SOURCES = [(576, 768), (1080, 1920), (300, 401), (777, 518), (100, 80), (1036, 1036), (259, 259), (518, 518), (37, 1000),
           (2000, 3000), (517, 519), (1037, 1035), (1036, 2072), (13, 7)]
TARGETS = [(518, 518), (518, 686)]


def cases():
    """(name, h0, w0, H, W, kind, seed) of every fixture: each source size to each target, random and smooth images,
    plus 1036x1372 -> 518x686 (2x down in both axes, not square)."""
    out = []
    for i, (h0, w0) in enumerate(SOURCES + [(1036, 1372)]):
        for H, W in (TARGETS if (h0, w0) != (1036, 1372) else [(518, 686)]):
            for kind in ("rand", "grad"):
                seed = 1000 + 10 * i + (kind == "grad")
                out.append((f"{h0}x{w0}_to_{H}x{W}_{kind}", h0, w0, H, W, kind, seed))
    return out


def synth_image(h0: int, w0: int, kind: str, seed: int) -> np.ndarray:
    """uint8 [h0, w0, 3]: uniform noise ('rand') or smooth triangle-wave colour ramps with seeded slopes and phases
    ('grad'; integer arithmetic only, so it regenerates identically everywhere)."""
    rng = np.random.default_rng(seed)
    if kind == "rand":
        return rng.integers(0, 256, size=(h0, w0, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:h0, 0:w0].astype(np.int64)
    ky, kx, ph = rng.integers(200, 900, 3), rng.integers(200, 900, 3), rng.integers(0, 512, 3)
    v = [(yy * ky[c] // h0 + xx * kx[c] // w0 + ph[c]) % 512 for c in range(3)]
    return np.stack([np.where(t < 256, t, 511 - t) for t in v], -1).astype(np.uint8)
