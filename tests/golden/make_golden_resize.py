"""Generates tests/golden/resize/*.npz: what OpenCV's cv2.resize(img, (W, H)) (INTER_LINEAR, uint8, the host resize of
the reference's infer.py:17) returns for seeded images (tests/resize_ref.py: cases, synth_image). Each file holds the
seed, the sizes, the sha256 of the output and a strided sample of it, so it stays a few KB; the tests regenerate the
input from the seed. Needs OpenCV. Re-run: python tests/golden/make_golden_resize.py"""
import hashlib
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.resize_ref import cases, synth_image  # noqa: E402


def main():
    out_dir = os.path.join(ROOT, "tests", "golden", "resize")
    os.makedirs(out_dir, exist_ok=True)
    for name, h0, w0, H, W, kind, seed in cases():
        out = cv2.resize(synth_image(h0, w0, kind, seed), (W, H))
        assert out.shape == (H, W, 3) and out.dtype == np.uint8
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), seed=seed, h0=h0, w0=w0, H=H, W=W, kind=kind,
                            sha256=hashlib.sha256(out.tobytes()).hexdigest(), sample=out[::37, ::41],
                            opencv=cv2.__version__)
        print(name, hashlib.sha256(out.tobytes()).hexdigest()[:16])


if __name__ == "__main__":
    main()
