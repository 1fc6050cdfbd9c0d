"""Generates tests/golden/cubic/*.npz: what DepthAnythingV2.image2tensor's host steps (cvtColor(BGR -> RGB) / 255.0,
cv2.resize(..., INTER_CUBIC) in float64, ImageNet normalise in float64, astype(float32)) give for seeded images
(tests/cubic_ref.py: cases, synth_image) at the size DepthAnythingV2._input_size picks. Each file holds the seed, the
sizes, the sha256 of the float64 cv2.resize output and of the fp32 [3, H, W] tensor, and a strided sample of the tensor
(cubic_ref.sample), so it stays a few KB; the tests regenerate the input from the seed. Needs OpenCV. Re-run:
python tests/golden/make_golden_cubic.py"""
import hashlib
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.cubic_ref import MEAN, STD, cases, input_size, sample, synth_image  # noqa: E402


def main():
    out_dir = os.path.join(ROOT, "tests", "golden", "cubic")
    os.makedirs(out_dir, exist_ok=True)
    for name, h0, w0, size, kind, seed in cases():
        img = synth_image(h0, w0, kind, seed)
        H, W = input_size(h0, w0, size)
        rgb = cv2.resize(cv2.cvtColor(img, cv2.COLOR_BGR2RGB) / 255.0, (W, H), interpolation=cv2.INTER_CUBIC)
        assert rgb.shape == (H, W, 3) and rgb.dtype == np.float64
        x = np.ascontiguousarray(np.transpose((rgb - MEAN) / STD, (2, 0, 1))).astype(np.float32)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), seed=seed, h0=h0, w0=w0, size=size, H=H, W=W,
                            kind=kind, sha256_resize=hashlib.sha256(rgb.tobytes()).hexdigest(),
                            sha256_tensor=hashlib.sha256(x.tobytes()).hexdigest(), sample=sample(x),
                            opencv=cv2.__version__)
        print(name, H, W, hashlib.sha256(x.tobytes()).hexdigest()[:16])


if __name__ == "__main__":
    main()
