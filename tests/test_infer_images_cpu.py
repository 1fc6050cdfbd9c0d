"""Pins tests/cubic_ref.py, the numpy restatement of DepthAnythingV2.image2tensor (cvtColor / 255.0, cv2's float64
INTER_CUBIC, ImageNet normalise; done on the device by DepthAnythingV2.infer_images), against the digests cv2 itself
produced (tests/golden/cubic/, make_golden_cubic.py), against cv2.resize on a sweep of sizes and against image2tensor
itself where OpenCV imports. Four plausible restatement bugs must each fail a fixture. Also the host side of
infer_images that needs no GPU: how images are grouped and chunked, and which inputs are refused."""
import glob
import hashlib
import os

import numpy as np
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from tests import cubic_ref as C

CUBIC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cubic")
FIXTURES = sorted(glob.glob(os.path.join(CUBIC, "*.npz")))


def load_case(path):
    """(BGR uint8 image, input_size, H, W, sha256 of the float64 resize, sha256 of the fp32 tensor, tensor sample)."""
    z = np.load(path)
    img = C.synth_image(int(z["h0"]), int(z["w0"]), str(z["kind"]), int(z["seed"]))
    return (img, int(z["size"]), int(z["H"]), int(z["W"]), str(z["sha256_resize"]), str(z["sha256_tensor"]),
            z["sample"])


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_fixtures_cover_the_cases():
    names = {os.path.basename(p)[:-4] for p in FIXTURES}
    assert names == {c[0] for c in C.cases()} and len(names) == 44


@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: os.path.basename(p)[:-4])
def test_cubic_ref_reproduces_cv2_digests(path):
    img, size, H, W, sha_resize, sha_tensor, sample = load_case(path)
    assert (H, W) == pkg.DepthAnythingV2._input_size(img.shape[0], img.shape[1], size)
    rgb = C.resize_cubic_rgb(img, H, W)
    x = C.normalize_chw(rgb)
    assert digest(rgb) == sha_resize
    assert x.shape == (3, H, W) and np.array_equal(C.sample(x), sample) and digest(x) == sha_tensor


def test_identity_size_is_a_copy():
    """518x686 at input_size 518 keeps its size: every coefficient is (0, 1, 0, 0), so the resize returns u / 255."""
    img = C.synth_image(518, 686, "rand", 5)
    assert C.input_size(518, 686, 518) == (518, 686)
    assert np.array_equal(C.resize_cubic_rgb(img, 518, 686), img[..., ::-1] / 255.0)


def test_cubic_ref_matches_cv2_sweep():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(78)
    for _ in range(40):
        h0, w0 = (int(v) for v in rng.integers(2, 1500, 2))
        H, W = (int(v) for v in rng.integers(14, 900, 2))
        img = rng.integers(0, 256, size=(h0, w0, 3), dtype=np.uint8)
        ref = cv2.resize(cv2.cvtColor(img, cv2.COLOR_BGR2RGB) / 255.0, (W, H), interpolation=cv2.INTER_CUBIC)
        assert digest(C.resize_cubic_rgb(img, H, W)) == digest(ref), (h0, w0, H, W)


def test_cubic_ref_equals_image2tensor():
    """Against the method itself, on the CPU: a ViT-S DepthAnythingV2 needs no library to run its host transform."""
    pytest.importorskip("cv2")
    model = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=[48, 96, 192, 384])
    for i, (h0, w0) in enumerate([(576, 768), (13, 7), (300, 401), (1080, 1920)]):
        img = C.synth_image(h0, w0, "rand" if i % 2 else "grad", 300 + i)
        for size in (518, 98, 126):
            t, hw = model.image2tensor(img, size)
            assert hw == (h0, w0) and t.dtype == torch.float32
            assert digest(t[0].numpy()) == digest(C.image2tensor(img, size)), (h0, w0, size)


def _tensor_with_bug(img, H, W, bug):
    """cubic_ref.image2tensor at (H, W) with one deliberate deviation from OpenCV's arithmetic."""
    x = img[..., ::-1] / 255.0
    dt = np.float32 if bug == "fp32_accum" else np.float64
    x = x.astype(dt)

    def axis(dst, src):
        s, c = C.cubic_coeffs(dst, src, np.float64 if bug == "double_coeffs" else np.float32)
        idx = s[:, None] + np.arange(4)
        if bug == "reflect101":
            idx = np.abs(idx)
            idx = np.where(idx >= src, 2 * src - 2 - idx, idx)
        return np.clip(idx, 0, src - 1), c.astype(dt)

    cols, cx = axis(W, img.shape[1])
    rows, cy = axis(H, img.shape[0])
    h = x[:, cols[:, 0]] * cx[None, :, 0, None]
    for k in range(1, 4):
        h = h + x[:, cols[:, k]] * cx[None, :, k, None]
    t = [h[rows[:, k]] * cy[:, k, None, None] for k in range(4)]
    v = (t[0] + t[1]) + (t[2] + t[3]) if bug == "paired_vertical" else ((t[0] + t[1]) + t[2]) + t[3]
    return C.normalize_chw(v.astype(np.float64))


def test_bug_free_variant_reproduces_fixtures():
    """The harness of the simulated bugs, with no bug, gives the fixtures' bits (so a failure below is the bug's)."""
    for path in FIXTURES[:6]:
        img, size, H, W, _, sha_tensor, _ = load_case(path)
        assert digest(_tensor_with_bug(img, H, W, None)) == sha_tensor


@pytest.mark.parametrize("bug", ["double_coeffs", "reflect101", "paired_vertical", "fp32_accum"])
def test_fixtures_catch_simulated_bugs(bug):
    failed = []
    for path in FIXTURES:
        img, size, H, W, _, sha_tensor, _ = load_case(path)
        if H * W > 1_000_000 or img.size > 4_000_000:
            continue   # the smaller cases are enough to tell, and keep this quick
        if digest(_tensor_with_bug(img, H, W, bug)) != sha_tensor:
            failed.append(os.path.basename(path))
    assert failed, f"no fixture catches {bug}"


# ---- host side of infer_images
def test_chunks_group_by_input_size_in_order_of_first_appearance():
    shapes = [(1080, 1920), (576, 768), (1080, 1920), (13, 7), (720, 1280), (576, 768), (1080, 1920)]
    size = pkg.DepthAnythingV2._input_size
    chunks = pkg.DepthAnythingV2._chunks(shapes, 518, 2)
    assert size(1080, 1920) == size(720, 1280)   # same aspect ratio, same network input: one group
    assert [c[2] for c in chunks] == [[0, 2], [4, 6], [1, 5], [3]]
    for H, W, idx in chunks:
        assert all(size(*shapes[i], 518) == (H, W) for i in idx)
    assert pkg.DepthAnythingV2._chunks(shapes, 518, 32) == [(*size(1080, 1920), [0, 2, 4, 6]),
                                                            (*size(576, 768), [1, 5]), (*size(13, 7), [3])]
    many = pkg.DepthAnythingV2._chunks([(100, 100)] * 33, 98, 32)
    assert [len(c[2]) for c in many] == [32, 1] and many[0][2] + many[1][2] == list(range(33))


def test_infer_images_refuses_other_inputs_before_any_upload():
    model = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=[48, 96, 192, 384]).eval()
    good = np.zeros((20, 30, 3), np.uint8)
    for bad in (np.zeros((20, 30, 3), np.float32), np.zeros((20, 30), np.uint8), np.zeros((20, 30, 4), np.uint8),
                np.zeros((0, 30, 3), np.uint8)):
        with pytest.raises(ValueError):
            model.infer_images([good, bad])     # a CPU model would raise RuntimeError once it got past the checks
    with pytest.raises(ValueError):
        model.infer_images([good], max_batch=0)
    with pytest.raises(RuntimeError, match="CUDA"):
        model.infer_images([good])
