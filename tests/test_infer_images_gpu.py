"""DepthAnythingV2.infer_images and the two kernels behind it (include/amodal_b200.h) on a B200: the cubic resize +
normalise against the digests of cv2 itself (tests/golden/cubic/), the restore to each image's size against an fp64
reference, and the whole call against the single-image path: image2tensor -> forward -> the fp64 restore, and
infer_image itself where OpenCV imports."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import amodal_depth_anything_b200 as pkg
from amodal_depth_anything_b200 import ops
from oracle import synth
from tests import cubic_ref as C
from tests.test_infer_batch_gpu import GUARD, guard_intact, guarded, pack, same_bits
from tests.test_infer_images_cpu import FIXTURES, digest, load_case
from tools.gpu_check import up_coords

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -24


def _has_cv2():
    try:
        import cv2  # noqa: F401
        return True
    except ImportError:
        return False


def pack_guarded(arrays, fill=0xA5):
    """pack() with the packed buffer inside GUARD bytes of `fill` on each side (uint8 has no NaN to guard with)."""
    src, desc = pack(arrays)
    flat = torch.full((src.numel() + 2 * GUARD,), fill, dtype=torch.uint8, device="cuda")
    flat[GUARD:GUARD + src.numel()] = src
    return flat[GUARD:GUARD + src.numel()], desc


# ---- the resize: cv2's own digests, the fixtures of each target size in one batch and each image alone
def test_resize_cubic_matches_cv2_digests():
    groups = {}
    for p in FIXTURES:
        img, size, H, W, _, sha, sample = load_case(p)
        groups.setdefault((H, W), []).append((img, sha, sample, os.path.basename(p)))
    assert sum(len(v) for v in groups.values()) == len(FIXTURES) == 44
    for (H, W), items in groups.items():
        src, desc = pack_guarded([it[0] for it in items])
        flat, out = guarded((len(items), 3, H, W))
        ops.resize_cubic_normalize_batch(src, desc, H, W, out=out)
        assert guard_intact(flat)
        for b, (img, sha, sample, name) in enumerate(items):
            got = out[b].cpu().numpy()
            assert np.array_equal(C.sample(got), sample) and digest(got) == sha, name
            s1, d1 = pack_guarded([img])
            f1, o1 = guarded((1, 3, H, W))
            ops.resize_cubic_normalize_batch(s1, d1, H, W, out=o1)
            assert guard_intact(f1) and same_bits(o1[0], out[b]), name


def test_resize_cubic_equals_image2tensor():
    if not _has_cv2():
        pytest.skip("OpenCV is not installed")
    model = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=[48, 96, 192, 384])   # host transform only
    for i, (h0, w0) in enumerate([(1080, 1920), (13, 7), (777, 518), (300, 401)]):
        img = C.synth_image(h0, w0, "rand", 400 + i)
        for size in (518, 98):
            ref, _ = model.image2tensor(img, size)
            src, desc = pack([img])
            out = ops.resize_cubic_normalize_batch(src, desc, *ref.shape[-2:])
            assert same_bits(out.cpu(), ref), (h0, w0, size)


# ---- the restore: fp64 reference of the same fp32 coordinates, and the bound 4 * 2^-24 * (the blend of |values|)
def restore_matrix(n_in, n_out):
    """[n_out, n_in] fp64 weights with the kernel's fp32 lambdas: (fp32(1 - l), l) at (i0, i1)."""
    i0, i1, lam = up_coords(n_in, n_out)
    l1 = lam.astype(np.float32)
    l0 = (np.float32(1) - l1).astype(np.float64)
    A = np.zeros((n_out, n_in))
    np.add.at(A, (np.arange(n_out), i0), l0)
    np.add.at(A, (np.arange(n_out), i1), l1.astype(np.float64))
    return torch.from_numpy(A).cuda()


def restore_ref(d, h, w):
    """(fp64 reference, bound) of one [H, W] fp32 map restored to (h, w)."""
    Ah, Aw = restore_matrix(d.shape[0], h), restore_matrix(d.shape[1], w)
    dd = d.double()
    return Ah @ dd @ Aw.T, 4 * EPS * (Ah @ dd.abs() @ Aw.T)


def restore_into(depth, sizes):
    """ops.upsample_restore_batch into a NaN-filled packed buffer -> (buffer, list of [h, w] views)."""
    rows, end = ops.pack_layout([(h, w, 4) for h, w in sizes])
    buf = torch.full(((end + 3) // 4 + GUARD,), float("nan"), device="cuda")
    desc = torch.tensor(rows, dtype=torch.int64, device="cuda")
    ops.upsample_restore_batch(depth, desc, buf)
    return buf, [buf[o // 4:o // 4 + h * w].view(h, w) for o, h, w in rows]


RESTORE_SIZES = [(1080, 1920), (1, 700), (500, 1), (1, 1), (98, 168), (37, 1000), (2000, 3000), (97, 167), (2, 2)]


@pytest.mark.parametrize("H,W", [(98, 168), (518, 924), (2, 2)])
def test_restore_meets_fp64_bound(H, W):
    g = torch.Generator().manual_seed(H + W)
    B = len(RESTORE_SIZES) + 1
    flat, depth = guarded((B, H, W))
    depth.copy_((torch.rand(B, H, W, generator=g) * 10 - 3).cuda())
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    depth[0] = (yy * 0.37 + xx * 1.3 + 2.0).cuda()                        # a ramp
    depth[1] = depth[1] * 1e-3 + 500                                        # narrow range far from 0
    sizes = [(H, W)] + RESTORE_SIZES                                        # map 0 at its own size: identity
    buf, outs = restore_into(depth, sizes)
    assert guard_intact(flat)
    n_out = sum(h * w for h, w in sizes)
    assert int(torch.isnan(buf).sum()) == buf.numel() - n_out               # nothing written between or after images
    worst = {}
    for b, ((h, w), o) in enumerate(zip(sizes, outs)):
        ref, bound = restore_ref(depth[b], h, w)
        err = (o.double() - ref).abs()
        assert not torch.isnan(o).any() and bool((err <= bound).all()), (b, h, w, float((err - bound).max()))
        _, alone = restore_into(depth[b:b + 1].contiguous(), [(h, w)])
        assert same_bits(alone[0], o), (b, h, w)
        aten = F.interpolate(depth[b][None, None], (h, w), mode="bilinear", align_corners=True)[0, 0]
        worst[(h, w)] = float((aten - o).abs().max())
    assert same_bits(outs[0], depth[0])
    print(f"restore {H}x{W}: max |kernel - F.interpolate| per output size: {worst}")


# ---- the whole call: ViT-S at a small input size, images of several size groups interleaved
C_RAW = [48, 96, 192, 384]
E2E_SHAPES = [(1080, 1920), (576, 768), (13, 7), (720, 1280), (300, 401), (768, 576), (576, 768), (1080, 1920), (40, 41)]
E2E_SIZE = 98


@pytest.fixture(scope="module")
def vits_raw():
    model = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=C_RAW)
    model.load_state_dict(synth.make_state_dict_raw("vits", 64, C_RAW, 52), strict=True)
    return model.cuda().eval()


def e2e_images():
    return [C.synth_image(h, w, "rand" if i % 3 else "grad", 500 + i) for i, (h, w) in enumerate(E2E_SHAPES)]


def test_infer_images_matches_single_image_path(vits_raw):
    imgs = e2e_images()
    assert len({pkg.DepthAnythingV2._input_size(h, w, E2E_SIZE) for h, w in E2E_SHAPES}) >= 4
    outs = vits_raw.infer_images(imgs, E2E_SIZE)
    cv2_ok = _has_cv2()
    for i, img in enumerate(imgs):
        h, w = img.shape[:2]
        assert outs[i].shape == (h, w) and outs[i].dtype == torch.float32 and outs[i].is_cuda
        x = torch.from_numpy(C.image2tensor(img, E2E_SIZE))[None].cuda()     # image2tensor, bit-exact
        d = vits_raw(x)[0]
        ref, bound = restore_ref(d, h, w)
        err = (outs[i].double() - ref).abs()
        assert bool((err <= bound).all()), E2E_SHAPES[i]
        _, one = restore_into(d[None].contiguous(), [(h, w)])
        assert same_bits(outs[i], one[0]), E2E_SHAPES[i]                   # the forward is batch-invariant
        if cv2_ok:
            single = torch.from_numpy(vits_raw.infer_image(img, E2E_SIZE)).cuda().double()
            assert bool(((single - ref).abs() <= bound).all()), E2E_SHAPES[i]


def test_infer_images_bit_equal_across_batches_and_orders(vits_raw):
    imgs = e2e_images()
    ref = [o.cpu() for o in vits_raw.infer_images(imgs, E2E_SIZE)]
    for mb in (1, 5, 32):
        got = vits_raw.infer_images(imgs, E2E_SIZE, max_batch=mb)
        assert all(same_bits(g.cpu(), r) for g, r in zip(got, ref)), mb
    perm = [8, 3, 0, 6, 1, 7, 2, 5, 4]
    got = vits_raw.infer_images([imgs[i] for i in perm], E2E_SIZE, max_batch=3)
    assert all(same_bits(g.cpu(), ref[i]) for g, i in zip(got, perm))


def test_infer_images_chunks_33(vits_raw):
    imgs = e2e_images()
    many = [imgs[(i * 4) % len(imgs)] for i in range(33)]
    one = [o.cpu() for o in vits_raw.infer_images(many, E2E_SIZE, max_batch=1)]
    got = vits_raw.infer_images(many, E2E_SIZE, max_batch=32)
    assert len(got) == 33 and all(same_bits(g.cpu(), r) for g, r in zip(got, one))


def test_infer_images_on_side_stream(vits_raw):
    imgs = e2e_images()
    ref = [o.cpu() for o in vits_raw.infer_images(imgs, E2E_SIZE)]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = [o.clone() for o in vits_raw.infer_images(imgs, E2E_SIZE)]
    s.synchronize()
    assert all(same_bits(g.cpu(), r) for g, r in zip(got, ref))


# ---- the configuration the benchmark times: infer.py's un-guided ViT-G head sizes at input_size 518
def test_infer_images_vitg_518():
    cfg = pkg.MODEL_CONFIGS["vitg"]
    torch.manual_seed(0)
    model = pkg.DepthAnythingV2(encoder="vitg", features=cfg["features"], out_channels=cfg["out_channels"])
    with torch.no_grad():
        getattr(model.depth_head.scratch.output_conv2, "2").bias.fill_(1.0)   # keep a random head off the ReLU floor
    model = model.cuda().eval()
    imgs = [C.synth_image(1080, 1920, "rand", 600), C.synth_image(720, 1280, "grad", 601)]
    outs = model.infer_images(imgs, 518)
    for img, o in zip(imgs, outs):
        x = torch.from_numpy(C.image2tensor(img, 518))[None].cuda()
        assert x.shape[-2:] == (518, 924)
        ref, bound = restore_ref(model(x)[0], *img.shape[:2])
        assert bool(((o.double() - ref).abs() <= bound).all()) and float(o.max()) > 0
