"""AmodalInference.batch and the batched pre/post-processing kernels behind it (include/amodal_b200.h, ada_*_batch) on a
B200: the uint8 bilinear resize against the digests of cv2.resize itself (tests/golden/resize/), every batched kernel
bit-equal per image to the single-image op, and the whole batched pipeline bit-equal per image to single-image calls."""
import os

import numpy as np
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from amodal_depth_anything_b200 import ops
from oracle import amodal_oracle as O
from oracle import infer_oracle as IO
from oracle import synth
from tests import resize_ref as R
from tests.test_infer_batch_cpu import FIXTURES, digest, load_case
from tests.test_infer_oracle_golden import synth_image_mask

pytestmark = pytest.mark.gpu

GUARD = 4096  # guard elements on each side of an output


def pack(arrays):
    """Host uint8 arrays -> (packed device buffer, int64 [B,3] device descriptor table)."""
    arrays = [np.ascontiguousarray(a) for a in arrays]
    rows, end = ops.pack_layout([a.shape for a in arrays])
    buf = np.zeros(end, np.uint8)
    for (o, _, _), a in zip(rows, arrays):
        buf[o:o + a.size] = a.reshape(-1)
    return torch.from_numpy(buf).cuda(), torch.tensor(rows, dtype=torch.int64, device="cuda")


def guarded(shape, dtype=torch.float32, fill=float("nan")):
    """(flat buffer filled with `fill`, contiguous view of `shape` inside it with GUARD elements on each side)."""
    n = int(np.prod(shape))
    flat = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device="cuda")
    return flat, flat[GUARD:GUARD + n].view(shape)


def guard_intact(flat):
    return bool(torch.isnan(flat[:GUARD]).all() and torch.isnan(flat[-GUARD:]).all())


def same_bits(a, b):
    """Bit equality of fp32 tensors, NaNs included."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ---- the resize: cv2's own digests, all fixtures of a target size in one batch and each image alone
def _fixtures_by_target():
    groups = {}
    for p in FIXTURES:
        img, H, W, sha, sample = load_case(p)
        groups.setdefault((H, W), []).append((img, sha, sample))
    return groups


def test_resize_batch_matches_cv2_digests():
    groups = _fixtures_by_target()
    assert sum(len(v) for v in groups.values()) == len(FIXTURES) == 58
    for (H, W), items in groups.items():
        src, desc = pack([img for img, _, _ in items])
        out = ops.resize_linear_batch(src, desc, H, W).cpu().numpy()
        for b, (img, sha, sample) in enumerate(items):
            assert np.array_equal(out[b, ::37, ::41], sample), (img.shape, H, W)
            assert digest(out[b]) == sha, (img.shape, H, W)


def test_resize_one_image_at_a_time_matches_cv2_digests():
    for p in FIXTURES:
        img, H, W, sha, _ = load_case(p)
        src, desc = pack([img])
        flat, out = guarded((1, H, W, 3), torch.uint8, 0xA5)
        ops.resize_linear_batch(src, desc, H, W, out=out)
        assert digest(out[0].cpu().numpy()) == sha, os.path.basename(p)
        assert bool((flat[:GUARD] == 0xA5).all() and (flat[-GUARD:] == 0xA5).all())


# ---- the nearest pre kernels on a mixed batch whose masks have other sizes than their images
MIXED = [((300, 401), (150, 200)), ((1080, 1920), (540, 960)), ((13, 7), (26, 14)), ((518, 518), (1036, 1036)),
         ((777, 518), (777, 518))]


def test_pre_kernels_batch_equal_single_image_ops():
    S = 518
    imgs, masks = [], []
    for i, ((h, w), (mh, mw)) in enumerate(MIXED):
        imgs.append(synth_image_mask(h, w, 60 + i)[0])
        masks.append(synth_image_mask(mh, mw, 70 + i)[1].astype(np.uint8))
    B = len(imgs)
    src_img, d_img = pack(imgs)
    src_mask, d_mask = pack(masks)
    resized = ops.resize_linear_batch(src_img, d_img, S, S)
    for b, img in enumerate(imgs):
        assert np.array_equal(resized[b].cpu().numpy(), R.resize_linear_u8(img, S, S))
    d_res = torch.tensor([(b * S * S * 3, S, S) for b in range(B)], dtype=torch.int64, device="cuda")
    fx, x = guarded((B, 3, S, S))
    fr, rgb = guarded((B, 3, S, S))
    fm, m01 = guarded((B, 1, S, S))
    fg, guide = guarded((B, 1, S, S))
    ops.image_nearest_batch(resized.view(-1), d_res, S, S, normalize=True, out=x)
    ops.image_nearest_batch(src_img, d_img, S, S, out=rgb)
    ops.mask_nearest_batch(src_mask, d_mask, S, S, mask01=m01, guide=guide)
    assert all(guard_intact(f) for f in (fx, fr, fm, fg))
    for b in range(B):
        assert same_bits(x[b:b + 1], ops.image_nearest(resized[b].contiguous(), S, S, normalize=True))
        assert same_bits(rgb[b:b + 1], ops.image_nearest(torch.from_numpy(imgs[b]).cuda(), S, S))
        m1, g1 = ops.mask_nearest(torch.from_numpy(masks[b]).cuda(), S, S)
        assert same_bits(m01[b:b + 1], m1) and same_bits(guide[b:b + 1], g1)
    assert not torch.isnan(x).any() and m01.sum() > 0


# ---- batched min-max and blend
def test_minmax_and_blend_batch_equal_single_image_ops():
    H, W = 140, 154
    g = torch.Generator().manual_seed(9)
    depth = torch.rand(5, H, W, generator=g) * 7 - 2
    depth[1] = 3.25                                        # constant map: the reference's 0/0 gives NaN everywhere
    depth[3] = depth[3] * 1e-3 + 40                        # narrow range far from 0
    depth = depth.cuda()
    base, obs = ops.minmax_normalize_batch(depth)
    for b in range(5):
        b1, o1 = ops.minmax_normalize(depth[b:b + 1])
        assert same_bits(base[b:b + 1], b1) and same_bits(obs[b:b + 1], o1)
    assert torch.isnan(base[1]).all() and not torch.isnan(base[[0, 2, 3, 4]]).any()

    raw = torch.rand(5, H, W, generator=g).cuda()
    amodal = torch.rand(5, H, W, generator=g).cuda()
    mask = torch.stack([torch.from_numpy(synth_image_mask(H, W, 90 + b)[1]).float() for b in range(5)]).cuda()
    mask[1] = 0                                            # empty mask: raw everywhere, no seam
    mask[2] = 1                                            # full mask: amodal inside; the zero-padded 3x3 sum is < 9
                                                           # on the border ring, so the reference blurs it
    mask[4, 0, :9] = 1                                     # a seam that touches the border
    out = ops.blend_seam_batch(raw, amodal, mask)
    for b in range(5):
        assert same_bits(out[b], ops.blend_seam(raw[b], amodal[b], mask[b]))
    assert same_bits(out[1], raw[1]) and same_bits(out[2, 1:-1, 1:-1], amodal[2, 1:-1, 1:-1])
    assert (out[2, 0] != amodal[2, 0]).any()
    assert (out[0] != torch.where(mask[0] > 0, amodal[0], raw[0])).sum() > 100   # the seam is exercised


# ---- the pipeline, with the synthetic ViT-S pair of test_infer_gpu.test_pipeline_matches_oracle
PIPE_SHAPES = [(576, 768), (1080, 1920), (300, 401), (518, 518), (1036, 1036), (13, 7)]
C_RAW = [48, 96, 192, 384]


@pytest.fixture(scope="module")
def vits_pipe():
    sd_raw = synth.make_state_dict_raw("vits", 64, C_RAW, 52)
    sd_am = synth.make_state_dict("vits", "mask+observation", 53)
    raw = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=C_RAW)
    raw.load_state_dict(sd_raw, strict=True)
    am = pkg.AmodalDAv2(guide_type="mask+observation", encoder="vits", pretrained=False)
    am.load_state_dict(sd_am, strict=True)
    return pkg.AmodalInference(raw.cuda().eval(), am.cuda().eval()), sd_raw, sd_am


def pipe_inputs():
    imgs, masks = [], []
    for i, (h, w) in enumerate(PIPE_SHAPES):
        img, _ = synth_image_mask(h, w, 100 + i)
        _, m = synth_image_mask(max(h // 2, 8), max(w // 3, 8), 110 + i)   # masks of another size, as infer.py allows
        imgs.append(img)
        masks.append(m.astype(np.float32) * 3 if i % 2 else m)              # any dtype, non-zero = object
    return imgs, masks


def _host(d):
    return {k: v.cpu() for k, v in d.items()}


def test_pipeline_batch_bit_equal_to_single_calls(vits_pipe):
    pipe, sd_raw, sd_am = vits_pipe
    imgs, masks = pipe_inputs()
    got = _host(pipe.batch(imgs, masks))
    S = pipe.size
    assert got["base_depth"].shape == (6, S, S) and got["pred"].shape == (6, 1, S, S) and got["depth_agg"].shape == (6, S, S)
    try:
        import cv2  # noqa: F401
        have_cv2 = True
    except ImportError:
        have_cv2 = False
    for i in range(6):
        one = _host(pipe.batch([imgs[i]], [masks[i]]))
        for k in got:
            assert same_bits(got[k][i:i + 1], one[k]), (PIPE_SHAPES[i], k)
        if have_cv2:
            ref = _host(pipe(imgs[i], masks[i]))
            assert same_bits(got["base_depth"][i], ref["base_depth"]), PIPE_SHAPES[i]
            assert same_bits(got["pred"][i:i + 1], ref["pred"]), PIPE_SHAPES[i]
            assert same_bits(got["depth_agg"][i], ref["depth_agg"]), PIPE_SHAPES[i]
    assert not torch.isnan(got["depth_agg"]).any()


def test_pipeline_batch_matches_oracle(vits_pipe):
    """Against the fp32 oracle pipeline fed with the numpy cv2 restatement; the bars of test_pipeline_matches_oracle."""
    pipe, sd_raw, sd_am = vits_pipe
    imgs, masks = pipe_inputs()
    got = _host(pipe.batch(imgs, masks))
    for i in (0, 4, 5):   # 576x768, the 2x case 1036x1036, 13x7: the oracle runs on the CPU
        ref = IO.infer_single_image(imgs[i], R.resize_linear_u8(imgs[i], 518, 518), masks[i],
                                    lambda x: O.forward_raw(sd_raw, "vits", x),
                                    lambda x, gm, ob: O.forward(sd_am, "vits", "mask+observation", x, None, gm, ob))
        e_base = (got["base_depth"][i] - ref["base_depth"]).abs().max().item()
        e_pred = ((got["pred"][i:i + 1] - ref["pred"]).abs() / ref["pred"]).max().item()
        e_agg = (got["depth_agg"][i] - ref["depth_agg"]).abs().max().item()
        print(PIPE_SHAPES[i], f"base abs {e_base:.2e}  pred rel {e_pred:.2e}  agg abs {e_agg:.2e}")
        assert e_base < 3e-2 and e_pred < 1e-2 and e_agg < 3e-2


def test_pipeline_chunks_bit_equal(vits_pipe):
    pipe = vits_pipe[0]
    imgs, masks = pipe_inputs()
    imgs33 = [imgs[i % 6] for i in range(33)]
    masks33 = [masks[(i * 5) % 6] for i in range(33)]   # other image / mask pairings than above
    chunked = _host(pipe.batch(imgs33, masks33, max_batch=32))
    single = _host(pipe.batch(imgs33, masks33, max_batch=1))
    assert chunked["pred"].shape[0] == 33
    for k in chunked:
        assert same_bits(chunked[k], single[k]), k


def test_pipeline_batch_on_side_stream(vits_pipe):
    pipe = vits_pipe[0]
    imgs, masks = pipe_inputs()
    ref = _host(pipe.batch(imgs, masks))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out = pipe.batch(imgs, masks)
        out = {k: v.clone() for k, v in out.items()}
    s.synchronize()
    for k in ref:
        assert same_bits(out[k].cpu(), ref[k]), k
