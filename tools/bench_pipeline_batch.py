"""AmodalInference.batch against one-image-per-call AmodalInference.__call__ on the reference's real model pair:
un-guided ViT-G (features 384, out_channels 1536 x4, infer.py:59) + guided ViT-L, 518x518, random-init weights (as
tools/bench_pipeline.py), 32 seeded 1080x1920 images with masks -- the size of a typical photo, so every image takes the
resize of infer.py:17 (cv2.resize on the host for __call__, the device kernel for batch).

Each path drives its own copy of the two models: a model handle re-plans its workspace and drops its CUDA graph whenever
the input batch changes, so sharing one pair would time that switch instead of either path's steady state. The two paths
are alternated over --repeats rounds in one process. Prints one JSON line: device-event and wall time per image of each
path (median over rounds; the single path includes its host cv2.resize and each result's D2H, the batch path one D2H of
all results), the time of the batch path's own pre/post kernels (torch.profiler, a separate pass after the timed rounds),
whether the two paths' outputs are bit-equal, and the card's name and power limit."""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import amodal_depth_anything_b200 as pkg

PRE_POST_KERNELS = ("resize_linear_kernel", "image_nearest_kernel", "mask_nearest_kernel", "minmax_init_kernel",
                    "minmax_kernel", "normalize_kernel", "blend_seam_kernel")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        return None


def make_pipe():
    cfg = pkg.MODEL_CONFIGS["vitg"]
    torch.manual_seed(0)
    raw = pkg.DepthAnythingV2(encoder="vitg", features=cfg["features"], out_channels=cfg["out_channels"]).cuda().eval()
    am = pkg.AmodalDAv2(guide_type="mask+observation", encoder="vitl", pretrained=False).cuda().eval()
    with torch.no_grad():
        am.encoder.pretrained.patch_embed_guidance.proj.weight.normal_(std=0.02)
        # random-init head: keep the un-guided output off the ReLU floor, otherwise min == max and the reference's
        # min-max normalisation (infer.py:22) is 0/0
        getattr(raw.depth_head.scratch.output_conv2, "2").bias.fill_(1.0)
    raw.repack()
    return raw, am


def inputs(n, h, w):
    rng = np.random.default_rng(0)
    imgs, masks = [], []
    for i in range(n):
        imgs.append(rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8))
        m = np.zeros((h, w), np.uint8)
        y0, x0 = int(rng.integers(0, h // 2)), int(rng.integers(0, w // 2))
        m[y0:y0 + h // 3, x0:x0 + w // 3] = 255
        masks.append(m)
    return imgs, masks


def run_single(pipe, imgs, masks):
    outs = []
    for img, m in zip(imgs, masks):
        o = pipe(img, m)
        outs.append({k: v.cpu() for k, v in o.items()})      # the caller's read of each result, as infer.py:105 does
    return {k: torch.cat([o[k].reshape(1, *o[k].shape[-2:]) if k != "pred" else o[k] for o in outs]) for k in outs[0]}


def run_batch(pipe, imgs, masks):
    return {k: v.cpu() for k, v in pipe.batch(imgs, masks).items()}


def timed(fn, *args):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    out = fn(*args)
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=32)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (sm_100)"
    raw, am = make_pipe()
    single = pkg.AmodalInference(raw, am)
    batched = pkg.AmodalInference(copy.deepcopy(raw), copy.deepcopy(am))
    imgs, masks = inputs(a.images, a.height, a.width)
    n = len(imgs)
    for _ in range(2):                                   # warm-up: plan, then capture each path's CUDA graphs
        ref_single = run_single(single, imgs, masks)
        ref_batch = run_batch(batched, imgs, masks)
    t = {"single": [], "batch": []}
    for _ in range(a.repeats):
        out_s, dev_ms, wall_ms = timed(run_single, single, imgs, masks)
        t["single"].append((dev_ms / n, wall_ms / n))
        out_b, dev_ms, wall_ms = timed(run_batch, batched, imgs, masks)
        t["batch"].append((dev_ms / n, wall_ms / n))
    bit_equal = all(torch.equal(out_s[k].view(torch.int32), out_b[k].view(torch.int32)) for k in out_s)
    stable = all(torch.equal(ref_batch[k].view(torch.int32), out_b[k].view(torch.int32)) for k in out_b)

    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_batch(batched, imgs, masks)
        torch.cuda.synchronize()
    pre_post_us, all_us = {}, 0.0
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        all_us += us
        for kname in PRE_POST_KERNELS:
            if kname in ev.key:
                pre_post_us[kname] = pre_post_us.get(kname, 0.0) + us
    med = lambda v, i: float(np.median([x[i] for x in v]))  # noqa: E731
    print(json.dumps({
        "card": card(), "pipeline": f"vitg un-guided + vitl guided, 518x518, {n} images of {a.height}x{a.width}",
        "repeats": a.repeats,
        "single_ms_per_image_device": med(t["single"], 0), "single_ms_per_image_wall": med(t["single"], 1),
        "batch_ms_per_image_device": med(t["batch"], 0), "batch_ms_per_image_wall": med(t["batch"], 1),
        "single_rounds": t["single"], "batch_rounds": t["batch"],
        "batch_pre_post_kernels_ms": {k: v / 1e3 for k, v in pre_post_us.items()},
        "batch_pre_post_ms_total": sum(pre_post_us.values()) / 1e3,
        "batch_profiled_kernels_ms_total": all_us / 1e3,
        "outputs_bit_equal": bool(bit_equal), "batch_repeatable": bool(stable),
        "finite": bool(torch.isfinite(out_b["depth_agg"]).all()),
    }))


if __name__ == "__main__":
    main()
