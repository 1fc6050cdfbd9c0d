"""DepthAnythingV2.infer_images against a loop of infer_image on the un-guided ViT-G with infer.py's head sizes (features
384, out_channels 1536 x4, infer.py:59), random-init weights, input_size 518. Two workloads of 32 seeded images:
  * one:   32 images of 1080x1920 -- one size group, network input 518x924;
  * mixed: 8 each of 1080x1920, 1920x1080, 768x576 and 1000x1000, interleaved -- four size groups.
What is timed is what a user waits for: infer_images plus a .cpu() of every result, against infer_image per image (its
host cv2 resize, a batch-1 forward, F.interpolate and its own .cpu()). The host clock ends on a device synchronise.

Each path drives its own copy of the model: a handle re-plans its workspace whenever (B, H, W) changes, so sharing one
would add a re-plan at every switch between the paths. Every shape is warmed up first; the two paths are alternated over
--repeats rounds and the median is reported. The two new kernels' times come from a separate torch.profiler pass. Both
paths' outputs come from bit-equal network inputs through a batch-invariant forward, and each restore is within
4 * 2^-24 of the exact bilinear of the non-negative depth, so they must agree within 8 * 2^-24 * max(|a|, |b|): the JSON
reports the largest ratio to that bound. Prints one JSON line (also written to --out) with the card's name and power
limit, read in the same run."""
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

KERNELS = ("resize_cubic_normalize_kernel", "upsample_restore_kernel")
WORKLOADS = {"one": [(1080, 1920)] * 4, "mixed": [(1080, 1920), (1920, 1080), (768, 576), (1000, 1000)]}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=60)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None


def make_model():
    cfg = pkg.MODEL_CONFIGS["vitg"]
    torch.manual_seed(0)
    model = pkg.DepthAnythingV2(encoder="vitg", features=cfg["features"], out_channels=cfg["out_channels"])
    with torch.no_grad():
        getattr(model.depth_head.scratch.output_conv2, "2").bias.fill_(1.0)   # keep a random head off the ReLU floor
    return model.cuda().eval()


def images(shapes, n, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, size=(*shapes[i % len(shapes)], 3), dtype=np.uint8) for i in range(n)]


def run_batch(model, imgs):
    return [o.cpu() for o in model.infer_images(imgs, 518)]


def run_single(model, imgs):
    return [torch.from_numpy(model.infer_image(img, 518)) for img in imgs]


def timed(fn, *args):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(*args)
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def agreement(a_list, b_list):
    """(all bit-equal, largest |a - b| / (8 * 2^-24 * max(|a|, |b|)) over every pixel with a nonzero bound)."""
    worst, equal = 0.0, True
    for a, b in zip(a_list, b_list):
        a, b = a.double(), b.double()
        equal &= bool(torch.equal(a, b))
        bound = 8 * 2.0 ** -24 * torch.maximum(a.abs(), b.abs())
        diff = (a - b).abs()
        if bool(((bound == 0) & (diff > 0)).any()):
            return equal, float("inf")
        worst = max(worst, float((diff / bound.clamp_min(1e-300)).max()))
    return equal, worst


def kernel_ms(model, imgs):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model.infer_images(imgs, 518)
        torch.cuda.synchronize()
    ms = {}
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        for k in KERNELS:
            if k in ev.key:
                ms[k] = ms.get(k, 0.0) + us / 1e3
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=32)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (sm_100)"
    import cv2  # noqa: F401  (infer_image resizes on the host with OpenCV)
    batched = make_model()
    single = copy.deepcopy(batched)
    result = {"card": card(), "model": "vitg un-guided (features 384, out_channels 1536 x4), input_size 518",
              "repeats": a.repeats, "workloads": {}}
    for name, shapes in WORKLOADS.items():
        imgs = images(shapes, a.images, seed=len(result["workloads"]))
        for _ in range(2):   # warm-up: every shape of both paths is planned before anything is timed
            run_single(single, imgs)
            run_batch(batched, imgs)
        t = {"single": [], "batch": []}
        for _ in range(a.repeats):
            out_s, ms = timed(run_single, single, imgs)
            t["single"].append(ms)
            out_b, ms = timed(run_batch, batched, imgs)
            t["batch"].append(ms)
        equal, worst = agreement(out_s, out_b)
        n = len(imgs)
        result["workloads"][name] = {
            "images": f"{n} of " + ", ".join(f"{h}x{w}" for h, w in dict.fromkeys(shapes)),
            "network_inputs": sorted({"%dx%d" % pkg.DepthAnythingV2._input_size(h, w, 518) for h, w in shapes}),
            "infer_image_loop_ms_per_image": float(np.median(t["single"])) / n,
            "infer_images_ms_per_image": float(np.median(t["batch"])) / n,
            "infer_image_loop_rounds_ms": t["single"], "infer_images_rounds_ms": t["batch"],
            "speedup": float(np.median(t["single"]) / np.median(t["batch"])),
            "new_kernels_ms_per_call": kernel_ms(batched, imgs),
            "outputs_bit_equal": equal, "max_diff_over_restore_bound": worst,
            "finite": all(bool(torch.isfinite(o).all()) for o in out_b),
        }
    result["workspace_bytes"] = {"infer_images": batched.workspace_bytes(), "infer_image": single.workspace_bytes()}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
