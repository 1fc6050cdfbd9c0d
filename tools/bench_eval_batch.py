"""The validation loop (discriminative_trainer.py:470-670) two ways on the guided ViT-L at 518x518 with seeded random
weights (oracle/synth.make_state_dict), over --samples seeded samples, at two ground-truth sizes: all 518x518, and mixed
sizes up to 1080x1920.

(a) the per-sample recipe of INTEGRATION.md: the model at batch 1, ops.eval_sample, ops.eval_sample_dict (one host read
    per sample), the mean on the host;
(b) AmodalEvaluator.add at batch 32, then one result().

Both paths upload each sample's ground truth from host arrays: (a) one pageable copy per map, as a loader without pinned
memory hands them over, (b) its packed pinned upload. The inputs x / guide_mask / observation are on the device for both.
The ground truths cycle through --distinct seeded sets (a 1080x1920 sample is 20 MB of host arrays). Each path drives its
own model handle (a handle re-plans its workspace when the batch changes); the paths alternate over --rounds rounds in
one process and the median ms per sample is reported. A separate torch.profiler pass times eval_batch_kernel at batch 32
(both size mixes) and ada_eval_sample on the three golden eval shapes. Prints one JSON line with the card's name and
power limit, and whether the two paths' rows are bit-equal."""
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
from amodal_depth_anything_b200 import ops
from oracle import eval_oracle as EO
from oracle import synth

MIXED = [(1080, 1920), (375, 1242), (720, 1280), (518, 518), (480, 640), (200, 333), (1080, 810), (352, 1216)]
GOLDEN_SHAPES = [(518, 518, 375, 1242), (126, 98, 200, 333), (70, 70, 518, 518)]  # h, w, H, W of tests/golden/eval
KEYS = ("depth_gt", "depth_obs", "visible_mask", "object_mask")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        return None


def targets(sizes, n, seed):
    out = []
    for i in range(n):
        H, W = sizes[i % len(sizes)]
        s = EO.synth_sample(seed + i, 14, 14, H, W)
        out.append({k: s[k].numpy() for k in KEYS})
    return out


def path_a(model, x, gm, ob, tg):
    rows, sums = [], {}
    for i in range(x.shape[0]):
        t = tg[i % len(tg)]
        pred = model(x[i:i + 1], guide_mask=gm[i:i + 1], observation=ob[i:i + 1])
        out = ops.eval_sample(pred, *[torch.from_numpy(t[k]).cuda() for k in KEYS])
        m = ops.eval_sample_dict(out)
        rows.append(out)
        for v in ("pred", "aligned"):
            for name, val in m[v].items():
                sums[(v, name)] = sums.get((v, name), 0.0) + val
    return torch.stack(rows)


def path_b(ev, x, gm, ob, tg, bs):
    ev.reset()
    rows = []
    for i in range(0, x.shape[0], bs):
        ts = [tg[j % len(tg)] for j in range(i, min(i + bs, x.shape[0]))]
        rows.append(ev.add(x[i:i + bs], *[[t[k] for t in ts] for k in KEYS], guide_mask=gm[i:i + bs],
                           observation=ob[i:i + bs]))
    ev.result()
    return torch.cat(rows)


def wall(fn, *args):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(*args)
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def kernel_us(fn, reps=10):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for e in prof.key_averages():
        if "eval_batch_kernel" in e.key:
            us += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            n += e.count
    return us / max(n, 1)


@torch.no_grad()
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=256)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=32)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (sm_100)"
    sd = synth.make_state_dict("vitl", "mask+observation", seed=0)
    model_a = pkg.AmodalDAv2(guide_type="mask+observation", encoder="vitl", pretrained=False)
    model_a.load_state_dict(sd, strict=True)
    model_a = model_a.cuda().eval()
    model_b = copy.deepcopy(model_a)
    ev = pkg.AmodalEvaluator(model_b)
    g = torch.Generator(device="cuda").manual_seed(0)
    N, S = a.samples, 518
    x = torch.rand(N, 3, S, S, device="cuda", generator=g)
    gm = (torch.rand(N, 1, S, S, device="cuda", generator=g) > 0.5).float() * 2 - 1
    ob = torch.rand(N, 1, S, S, device="cuda", generator=g) * 2 - 1
    res = {"card": card(), "model": f"vitl mask+observation, {S}x{S}, seeded random weights", "samples": N,
           "batch": a.batch, "rounds": a.rounds, "distinct_targets": a.distinct}
    for name, sizes in (("gt518", [(S, S)]), ("gt_mixed", MIXED)):
        tg = targets(sizes, a.distinct, 1000)
        path_a(model_a, x[:2], gm[:2], ob[:2], tg)                       # warm-up: plan both handles
        path_b(ev, x[:a.batch], gm[:a.batch], ob[:a.batch], tg, a.batch)
        ta, tb = [], []
        for _ in range(a.rounds):
            rows_a, ms = wall(path_a, model_a, x, gm, ob, tg)
            ta.append(ms / N)
            rows_b, ms = wall(path_b, ev, x, gm, ob, tg, a.batch)
            tb.append(ms / N)
        bit_equal = torch.equal(rows_a.view(torch.int64), rows_b.view(torch.int64))
        t32 = tg[:a.batch] if len(tg) >= a.batch else [tg[i % len(tg)] for i in range(a.batch)]
        pred32 = model_b(x[:a.batch], guide_mask=gm[:a.batch], observation=ob[:a.batch])
        buf, desc = pkg.evaluate.pack_targets([(S, S)] * a.batch, *[[t[k] for t in t32] for k in KEYS])
        d_buf, d_desc = torch.from_numpy(buf).cuda(), torch.from_numpy(desc).cuda()
        res[name] = {"sizes": sizes, "a_ms_per_sample": float(np.median(ta)), "b_ms_per_sample": float(np.median(tb)),
                     "a_rounds": ta, "b_rounds": tb, "rows_bit_equal": bool(bit_equal),
                     "eval_kernel_us_batch": kernel_us(lambda: ops.eval_batch(pred32, d_buf, d_desc))}
    golden = {}
    for h, w, H, W in GOLDEN_SHAPES:
        s = EO.synth_sample(7, h, w, H, W)
        args = [s[k].cuda() for k in ("pred",) + KEYS]
        golden[f"{h}x{w}->{H}x{W}"] = kernel_us(lambda: ops.eval_sample(*args))
    res["eval_sample_kernel_us_golden_shapes"] = golden
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
