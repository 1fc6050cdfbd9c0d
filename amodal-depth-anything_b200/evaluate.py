"""Device-resident version of the reference's validation loop (eval.py -> discriminative_trainer.py:470-670; SURVEY.md
section 8 row f3) over batches: the model at the caller's batch size, then the per-sample post-ops of :542-613 for every
sample of the batch in one kernel (ada_eval_batch) and the per-bucket dataset sums in a second (ada_eval_accumulate).
The reference reads every sample's metrics back to the host and averages them there (val_metrics.update(name, value));
here nothing is read back until result().

Each sample's row is bit-equal to the model at batch 1 plus ops.eval_sample on it, and the dataset table is the same bits
however the samples are split into add() calls: the model and the eval kernel are batch-invariant, and the accumulator
adds rows in order. The difficulty bucket of a sample (discriminative_trainer.py:555-580) is the caller's to compute;
the evaluator only takes its name.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import ops

N_SLOTS = 22  # per accumulator group: n_used, n_skipped, 10 metric sums of pred, 10 of the aligned prediction


def _maps(name, maps, B):
    if len(maps) != B:
        raise ValueError(f"{name}: {len(maps)} maps for {B} samples")
    out = [np.asarray(m) for m in maps]
    for m in out:
        if m.ndim != 2:
            raise ValueError(f"{name}: maps must be [H, W], got shape {m.shape}")
    return out


def pack_targets(pred_shapes, depth_gt, depth_obs, visible_mask, object_mask, alloc=None):
    """Packs the ground truth of B samples for ada_eval_batch. pred_shapes: the [h, w] of each prediction, which lie one
    after another in the prediction buffer (a model output [B, 1, h, w] is exactly that). The other four are lists of B
    [H_i, W_i] arrays (numpy or CPU torch): depths as fp32, masks thresholded non-zero -> 1, each map at a 16-byte boundary
    (ops.pack_layout). alloc(nbytes) returns the uint8 numpy buffer to fill (np.empty when None).
    Returns (buffer, desc int64 [B, 9] in ada_eval_desc order)."""
    B = len(pred_shapes)
    gts, obss = _maps("depth_gt", depth_gt, B), _maps("depth_obs", depth_obs, B)
    viss, objs = _maps("visible_mask", visible_mask, B), _maps("object_mask", object_mask, B)
    for b in range(B):
        if not gts[b].shape == obss[b].shape == viss[b].shape == objs[b].shape:
            raise ValueError(f"sample {b}: depth_gt {gts[b].shape}, depth_obs {obss[b].shape}, visible_mask "
                             f"{viss[b].shape} and object_mask {objs[b].shape} differ")
    shapes = []
    for g in gts:
        H, W = g.shape
        shapes += [(H, W, 4), (H, W, 4), (H, W), (H, W)]     # fp32 maps as their bytes
    lay, end = ops.pack_layout(shapes)
    buf = alloc(end) if alloc is not None else np.empty(end, np.uint8)
    desc = np.empty((B, 9), np.int64)
    pred_off = 0
    for b in range(B):
        o_gt, o_obs, o_vis, o_obj = (lay[4 * b + k][0] for k in range(4))
        H, W = gts[b].shape
        h, w = pred_shapes[b]
        desc[b] = (pred_off, o_gt, o_obs, o_vis, o_obj, h, w, H, W)
        pred_off += h * w
        n = H * W
        buf[o_gt:o_gt + 4 * n].view(np.float32)[:] = gts[b].astype(np.float32, copy=False).ravel()
        buf[o_obs:o_obs + 4 * n].view(np.float32)[:] = obss[b].astype(np.float32, copy=False).ravel()
        np.not_equal(viss[b], 0, out=buf[o_vis:o_vis + n].reshape(H, W).view(np.bool_))
        np.not_equal(objs[b], 0, out=buf[o_obj:o_obj + n].reshape(H, W).view(np.bool_))
    return buf, desc


def bucket_ids(buckets, labels, B):
    """Bucket names -> int32 indices into `buckets`; labels None -> None (the samples count in "overall" only)."""
    if labels is None:
        return None
    if len(labels) != B:
        raise ValueError(f"{len(labels)} bucket labels for {B} samples")
    index = {name: k for k, name in enumerate(buckets)}
    for name in labels:
        if name not in index:
            raise ValueError(f"unknown bucket {name!r}; the evaluator's buckets are {tuple(buckets)}")
    return np.array([index[name] for name in labels], np.int32)


def table(acc, buckets):
    """Host accumulator [(len(buckets) + 1), 22] -> {"overall": entry, bucket: entry}; entry = {"n", "n_skipped",
    "pred": {metric: mean}, "aligned": {metric: mean}} (mean NaN where no sample was used)."""
    acc = np.asarray(acc, np.float64).reshape(len(buckets) + 1, N_SLOTS)

    def entry(r):
        n = float(r[0])
        mean = [float(v) / n if n > 0 else math.nan for v in r[2:]]
        return {"n": int(r[0]), "n_skipped": int(r[1]), "pred": dict(zip(ops.EVAL_METRICS, mean[:10])),
                "aligned": dict(zip(ops.EVAL_METRICS, mean[10:]))}
    res = {"overall": entry(acc[0])}
    for k, name in enumerate(buckets):
        res[name] = entry(acc[1 + k])
    return res


class AmodalEvaluator:
    """The validation loop of discriminative_trainer.py:470-670 on the device: add() per batch, result() once.
    Every call runs on the current stream of the model's device; keep one evaluator to one stream."""

    def __init__(self, model, buckets=()):
        self.model = model
        self.buckets = tuple(buckets)
        if len(set(self.buckets)) != len(self.buckets) or "overall" in self.buckets:
            raise ValueError(f"bucket names must be distinct and not 'overall': {self.buckets}")
        self.device = next(model.parameters()).device
        self._acc = torch.zeros((len(self.buckets) + 1) * N_SLOTS, dtype=torch.float64, device=self.device)
        self._pinned = None      # reused host staging: packed targets, and descriptor rows + bucket labels
        self._pinned_desc = None
        self._uploaded = None    # event after the last upload from the staging buffers (they are rewritten after it)

    def reset(self):
        self._acc.zero_()

    def _host_u8(self, n):
        if self._pinned is None or self._pinned.numel() < n:
            self._pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        return self._pinned.numpy()[:n]

    def _stage(self, pred_shapes, depth_gt, depth_obs, visible_mask, object_mask, bucket):
        """Packs the targets into the pinned staging buffer and uploads them, then the descriptor rows with the bucket
        labels behind them: one copy each."""
        B = len(pred_shapes)
        ids = bucket_ids(self.buckets, bucket, B)
        if self._uploaded is not None:
            self._uploaded.synchronize()         # the previous upload may still read the staging buffers
        buf, desc = pack_targets(pred_shapes, depth_gt, depth_obs, visible_mask, object_mask, self._host_u8)
        n_tab = 9 * B + (B + 1) // 2             # int64 slots: desc rows, then the int32 labels two to a slot
        if self._pinned_desc is None or self._pinned_desc.numel() < n_tab:
            self._pinned_desc = torch.empty(n_tab, dtype=torch.int64, pin_memory=True)
        tab = self._pinned_desc.numpy()
        tab[:9 * B] = desc.ravel()
        if ids is not None:
            tab[9 * B:n_tab].view(np.int32)[:B] = ids
        data = torch.empty(buf.size, dtype=torch.uint8, device=self.device)
        dtab = torch.empty(n_tab, dtype=torch.int64, device=self.device)
        data.copy_(self._pinned[:buf.size], non_blocking=True)
        dtab.copy_(self._pinned_desc[:n_tab], non_blocking=True)
        self._uploaded = torch.cuda.Event()
        self._uploaded.record()
        d_bucket = None if ids is None else dtab[9 * B:].view(torch.int32)[:B]
        return data, dtab[:9 * B].view(B, 9), d_bucket

    @torch.no_grad()
    def add(self, x, depth_gt, depth_obs, visible_mask, object_mask, *, guide_rgb=None, guide_mask=None,
            observation=None, bucket=None):
        """One validation batch: runs model(x, guide_rgb=..., guide_mask=..., observation=...) at the batch size of x
        (discriminative_trainer.py:537-541), then the post-ops of :542-613 for each sample against its own ground truth.
        depth_gt, depth_obs, visible_mask, object_mask: lists of B [H_i, W_i] arrays (numpy or CPU torch; masks non-zero =
        inside). bucket: None or B names from `buckets`. Returns the [B, 24] float64 device rows (layout of
        ops.eval_sample); no host synchronisation beyond waiting for the previous call's upload."""
        with torch.cuda.device(self.device):
            pred = self.model(x, guide_rgb=guide_rgb, guide_mask=guide_mask, observation=observation)
            B, h, w = pred.shape[0], pred.shape[-2], pred.shape[-1]
            data, desc, d_bucket = self._stage([(h, w)] * B, depth_gt, depth_obs, visible_mask, object_mask, bucket)
            rows = ops.eval_batch(pred.contiguous(), data, desc)
            ops.eval_accumulate(rows, d_bucket, len(self.buckets), self._acc)
        return rows

    def result(self):
        """One host read of the accumulator -> {"overall": entry, <bucket>: entry}, entry = {"n", "n_skipped",
        "pred": {metric: mean}, "aligned": {metric: mean}}, metric names of ops.EVAL_METRICS. A sample with a NaN among its
        20 metric values is counted in n_skipped and left out of the means (discriminative_trainer.py:596-597)."""
        return table(self._acc.cpu().numpy(), self.buckets)
