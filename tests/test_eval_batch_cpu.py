"""Host side of the batched validation loop (amodal-depth-anything_b200/evaluate.py): the packing of per-sample targets of
any size for ada_eval_batch, its rejection of malformed input, and the oracle's dataset table (skip rule, per-bucket
means) that tests/test_eval_batch_gpu.py holds the device accumulator to."""
import math

import numpy as np
import pytest
import torch

from amodal_depth_anything_b200 import evaluate as E
from oracle import eval_aggregate as EA
from oracle import eval_oracle as EO

SHAPES = [(1, 1), (7, 13), (375, 1242), (33, 5)]


def _targets(seed=0):
    rng = np.random.default_rng(seed)
    gts = [rng.random(s, dtype=np.float32) for s in SHAPES]
    obss = [torch.from_numpy(rng.random(s, dtype=np.float32)) for s in SHAPES]          # CPU torch is accepted too
    vis = [rng.integers(0, 3, s).astype(np.uint8) for s in SHAPES]
    obj = [torch.from_numpy(rng.random(s) > 0.5) for s in SHAPES]
    return gts, obss, vis, obj


def test_pack_targets_round_trip():
    gts, obss, vis, obj = _targets()
    preds = [(518, 518), (14, 28), (1, 1), (70, 98)]
    buf, desc = E.pack_targets(preds, gts, obss, vis, obj)
    assert buf.dtype == np.uint8 and desc.shape == (len(SHAPES), 9) and desc.dtype == np.int64
    off = 0
    for b, (H, W) in enumerate(SHAPES):
        p, o_gt, o_obs, o_vis, o_obj, h, w, H_, W_ = (int(v) for v in desc[b])
        assert (p, h, w, H_, W_) == (off, *preds[b], H, W)
        off += preds[b][0] * preds[b][1]
        for o in (o_gt, o_obs, o_vis, o_obj):
            assert o % 16 == 0
        n = H * W
        assert np.array_equal(buf[o_gt:o_gt + 4 * n].view(np.float32).reshape(H, W), gts[b])
        assert np.array_equal(buf[o_obs:o_obs + 4 * n].view(np.float32).reshape(H, W), obss[b].numpy())
        assert np.array_equal(buf[o_vis:o_vis + n].reshape(H, W), (vis[b] != 0).astype(np.uint8))
        assert np.array_equal(buf[o_obj:o_obj + n].reshape(H, W), obj[b].numpy().astype(np.uint8))
    # the maps do not overlap and the buffer ends with the last one
    spans = sorted((int(desc[b, k]), int(desc[b, k]) + SHAPES[b][0] * SHAPES[b][1] * (4 if k < 3 else 1))
                   for b in range(len(SHAPES)) for k in (1, 2, 3, 4))
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])) and spans[-1][1] == buf.size


def test_pack_targets_into_given_buffer():
    gts, obss, vis, obj = _targets(1)
    pool = np.full(1 << 23, 0xAB, np.uint8)
    buf, desc = E.pack_targets([(5, 5)] * 4, gts, obss, vis, obj, alloc=lambda n: pool[:n])
    ref, ref_desc = E.pack_targets([(5, 5)] * 4, gts, obss, vis, obj)
    assert np.shares_memory(buf, pool) and np.array_equal(desc, ref_desc)
    n = SHAPES[-1][0] * SHAPES[-1][1]
    assert np.array_equal(buf[desc[-1, 4]:desc[-1, 4] + n], ref[desc[-1, 4]:desc[-1, 4] + n])


@pytest.mark.parametrize("bad", ["shape", "ndim3", "ndim1", "count"])
def test_pack_targets_rejects_malformed_input(bad):
    gts, obss, vis, obj = _targets()
    if bad == "shape":
        vis[2] = vis[2][:, :-1]
    elif bad == "ndim3":
        gts[1] = gts[1][None]
    elif bad == "ndim1":
        obj[0] = obj[0].reshape(-1)
    else:
        obss = obss[:-1]
    with pytest.raises(ValueError):
        E.pack_targets([(14, 14)] * 4, gts, obss, vis, obj)


def test_bucket_ids():
    assert E.bucket_ids(("easy", "hard"), None, 3) is None
    ids = E.bucket_ids(("easy", "hard"), ["hard", "easy", "hard"], 3)
    assert ids.dtype == np.int32 and ids.tolist() == [1, 0, 1]
    with pytest.raises(ValueError):
        E.bucket_ids(("easy", "hard"), ["easy", "medium", "hard"], 3)
    with pytest.raises(ValueError):
        E.bucket_ids(("easy", "hard"), ["easy"], 3)


def _res(v, nan=None):
    r = {"scale": 1.0, "shift": 0.0, "pred": {m: v for m in EO.METRICS}, "aligned": {m: 2 * v for m in EO.METRICS}}
    if nan:
        r[nan[0]][nan[1]] = math.nan
    return r


def test_aggregate_known_answers():
    results = [_res(1.0), _res(2.0), _res(4.0, ("aligned", "rmse_log")), _res(8.0), _res(16.0, ("pred", "i_rmse"))]
    labels = ["a", "b", "a", None, "a"]
    t = EA.aggregate(results, ("a", "b", "c"), labels)
    assert t["overall"]["n"] == 3 and t["overall"]["n_skipped"] == 2
    assert t["overall"]["pred"]["rmse_linear"] == (1.0 + 2.0 + 8.0) / 3
    assert t["overall"]["aligned"]["delta1_acc"] == (2.0 + 4.0 + 16.0) / 3
    assert (t["a"]["n"], t["a"]["n_skipped"]) == (1, 2) and t["a"]["pred"]["log10"] == 1.0
    assert (t["b"]["n"], t["b"]["n_skipped"]) == (1, 0) and t["b"]["aligned"]["i_rmse"] == 4.0
    assert (t["c"]["n"], t["c"]["n_skipped"]) == (0, 0) and math.isnan(t["c"]["pred"]["abs_relative_difference"])
    assert EA.skipped(results[2]) and not EA.skipped(results[0])


def test_table_matches_aggregate():
    """evaluate.table (means of the device accumulator) and the oracle agree on an accumulator summed on the host."""
    results = [_res(0.5 * i, ("pred", "log10") if i == 3 else None) for i in range(1, 7)]
    labels = ["x", "y", "x", "x", "y", "y"]
    acc = np.zeros((3, E.N_SLOTS))
    for r, lab in zip(results, labels):
        row = [r["pred"][m] for m in EO.METRICS] + [r["aligned"][m] for m in EO.METRICS]
        for g in (0, 1 + ("x", "y").index(lab)):
            if EA.skipped(r):
                acc[g, 1] += 1
            else:
                acc[g, 0] += 1
                acc[g, 2:] += row
    assert E.table(acc, ("x", "y")) == EA.aggregate(results, ("x", "y"), labels)
