"""ada_eval_batch / ada_eval_accumulate and AmodalEvaluator (the validation loop over batches of samples of any size,
SURVEY.md section 8 row f3) on a B200: the golden fixtures in one batch and alone, bit-equal rows in any batch and on
every run, no read or write outside a sample's maps or its output row, the skip rule, dataset tables that do not depend
on how the samples are split into calls, and the evaluator end to end against the model at batch 1 plus eval_sample."""
import ctypes
import math

import numpy as np
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from amodal_depth_anything_b200 import _lib as L
from amodal_depth_anything_b200 import evaluate as E
from amodal_depth_anything_b200 import ops
from oracle import eval_aggregate as EA
from oracle import eval_oracle as EO
from oracle import synth
from tests.test_eval_gpu import _check
from tests.test_eval_oracle_golden import golden_cases, load_case

pytestmark = pytest.mark.gpu

ARGS = ("pred", "depth_gt", "depth_obs", "visible_mask", "object_mask")


def _bits(t):
    return t.contiguous().view(torch.int64).cpu()


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _eval_batch(samples, spaced=False, out=None):
    """ops.eval_batch over samples (evaluate_sample argument dicts, CPU). spaced: every prediction and map sits between
    0xFF bytes (NaN as fp32, 0xFF as a mask), 64 of them on either side."""
    preds = [s["pred"].reshape(s["pred"].shape[-2:]) for s in samples]
    buf, desc = E.pack_targets([p.shape for p in preds], *[[s[k] for s in samples] for k in ARGS[1:]])
    if not spaced:
        pred = torch.cat([p.reshape(-1) for p in preds])
    else:
        gap = 64
        off = gap // 4
        pred = torch.full((sum(p.numel() for p in preds) + gap // 4 * (len(preds) + 1),), math.nan)
        for b, p in enumerate(preds):
            pred[off:off + p.numel()] = p.reshape(-1)
            desc[b, 0] = off
            off += p.numel() + gap // 4
        sizes = [4, 4, 1, 1]
        new = np.full(int(sum(desc[b, 7] * desc[b, 8] * sz for b in range(len(samples)) for sz in sizes))
                      + (gap + 16) * (4 * len(samples) + 1), 0xFF, np.uint8)
        off = gap
        desc = desc.copy()
        for b in range(len(samples)):
            n = int(desc[b, 7] * desc[b, 8])
            for k, sz in enumerate(sizes):
                o = int(desc[b, 1 + k])
                new[off:off + n * sz] = buf[o:o + n * sz]
                desc[b, 1 + k] = off
                off = (off + n * sz + gap + 15) // 16 * 16      # fp32 maps stay 4-byte aligned, as the ABI requires
        assert off <= new.size
        buf = new
    return ops.eval_batch(pred.cuda(), torch.from_numpy(buf).cuda(), torch.from_numpy(desc).cuda(), out=out)


def _single(s):
    return ops.eval_sample(*[s[k].cuda() for k in ARGS])


def _goldens():
    return [load_case(p) for p in golden_cases()]


def _mixed():
    """Goldens plus ground truths of 1x1, 7x13 and 1080x1920 and a prediction larger than its ground truth."""
    return [s for s, _ in _goldens()] + [EO.synth_sample(101, 14, 14, 1, 1), EO.synth_sample(102, 28, 42, 7, 13),
                                         EO.synth_sample(103, 518, 518, 1080, 1920), EO.synth_sample(104, 140, 154, 70, 60),
                                         EO.synth_sample(105, 70, 98, 500, 333), EO.synth_sample(106, 98, 70, 64, 64)]


def test_goldens_in_one_batch_and_alone():
    cases = _goldens()
    together = _eval_batch([s for s, _ in cases])
    for b, (s, want) in enumerate(cases):
        for row in (together[b], _eval_batch([s])[0]):
            got = ops.eval_sample_dict(row)
            assert got["n_visible"] == int(s["visible_mask"].sum()) and got["n_object"] == int(s["object_mask"].sum())
            _check(got, want)
            _check(got, EO.evaluate_sample(**s))


def test_rows_do_not_depend_on_the_batch_or_the_run():
    samples = _mixed()
    rows = _eval_batch(samples)
    again = _eval_batch(samples)
    rev = _eval_batch(samples[::-1])
    assert _same(rows, again)
    for b, s in enumerate(samples):
        assert _same(rows[b], _eval_batch([s])[0]), b
        assert _same(rows[b], rev[len(samples) - 1 - b]), b
        assert _same(rows[b], _single(s)), b


def test_no_access_outside_a_sample():
    samples = _mixed()
    B = len(samples)
    out = torch.full((B + 2, 24), math.nan, dtype=torch.float64, device="cuda")
    guard = _bits(out[0])
    _eval_batch(samples, spaced=True, out=out[1:B + 1])
    assert torch.equal(_bits(out[0]), guard) and torch.equal(_bits(out[B + 1]), guard)
    assert _same(out[1:B + 1], _eval_batch(samples))


def _degenerate():
    empty_obj = EO.synth_sample(201, 70, 70, 90, 120)
    empty_obj["object_mask"] = torch.zeros_like(empty_obj["object_mask"])
    empty_vis = EO.synth_sample(202, 70, 70, 90, 120)
    empty_vis["visible_mask"] = torch.zeros_like(empty_vis["visible_mask"])
    negative = EO.synth_sample(64, 70, 70, 120, 160)
    negative["depth_obs"] = 1.0 - 2.0 * negative["depth_gt"]   # as test_eval_sample_nan_semantics
    return [EO.synth_sample(200, 70, 70, 90, 120), empty_obj, empty_vis, negative]


def test_degenerate_samples_in_a_batch():
    samples = _degenerate()
    rows = _eval_batch(samples)
    for b, s in enumerate(samples):
        assert _same(rows[b], _single(s))
    got = [ops.eval_sample_dict(r) for r in rows]
    want = [EO.evaluate_sample(**s) for s in samples]
    for b in (0, 1, 3):
        for v in ("pred", "aligned"):
            for m in EO.METRICS:
                assert math.isnan(got[b][v][m]) == math.isnan(want[b][v][m]), (b, v, m)
    # an empty visible mask: the kernel's 2x2 normal equations are singular (scale and shift NaN, so the aligned depth is
    # NaN: no delta comparison holds and every other aligned metric is NaN); np.linalg.lstsq returns its minimum-norm
    # answer 0 instead. The raw prediction's metrics agree.
    assert math.isnan(got[2]["scale"]) and math.isnan(got[2]["shift"])
    for m in EO.METRICS:
        assert got[2]["aligned"][m] == 0.0 if m.startswith("delta") else math.isnan(got[2]["aligned"][m]), m
    assert got[2]["n_visible"] == 0 and got[1]["n_object"] == 0
    for m in EO.METRICS:
        a, w = got[2]["pred"][m], want[2]["pred"][m]
        assert abs(a - w) <= (1e-5 if m.startswith("delta") else 1e-4 * max(abs(w), 1e-3)), m
    assert [EA.skipped(g) for g in got] == [False, True, True, True]
    acc = torch.zeros(E.N_SLOTS, dtype=torch.float64, device="cuda")
    ops.eval_accumulate(rows, None, 0, acc)
    t = E.table(acc.cpu().numpy(), ())
    assert (t["overall"]["n"], t["overall"]["n_skipped"]) == (1, 3)
    assert t["overall"]["pred"] == got[0]["pred"] and t["overall"]["aligned"] == got[0]["aligned"]


def _model(enc="vits"):
    torch.manual_seed(0)
    m = pkg.AmodalDAv2(guide_type="mask+observation", encoder=enc, pretrained=False)
    m.load_state_dict(synth.make_state_dict(enc, "mask+observation", seed=3), strict=True)
    return m.cuda().eval()


def _targets(n, sizes, seed):
    ts = []
    for i in range(n):
        H, W = sizes[i % len(sizes)]
        s = EO.synth_sample(seed + i, 14, 14, H, W)
        if not s["visible_mask"].any():      # the oracle's lstsq answers 0 where the kernel's scale is NaN (see above)
            s["visible_mask"] = ~s["object_mask"]
        if i % 7 == 3:
            s["object_mask"] = torch.zeros_like(s["object_mask"])     # skipped: 0/0
        ts.append(s)
    return ts


def _add_all(ev, inp, ts, labels, chunk):
    rows = []
    for i in range(0, len(ts), chunk):
        sl = slice(i, i + chunk)
        rows.append(ev.add(inp["x"][sl].cuda(), *[[t[k] for t in ts[sl]] for k in ARGS[1:]],
                           guide_mask=inp["guide_mask"][sl].cuda(), observation=inp["observation"][sl].cuda(),
                           bucket=None if labels is None else labels[sl]))
    return torch.cat(rows), ev.result()


def _table_bits(t):
    return repr({g: (e["n"], e["n_skipped"], [float(e[v][m]).hex() for v in ("pred", "aligned") for m in EO.METRICS])
                 for g, e in t.items()})


def test_accumulator_does_not_depend_on_the_split():
    model = _model()
    n, buckets = 40, ("easy", "medium", "hard")
    inp = synth.make_inputs(n, 70, 70, seed=5)
    ts = _targets(n, [(40, 50), (70, 70), (33, 91)], seed=300)
    labels = [buckets[(i * 7) % 3] for i in range(n)]
    runs = []
    for chunk in (1, 5, 20):
        ev = E.AmodalEvaluator(model, buckets)
        runs.append(_add_all(ev, inp, ts, labels, chunk))
    rows, table = runs[0]
    for r, t in runs[1:]:
        assert _same(r, rows) and _table_bits(t) == _table_bits(table)
    # an in-order fp64 sum of the rows, divided on the host
    rh = rows.cpu().numpy()
    for g in ("overall",) + buckets:
        idx = [i for i in range(n) if g == "overall" or labels[i] == g]
        used = [i for i in idx if not np.isnan(rh[i, 2:22]).any()]
        assert (table[g]["n"], table[g]["n_skipped"]) == (len(used), len(idx) - len(used))
        for j, m in enumerate(EO.METRICS):
            for v, col in (("pred", 2 + j), ("aligned", 12 + j)):
                s = 0.0
                for i in used:
                    s += float(rh[i, col])
                assert table[g][v][m] == s / len(used), (g, v, m)
    # the oracle's table over the oracle's per-sample results
    with torch.no_grad():
        preds = model(inp["x"].cuda(), guide_mask=inp["guide_mask"].cuda(), observation=inp["observation"].cuda()).cpu()
    results = [EO.evaluate_sample(preds[i:i + 1], *[ts[i][k] for k in ARGS[1:]]) for i in range(n)]
    want = EA.aggregate(results, buckets, labels)
    for g in want:
        assert (table[g]["n"], table[g]["n_skipped"]) == (want[g]["n"], want[g]["n_skipped"])
        _check(dict(table[g], scale=1.0, shift=0.0), dict(want[g], scale=1.0, shift=0.0))


def test_evaluator_end_to_end():
    model = _model()
    sizes = [(375, 1242), (126, 98), (1, 1), (518, 518), (200, 333), (64, 700)]
    B = len(sizes)
    inp = synth.make_inputs(B, 126, 98, seed=7)
    ts = [EO.synth_sample(400 + i, 14, 14, H, W) for i, (H, W) in enumerate(sizes)]
    want = []
    with torch.no_grad():
        for i in range(B):
            pred = model(inp["x"][i:i + 1].cuda(), guide_mask=inp["guide_mask"][i:i + 1].cuda(),
                         observation=inp["observation"][i:i + 1].cuda())
            want.append(ops.eval_sample(pred, *[ts[i][k].cuda() for k in ARGS[1:]]))
    want = torch.stack(want)
    ev = E.AmodalEvaluator(model)
    rows, table = _add_all(ev, inp, ts, None, B)
    assert _same(rows, want)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ev2 = pkg.AmodalEvaluator(model)
        rows2, table2 = _add_all(ev2, inp, ts, None, B)
        rows2 = rows2.clone()
    side.synchronize()
    assert _same(rows2, want) and _table_bits(table2) == _table_bits(table)
    ev.reset()
    assert ev.result()["overall"]["n"] == 0


def test_abi_rejects_bad_arguments():
    lib = L.load()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    p = ctypes.c_void_p(buf.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    calls = [
        lambda: lib.ada_eval_batch(p, p, p, 0, p, st),
        lambda: lib.ada_eval_batch(p, p, p, -3, p, st),
        lambda: lib.ada_eval_batch(p, p, p, 65536, p, st),
        lambda: lib.ada_eval_batch(None, p, p, 1, p, st),
        lambda: lib.ada_eval_batch(p, None, p, 1, p, st),
        lambda: lib.ada_eval_batch(p, p, None, 1, p, st),
        lambda: lib.ada_eval_batch(p, p, p, 1, None, st),
        lambda: lib.ada_eval_accumulate(p, 0, None, 0, p, st),
        lambda: lib.ada_eval_accumulate(p, 65536, None, 0, p, st),
        lambda: lib.ada_eval_accumulate(p, 1, None, -1, p, st),
        lambda: lib.ada_eval_accumulate(None, 1, None, 0, p, st),
        lambda: lib.ada_eval_accumulate(p, 1, None, 0, None, st),
    ]
    for i, call in enumerate(calls):
        assert call() == L.ADA_EINVAL, i
        assert lib.ada_last_error().decode(), i
    torch.cuda.synchronize()
