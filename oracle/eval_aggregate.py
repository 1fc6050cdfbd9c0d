"""ORACLE -- TEST INFRASTRUCTURE (only tests/ and tools/ may import this).

The dataset table of the reference's validation loop (discriminative_trainer.py:470-670) in plain Python over the
per-sample results of eval_oracle.evaluate_sample: the skip rule and the per-bucket mean of each metric.
"""
from __future__ import annotations

from .eval_oracle import METRICS


def skipped(result):
    """The validation loop's skip rule (discriminative_trainer.py:596-597): a sample with a NaN among its 20 metric values
    (raw and aligned) is left out of every mean."""
    return any(v != v for part in ("pred", "aligned") for v in result[part].values())


def aggregate(results, buckets, labels):
    """Dataset table over evaluate_sample dicts: per bucket (labels[i] is a name of buckets, or None) and overall,
    {"n", "n_skipped", "pred": {metric: mean}, "aligned": {metric: mean}}, each mean over the samples not skipped, summed
    in order (NaN when none is left)."""
    groups = {"overall": list(range(len(results)))}
    for name in buckets:
        groups[name] = [i for i, lab in enumerate(labels or ()) if lab == name]
    table = {}
    for name, idx in groups.items():
        used = [results[i] for i in idx if not skipped(results[i])]
        n = len(used)
        entry = {"n": n, "n_skipped": len(idx) - n}
        for part in ("pred", "aligned"):
            entry[part] = {}
            for m in METRICS:
                s = 0.0
                for r in used:
                    s += r[part][m]
                entry[part][m] = s / n if n else float("nan")
        table[name] = entry
    return table
