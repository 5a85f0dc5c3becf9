"""Host logic of the multi-rank ROC and precision-recall curves (pangnn_b200/metrics.py) on CPU: world 2 and 3 over
gloo.

The merge, the bound of every rank's key range, the size gather and the padded gather run as in production; the
kernel entry points are replaced by numpy stand-ins: the run and reduce stand-ins of ``test_metrics_gloo.py`` and the
curve stand-in defined HERE.  Every rank must return exactly sklearn's arrays (the Python reference where sklearn
rejects +-inf).
"""
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_metrics_gloo import _cases, _compact, _cpu_metric_reduce, _cpu_metric_runs, _keys, _split

ALL, ROC, PR = 0, 1, 2                                        # ops.CURVE_*
FIRST, FOLLOWED = 1, 2


def _key_scores(keys):
    """fp32 scores of order keys (the inverse of ``_keys``)."""
    asc = ~keys.astype(np.int64) & 0xFFFFFFFF
    u = np.where(asc & 0x80000000, asc & 0x7FFFFFFF, ~asc & 0xFFFFFFFF)
    return u.astype(np.uint32).view(np.float32)


def _keep(pos, neg, mode, bpos=0, bneg=0, flags=FIRST):
    """The kernels' keep rule over one piece of runs, with the bound of the next piece."""
    npos, nneg = np.append(pos[1:], bpos), np.append(neg[1:], bneg)
    if mode == ROC:
        keep = (npos != pos) | (nneg != neg)
    elif mode == PR:
        keep = (pos != 0) | (npos != 0)
    else:
        keep = np.ones(pos.size, bool)
    if pos.size:
        keep[0] |= bool(flags & FIRST)
        keep[-1] |= not flags & FOLLOWED
    return keep


def _cpu_metric_curve(runs, params, bound, mode, out=None):
    R, P, N, tp0, fp0 = params.tolist()[:5]
    r = runs.numpy()[:R]
    bpos, bneg, flags = bound.tolist()
    keep = _keep(r[:, 1], r[:, 2], mode, bpos, bneg, flags)
    K = int(keep.sum())
    n = runs.size(0)
    thr, tp, fp = np.zeros(n, np.float32), np.zeros(n, np.int64), np.zeros(n, np.int64)
    thr[:K] = _key_scores(r[keep, 0])
    tp[:K] = (tp0 + np.cumsum(r[:, 1]))[keep]
    fp[:K] = (fp0 + np.cumsum(r[:, 2]))[keep]
    res = (torch.from_numpy(thr), torch.from_numpy(tp), torch.from_numpy(fp),
           torch.tensor([K, int(r[:, 1].sum()), int(r[:, 2].sum())]))
    if out is None:
        return res
    for o, v in zip(out, res):
        o[:v.numel()] = v
    return out


def _reference(scores, labels, drop):
    """Single-process Python reference: (roc fpr, tpr, thresholds), (pr precision, recall, thresholds), or None."""
    if scores.size == 0:
        return None
    yi = (labels == 1).astype(np.int64)
    runs = _compact(_keys(scores), yi, 1 - yi)
    P, N = int(yi.sum()), int(yi.size - yi.sum())
    out = []
    for mode in (ROC, PR):
        keep = _keep(runs[:, 1], runs[:, 2], mode if drop else ALL)
        thr = _key_scores(runs[keep, 0])
        tp, fp = np.cumsum(runs[:, 1])[keep].astype(np.float64), np.cumsum(runs[:, 2])[keep].astype(np.float64)
        if mode == ROC:
            tp, fp = np.r_[0.0, tp], np.r_[0.0, fp]
            with np.errstate(invalid="ignore"):
                out.append((fp / N if N else np.full(fp.size, np.nan), tp / P if P else np.full(tp.size, np.nan),
                            np.r_[np.inf, thr.astype(np.float64)]))
        else:
            rec = tp / P if P else np.ones(tp.size)
            out.append((np.r_[(tp / (tp + fp))[::-1], 1.0], np.r_[rec[::-1], 0.0], thr[::-1]))
    return tuple(out)


def _sklearn(scores, labels, drop):
    import warnings
    skm = pytest.importorskip("sklearn.metrics")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return (skm.roc_curve(labels, scores, drop_intermediate=drop),
                skm.precision_recall_curve(labels, scores, drop_intermediate=drop))


def _same(a, b):
    """Bit-equal arrays of the same dtype (NaN equals NaN; -0.0 equals +0.0)."""
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def _worker(rank, world, init_file, parts, out_dir):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        from pangnn_b200 import metrics, ops
        ops.metric_runs, ops.metric_reduce = _cpu_metric_runs, _cpu_metric_reduce
        ops.metric_curve = _cpu_metric_curve
        s, y = (torch.from_numpy(a) for a in parts[rank])
        res = {}
        for drop in (True, False):
            roc = metrics.roc_curve(s, y, drop_intermediate=drop)
            pr = metrics.precision_recall_curve(s, y, drop_intermediate=drop)
            res[drop] = None if roc is None else (tuple(t.numpy() for t in roc), tuple(t.numpy() for t in pr))
        torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _curve_cases():
    rng = np.random.default_rng(1)
    cases = dict(_cases())
    # distinct scores, one negative each between a few positives at both ends: the ROC rule drops every run of the
    # stretch, across the key-range cut between ranks
    E = 3000
    s = np.linspace(0.01, 0.99, E).astype(np.float32)
    y = np.zeros(E, np.float32)
    y[:50] = y[-50:] = 1
    cases["cut_inside_identical_runs"] = (s, y, None)
    # two thirds of the distinct scores in one histogram bin: at world 3 the middle rank's key range is empty, so the
    # first rank's bound comes from the last one
    one_bin = np.float32(0.75) + np.arange(400, dtype=np.float32) * np.float32(2 ** -24)
    s = np.concatenate((one_bin, rng.random(150).astype(np.float32) * 0.5)).astype(np.float32)
    cases["next_nonempty_rank_two_away"] = (s, (rng.random(s.size) < 0.3).astype(np.float32), None)
    return cases


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", list(_curve_cases()))
def test_distributed_curves_equal_sklearn(case, world):
    scores, labels, sizes = _curve_cases()[case]
    rng = np.random.default_rng(world)
    if sizes == "contiguous":
        b = np.linspace(0, scores.size, world + 1).astype(int)
        parts = [(scores[b[r]:b[r + 1]], labels[b[r]:b[r + 1]]) for r in range(world)]
    else:
        if sizes is not None and len(sizes) != world:
            sizes = sizes[:world - 1] + [scores.size - sum(sizes[:world - 1])]
        parts = _split(scores, labels, world, rng, sizes)
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, os.path.join(tmp, "rdv"), parts, tmp), nprocs=world, join=True)
        outs = [torch.load(os.path.join(tmp, f"r{r}.pt"), weights_only=False) for r in range(world)]
    for drop in (True, False):
        ref = _reference(scores, labels, drop) if np.isinf(scores).any() else _sklearn(scores, labels, drop)
        for o in outs:
            for got, want in zip(o[drop], ref):
                assert all(_same(g, w) for g, w in zip(got, want)), (case, drop)
    if case == "cut_inside_identical_runs":
        (fpr, _, _), _ = outs[0][True]
        assert fpr.size == 5                                   # (0, 0), the two ends of both positive stretches


@pytest.mark.parametrize("case", list(_curve_cases()))
def test_reference_equals_sklearn(case):
    """The Python reference used for +-inf scores is sklearn on every finite case."""
    scores, labels, _ = _curve_cases()[case]
    if np.isinf(scores).any():
        scores = np.where(np.isinf(scores), np.float32(0.5), scores).astype(np.float32)
    for drop in (True, False):
        for got, want in zip(_reference(scores, labels, drop), _sklearn(scores, labels, drop)):
            assert all(_same(g, w) for g, w in zip(got, want)), (case, drop)


def test_keep_rules_are_sklearns_second_differences():
    """The run-count rules against sklearn's drop_intermediate masks written with cumulative counts."""
    rng = np.random.default_rng(2)
    for _ in range(50):
        K = int(rng.integers(3, 40))
        pos, neg = rng.integers(0, 3, K), rng.integers(0, 3, K)
        neg[pos + neg == 0] = 1
        tps, fps = np.cumsum(pos), np.cumsum(neg)
        roc = np.r_[True, np.logical_or(np.diff(fps, 2), np.diff(tps, 2)), True]
        pr = np.r_[True, np.logical_or(np.diff(tps[:-1]), np.diff(tps[1:])), True]
        assert np.array_equal(_keep(pos, neg, ROC), roc)
        assert np.array_equal(_keep(pos, neg, PR), pr)
