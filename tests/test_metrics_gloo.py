"""Host logic of the multi-rank ranking metrics (pangnn_b200/metrics.py) on CPU: world 2 and 3 over gloo.

The splitters, the run exchange, the offsets and the final combine run as in production; only the two kernel entry
points (``ops.metric_runs``, ``ops.metric_reduce``) are replaced by torch-CPU stand-ins defined HERE.  Every rank
must return exactly the single-process reference computed from all scores at once.
"""
import os
import struct
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _keys(scores):
    """The kernels' order key: ascending = decreasing score, -0.0 folded onto +0.0."""
    u = scores.astype(np.float32).view(np.uint32).astype(np.int64)
    u[u == 0x80000000] = 0
    asc = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    return ~asc & 0xFFFFFFFF


def _compact(keys, pos, neg):
    order = np.argsort(keys, kind="stable")
    k, p, n = keys[order], pos[order], neg[order]
    uk, start = np.unique(k, return_index=True)
    return np.stack((uk, np.add.reduceat(p, start) if k.size else p, np.add.reduceat(n, start) if k.size else n), 1)


def _cpu_metric_runs(scores=None, labels=None, runs=None, info=None, hist=None):
    if runs is not None:
        r = runs.numpy()
        out = _compact(r[:, 0], r[:, 1], r[:, 2]) if r.size else np.zeros((0, 3), np.int64)
        flags = 0
    else:
        s, y = scores.numpy(), labels.double().numpy()
        flags = (1 if np.isnan(s).any() else 0) | (2 if not np.isin(y, (0.0, 1.0)).all() else 0)
        yi = (y == 1).astype(np.int64)
        out = _compact(_keys(s), yi, 1 - yi) if s.size else np.zeros((0, 3), np.int64)
    n = runs.size(0) if runs is not None else scores.numel()
    full = np.zeros((n, 3), np.int64)
    full[:out.shape[0]] = out
    info.copy_(torch.tensor([out.shape[0], int(out[:, 1].sum()), int(out[:, 2].sum()), 0, 0, flags]))
    if hist is not None:
        hist.copy_(torch.from_numpy(np.bincount(out[:, 0] >> 16, minlength=65536).astype(np.int64)))
    return torch.from_numpy(full)


def _s64(x):
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >> 63 else x


def _reduce(runs, R, P, N, tp, fp):
    """Exact per-range numerators in Python ints (the kernels' formulas)."""
    shift = 127 - P.bit_length()
    auc = ap = 0
    best = (float("-inf"), (1 << 64) - 1)
    for key, pos, neg in runs[:R].tolist():
        tp1, fp1 = tp + pos, fp + neg
        auc += neg * (tp + tp1)
        if pos:
            ap += pos * ((tp1 << shift) // (tp1 + fp1))
        if P and N:
            j = float(tp1) / float(P) - float(fp1) / float(N)
            if j > best[0] or (j == best[0] and key < best[1]):
                best = (j, key)
        tp, fp = tp1, fp1
    return auc, ap, best, shift


def _cpu_metric_reduce(runs, params, out=None):
    R, P, N, tp0, fp0 = params.tolist()
    auc, ap, (j, key), shift = _reduce(runs, R, P, N, tp0, fp0)
    m = (1 << 64) - 1
    vals = [auc & m, auc >> 64, ap & m, ap >> 64, struct.unpack("<q", struct.pack("<d", j))[0], key, R, shift]
    res = torch.tensor([_s64(v) for v in vals], dtype=torch.int64)
    if out is not None:
        out.copy_(res)
        return out
    return res


def _reference(scores, labels):
    """Single-process exact reference over all scores."""
    from pangnn_b200.metrics import _finish
    yi = (labels == 1).astype(np.int64)
    runs = _compact(_keys(scores), yi, 1 - yi) if scores.size else np.zeros((0, 3), np.int64)
    P, N = int(yi.sum()), int(yi.size - yi.sum())
    auc, ap, (j, key), _ = _reduce(runs, runs.shape[0], P, N, 0, 0)
    return _finish(auc, ap, struct.unpack("<q", struct.pack("<d", j))[0], key, runs.shape[0], P, N)


def _worker(rank, world, init_file, parts, out_dir):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        from pangnn_b200 import metrics, ops
        ops.metric_runs, ops.metric_reduce = _cpu_metric_runs, _cpu_metric_reduce
        s, y = parts[rank]
        res = metrics.ranking_metrics(torch.from_numpy(s), torch.from_numpy(y))
        torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _split(scores, labels, world, rng, sizes=None):
    if sizes is None:
        cut = np.sort(rng.integers(0, scores.size + 1, world - 1))
        sizes = np.diff(np.concatenate(([0], cut, [scores.size])))
    perm = rng.permutation(scores.size)
    parts, o = [], 0
    for k in sizes:
        idx = perm[o:o + k]
        parts.append((scores[idx], labels[idx]))
        o += k
    return parts


def _cases():
    rng = np.random.default_rng(0)
    E = 3000
    y = (rng.random(E) < 0.2).astype(np.float32)
    ties = np.round(rng.random(E) * 50) / 50
    ties = np.where(y == 1, np.minimum(ties + 0.2, 1.0), ties).astype(np.float32)
    one_bin = (np.float32(0.75) + rng.integers(0, 300, E).astype(np.float32) * np.float32(2 ** -24)).astype(np.float32)
    equal = np.full(E, 0.5, np.float32)
    mixed = np.concatenate((ties[:E // 2], np.array([np.inf, -np.inf, -0.0, 0.0] * 10, np.float32)))
    return {
        "random": (ties, y, None),
        "one_bin": (one_bin, y, None),
        "equal_everywhere": (equal, y, None),
        "empty_rank": (ties, y, [E // 2, 0, E - E // 2]),
        "one_class_on_some_ranks": (np.sort(ties), (np.arange(E) >= E - 400).astype(np.float32), "contiguous"),
        "one_class_globally": (ties, np.ones(E, np.float32), None),
        "signed_zeros_and_inf": (mixed, (rng.random(mixed.size) < 0.3).astype(np.float32), None),
    }


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", list(_cases()))
def test_distributed_ranking_metrics_equal_the_single_process_reference(case, world):
    scores, labels, sizes = _cases()[case]
    rng = np.random.default_rng(world)
    if sizes == "contiguous":                                 # rank 0 only negatives, the last rank only positives
        b = np.linspace(0, scores.size, world + 1).astype(int)
        parts = [(scores[b[r]:b[r + 1]], labels[b[r]:b[r + 1]]) for r in range(world)]
    else:
        if sizes is not None and len(sizes) != world:
            sizes = sizes[:world - 1] + [scores.size - sum(sizes[:world - 1])]
        parts = _split(scores, labels, world, rng, sizes)
    ref = _reference(scores, labels)
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, os.path.join(tmp, "rdv"), parts, tmp), nprocs=world, join=True)
        outs = [torch.load(os.path.join(tmp, f"r{r}.pt")) for r in range(world)]
    for o in outs:
        assert o == ref
    if case == "one_class_globally":
        assert ref["auroc"] is None and ref["youden_threshold"] is None and ref["average_precision"] == 1.0


def test_reference_matches_sklearn_formulas():
    """The stand-ins' formulas are the contract: AUROC / AP of a small hand-checked case."""
    s = np.array([0.9, 0.8, 0.8, 0.3, 0.1], np.float32)
    y = np.array([1, 0, 1, 0, 0], np.float32)
    r = _reference(s, y)
    # runs: 0.9 (1,0), 0.8 (1,1), 0.3 (0,1), 0.1 (0,1); AUROC = (1*(1+2) + 1*(2+2) + 1*(2+2)) / (2*2*3)
    assert r["auroc"] == pytest.approx(11 / 12, abs=1e-15)
    assert r["average_precision"] == pytest.approx(0.5 * (1 / 1) + 0.5 * (2 / 3), abs=1e-15)
    assert r["youden_threshold"] == np.float32(0.8) and r["num_runs"] == 4


def test_key_round_trip():
    from pangnn_b200.metrics import key_to_score
    vals = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, 1e-45, -3e38, 0.5], np.float32)
    keys = _keys(vals)
    for v, k in zip(vals, keys):
        assert key_to_score(int(k)) == v
    assert keys[0] == keys[1]                                           # -0.0 and +0.0 share a key
    s = vals[np.argsort(keys, kind="stable")]
    assert all(a >= b for a, b in zip(s[:-1], s[1:]))                  # ascending keys = decreasing scores
