"""ROC and precision-recall curves on one GPU (``metrics.roc_curve`` / ``metrics.precision_recall_curve``,
``pangnn_metric_curve``) bit for bit against sklearn, against a Python reference where sklearn rejects +-inf, and
against a numpy count reference at C3 size; input order, label dtypes, degenerate and invalid inputs, and the CSV files
of the training flow."""
import csv
import os

import numpy as np
import pytest
import torch

from tests.test_curves_gloo import ROC, PR, _keep, _reference, _same

pytestmark = pytest.mark.gpu
skm = pytest.importorskip("sklearn.metrics")

TILE = 2048                                                   # kMTile of csrc/metrics.cu
DEV = "cuda:0"


def _case(kind, E, rng):
    y = (rng.random(E) < 0.25).astype(np.float32)
    if kind == "ties":
        s = np.round(rng.random(E) * 50) / 50 + 0.1 * y
    elif kind == "equal":
        s = np.full(E, 0.25)
    elif kind == "saturated":                                 # a tail of ties at 1.0f
        s = 1.0 / (1.0 + np.exp(-(rng.standard_normal(E) * 3 + np.where(y == 1, 4.0, -4.0))))
        s[rng.random(E) < 0.05] = 1.0
    elif kind == "signed_zero":
        s = ((rng.random(E) < 0.4) * y).astype(np.float64)
        s[(s == 0) & (rng.random(E) < 0.5)] = -0.0
    elif kind == "tile_stretch":
        # distinct scores, and the runs ranked 1500..3499 all negative: identical (0, 1) runs across the first tile
        # edge, so the keep rule of run 2047 reads run 2048 from the next tile
        s = 1.0 - np.arange(E) / max(E, 1)
        y[1500:3500] = 0
        perm = rng.permutation(E)
        s, y = s[perm], y[perm]
    else:
        s = rng.random(E) + 0.5 * y
    return s.astype(np.float32), y


def _curves(s, y, drop, label_dtype=torch.float32):
    from pangnn_b200 import metrics
    sd, yd = torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV, label_dtype)
    roc = metrics.roc_curve(sd, yd, drop_intermediate=drop)
    pr = metrics.precision_recall_curve(sd, yd, drop_intermediate=drop)
    if roc is None:
        assert pr is None
        return None
    return tuple(t.cpu().numpy() for t in roc), tuple(t.cpu().numpy() for t in pr)


def _sklearn(s, y, drop):
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return skm.roc_curve(y, s, drop_intermediate=drop), skm.precision_recall_curve(y, s, drop_intermediate=drop)


def _assert_same(got, want):
    for g3, w3 in zip(got, want):
        for g, w in zip(g3, w3):
            assert _same(g, w), (g.dtype, w.dtype, g.shape, w.shape)


SIZES = [1, 2, 17, TILE - 1, TILE, TILE + 1, 5000, 100_000, 1_000_000]
KINDS = ["random", "ties", "equal", "saturated", "signed_zero", "tile_stretch"]


@pytest.mark.parametrize("E", SIZES)
@pytest.mark.parametrize("kind", KINDS)
def test_curves_equal_sklearn(kind, E):
    rng = np.random.default_rng(E + 3 * len(kind))
    s, y = _case(kind, E, rng)
    for drop in (True, False):
        _assert_same(_curves(s, y, drop), _sklearn(s, y, drop))


def test_tile_stretch_is_dropped_across_the_tile_edge():
    rng = np.random.default_rng(4)
    s, y = _case("tile_stretch", 5000, rng)
    (fpr, _, thr), (_, _, pthr) = _curves(s, y, True)
    (fpr_all, _, _), _ = _curves(s, y, False)
    assert fpr_all.size == 5001
    order = np.sort(s)[::-1]
    # runs 1500..3498 are followed by an identical negative run: neither rule keeps them, runs 2047 and 2048 included
    assert not np.isin(order[1500:3499], thr).any()
    assert not np.isin(order[1500:3499], pthr).any()
    assert fpr.size <= 5001 - 1999


def test_one_class_empty_and_invalid_inputs():
    from pangnn_b200 import metrics
    from pangnn_b200._abi import PangnnError
    s = np.linspace(0, 1, 100, dtype=np.float32)
    for y in (np.zeros(100, np.float32), np.ones(100, np.float32)):
        for drop in (True, False):
            got = _curves(s, y, drop)
            _assert_same(got, _sklearn(s, y, drop))
            (fpr, tpr, _), (_, rec, _) = got
            if y[0] == 0:
                assert np.isnan(tpr).all() and (rec[:-1] == 1.0).all()
            else:
                assert np.isnan(fpr).all()
    e = torch.zeros(0, device=DEV)
    assert metrics.roc_curve(e, e) is None and metrics.precision_recall_curve(e, e) is None
    bad = s.copy()
    bad[37] = np.nan
    with pytest.raises(PangnnError, match="roc_curve: a score is NaN"):
        _curves(bad, (s > 0.5).astype(np.float32), True)
    lab = (s > 0.5).astype(np.float32)
    lab[3] = 0.5
    with pytest.raises(PangnnError, match="label"):
        _curves(s, lab, False)
    with pytest.raises(PangnnError, match="precision_recall_curve: a label"):
        metrics.precision_recall_curve(torch.from_numpy(s).to(DEV), torch.full((100,), 2, device=DEV))


@pytest.mark.parametrize("E", [1, 17, TILE + 1, 50_000])
def test_infinite_scores_against_the_python_reference(E):
    rng = np.random.default_rng(E)
    y = (rng.random(E) < 0.3).astype(np.float32)
    s = (rng.standard_normal(E) + y).astype(np.float32)
    s[rng.random(E) < 0.1] = np.inf
    s[rng.random(E) < 0.1] = -np.inf
    s[rng.random(E) < 0.05] = -0.0
    for drop in (True, False):
        _assert_same(_curves(s, y, drop), _reference(s, y, drop))


@pytest.mark.parametrize("kind", ["ties", "saturated", "tile_stretch"])
def test_input_order_and_label_dtypes(kind):
    rng = np.random.default_rng(3)
    s, y = _case(kind, 300_001, rng)
    perm = rng.permutation(s.size)
    for drop in (True, False):
        ref = _curves(s, y, drop)
        _assert_same(_curves(s, y, drop), ref)
        _assert_same(_curves(s[perm], y[perm], drop), ref)
        for dt in (torch.int32, torch.int64, torch.uint8, torch.bool):
            _assert_same(_curves(s, y, drop, dt), ref)


def test_c3_scale_against_numpy_counts_and_youden():
    """E = 1e7 model-shaped probabilities with a saturated tail of ties at 1.0f, against runs from np.unique."""
    from pangnn_b200.metrics import ranking_metrics
    rng = np.random.default_rng(12)
    E = 10_000_000
    yb = rng.random(E) < 0.18
    logit = np.where(yb, rng.normal(4.0, 3.0, E), rng.normal(-4.0, 3.0, E))
    s = (1.0 / (1.0 + np.exp(-logit))).astype(np.float32)
    s[rng.random(E) < 0.02] = 1.0
    y = yb.astype(np.float32)
    u, inv = np.unique(-(s.astype(np.float64)), return_inverse=True)           # decreasing scores
    pos = np.bincount(inv, weights=y, minlength=u.size).astype(np.int64)
    neg = np.bincount(inv, minlength=u.size).astype(np.int64) - pos
    P, N = int(pos.sum()), int(neg.sum())
    for drop in (True, False):
        got = _curves(s, y, drop)
        want = []
        for mode in (ROC, PR):
            keep = _keep(pos, neg, mode) if drop else np.ones(u.size, bool)
            tp, fp, thr = np.cumsum(pos)[keep].astype(np.float64), np.cumsum(neg)[keep].astype(np.float64), -u[keep]
            if mode == ROC:
                want.append((np.r_[0.0, fp] / N, np.r_[0.0, tp] / P, np.r_[np.inf, thr]))
            else:
                want.append((np.r_[(tp / (tp + fp))[::-1], 1.0], np.r_[(tp / P)[::-1], 0.0],
                             thr[::-1].astype(np.float32)))
        _assert_same(got, want)
        if not drop:
            (fpr, tpr, thr), _ = got
            assert fpr.size == u.size + 1
            yt = ranking_metrics(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV))["youden_threshold"]
            if yt is not None:
                assert thr[int(np.argmax(tpr - fpr))] == yt


# ---- the training flow -----------------------------------------------------------------------------------------
def _read_csv(path):
    with open(path) as f:
        rows = list(csv.reader(f))
    return rows[0], [[float(v) if v else None for v in r] for r in rows[1:]]


@pytest.fixture(scope="module")
def flows(tmp_path_factory):
    from pangnn_b200 import ops, setup, train
    tmp = tmp_path_factory.mktemp("curves_flow")
    out = {}
    base = ["--simulate_dataset", "300", "3", "0.5", "10", "3", "-b", "32", "--seed", "1"]
    for name, extra in (("train", ["--train", "-e", "2", "-o", str(tmp / "train"), "-m", str(tmp / "absent.pkl")]),
                        ("inference", ["-o", str(tmp / "inference"), "-m", str(tmp / "train" / "absent.pkl")])):
        setup.reset()
        ops.clear_cache()
        out[name] = (train.run(setup.parse(base + extra), device=DEV), str(tmp / name))
    yield out
    setup.reset()
    ops.clear_cache()


@pytest.mark.parametrize("branch", ["train", "inference"])
def test_flow_writes_both_curves(flows, branch):
    from pangnn_b200 import metrics
    res, out_dir = flows[branch]
    prob, y = res["test"][0]["prob"], res["dataset"].test[0].y.to(DEV)
    head, rows = _read_csv(os.path.join(out_dir, "roc_curve.csv"))
    assert head == ["threshold", "fpr", "tpr"]
    fpr, tpr, thr = (t.cpu().numpy() for t in metrics.roc_curve(prob, y))
    assert _same(np.array(rows, np.float64).T, np.stack((thr, fpr, tpr)))
    head, rows = _read_csv(os.path.join(out_dir, "precision_recall_curve.csv"))
    assert head == ["threshold", "precision", "recall"]
    p, r, t = (a.cpu().numpy() for a in metrics.precision_recall_curve(prob, y, drop_intermediate=True))
    assert rows[-1] == [None, 1.0, 0.0]
    got = np.array(rows[:-1], np.float64).T
    assert _same(got[0].astype(np.float32), t) and np.array_equal(got[0], t.astype(np.float64))
    assert _same(got[1], p[:-1]) and _same(got[2], r[:-1])
