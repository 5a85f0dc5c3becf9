"""Exact ranking metrics on one GPU (pangnn_b200/metrics.py, csrc/metrics.cu) against sklearn, against exact rationals
computed with Python integers, and against ``train.youden_threshold``; order independence, degenerate and invalid
inputs, C3 scale, and the training flow's new statistics."""
import struct
from fractions import Fraction

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
skm = pytest.importorskip("sklearn.metrics")

TILE = 2048                                                   # kMTile of csrc/metrics.cu
DEV = "cuda:0"


def _exact(scores, labels):
    """(AUROC, AP) as Fractions from distinct-score runs in decreasing order (-0.0 == +0.0)."""
    s = scores.astype(np.float32).astype(np.float64) + 0.0     # + 0.0 folds -0.0
    y = labels.astype(np.int64)
    order = np.argsort(-s, kind="stable")
    s, y = s[order], y[order]
    P, N = int(y.sum()), int(y.size - y.sum())
    tp = fp = 0
    auc = 0
    ap = Fraction(0)
    i = 0
    while i < s.size:
        j = i
        while j < s.size and s[j] == s[i]:
            j += 1
        pos = int(y[i:j].sum())
        neg = (j - i) - pos
        auc += neg * (2 * tp + pos)
        tp, fp = tp + pos, fp + neg
        if pos:
            ap += Fraction(pos * tp, tp + fp)
        i = j
    return (Fraction(auc, 2 * P * N) if P and N else None), (ap / P if P else None)


def _case(kind, E, rng):
    y = (rng.random(E) < 0.25).astype(np.float32)
    if kind == "ties":
        s = np.round(rng.random(E) * 50) / 50 + 0.1 * y
    elif kind == "equal":
        s = np.full(E, 0.25)
    elif kind == "long_run":                                   # one run longer than several tiles in the middle
        s = rng.random(E) + y * 0.3
        s[E // 4: E // 4 + min(E // 2, 5 * TILE)] = 0.5
    elif kind == "inf":
        s = rng.standard_normal(E) + y
        s[rng.random(E) < 0.1] = np.inf
        s[rng.random(E) < 0.1] = -np.inf
    elif kind == "signed_zero":
        s = ((rng.random(E) < 0.4) * y).astype(np.float64)
        s[(s == 0) & (rng.random(E) < 0.5)] = -0.0
    else:
        s = rng.random(E) + 0.5 * y
    return s.astype(np.float32), y


def _finite(s):
    """sklearn rejects +-inf: the same ranking with +-inf moved just past the finite scores."""
    d = s.astype(np.float64)
    fin = d[np.isfinite(d)]
    hi, lo = (fin.max() + 1, fin.min() - 1) if fin.size else (1.0, -1.0)
    return np.where(d == np.inf, hi, np.where(d == -np.inf, lo, d))


def _run(s, y, label_dtype=torch.float32):
    from pangnn_b200.metrics import ranking_metrics
    return ranking_metrics(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV, label_dtype))


SIZES = [1, 2, 17, TILE - 1, TILE, TILE + 1, 1000, 100_000, 1_000_000]
KINDS = ["random", "ties", "equal", "long_run", "inf", "signed_zero"]


@pytest.mark.parametrize("E", SIZES)
@pytest.mark.parametrize("kind", KINDS)
def test_against_sklearn_and_exact(kind, E):
    rng = np.random.default_rng(E + len(kind))
    s, y = _case(kind, E, rng)
    r = _run(s, y)
    P = int(y.sum())
    N = E - P
    assert r["num_pos"] == P and r["num_neg"] == N
    assert r["num_runs"] == np.unique(s.astype(np.float64) + 0.0).size
    sk = _finite(s)
    if P and N:
        ref = skm.roc_auc_score(y, sk)
        assert abs(r["auroc"] - ref) <= 1e-12
    else:
        assert r["auroc"] is None
    if P:
        assert abs(r["average_precision"] - skm.average_precision_score(y, sk)) <= 1e-12
    else:
        assert r["average_precision"] is None
    if E <= 10_000:
        auc, ap = _exact(s, y)
        assert r["auroc"] == (float(auc) if auc is not None else None)           # bit-equal
        if ap is not None:
            assert abs(r["average_precision"] - float(ap)) <= 2 * np.spacing(float(ap))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("E", [1, 17, TILE + 1, 50_000])
def test_youden_equals_host_reference(kind, E):
    from pangnn_b200 import train
    rng = np.random.default_rng(7 * E)
    s, y = _case(kind, E, rng)
    ref = train.youden_threshold(torch.from_numpy(s), torch.from_numpy(y))
    got = _run(s, y)["youden_threshold"]
    assert (got is None and ref is None) or got == ref


def test_youden_none_cases():
    from pangnn_b200 import train
    s = np.array([0.1, 0.9], np.float32)
    for y in (np.array([1, 0], np.float32), np.array([1, 1], np.float32), np.array([0, 0], np.float32)):
        assert _run(s, y)["youden_threshold"] == train.youden_threshold(torch.from_numpy(s), torch.from_numpy(y))


@pytest.mark.parametrize("kind", ["ties", "random", "signed_zero"])
def test_order_independence_and_determinism(kind):
    rng = np.random.default_rng(3)
    s, y = _case(kind, 300_001, rng)
    a = _run(s, y)
    b = _run(s, y)
    perm = rng.permutation(s.size)
    c = _run(s[perm], y[perm])
    assert a == b == c


@pytest.mark.parametrize("dtype", [torch.float32, torch.int32, torch.int64, torch.uint8, torch.bool])
def test_label_dtypes(dtype):
    rng = np.random.default_rng(1)
    s, y = _case("ties", 5000, rng)
    assert _run(s, y, dtype) == _run(s, y)


def test_degenerate_and_invalid_inputs():
    from pangnn_b200 import ops
    from pangnn_b200._abi import PangnnError
    r = _run(np.zeros(0, np.float32), np.zeros(0, np.float32))
    assert r["auroc"] is None and r["average_precision"] is None and r["youden_threshold"] is None
    assert r["num_runs"] == 0
    s = np.linspace(0, 1, 100, dtype=np.float32)
    r = _run(s, np.zeros(100, np.float32))                                    # P = 0
    assert r["auroc"] is None and r["average_precision"] is None and r["youden_threshold"] is None
    r = _run(s, np.ones(100, np.float32))                                     # N = 0
    assert r["auroc"] is None and r["average_precision"] == 1.0 and r["youden_threshold"] is None
    bad = s.copy()
    bad[37] = np.nan
    with pytest.raises(PangnnError, match="NaN"):
        _run(bad, (s > 0.5).astype(np.float32))
    lab = (s > 0.5).astype(np.float32)
    lab[3] = 0.5
    with pytest.raises(PangnnError, match="label"):
        _run(s, lab)
    with pytest.raises(PangnnError, match="label"):
        _run(s, np.full(100, 2, np.int64), torch.int64)
    ops.LAUNCHES["count"] = 0
    _run(s, (s > 0.5).astype(np.float32))
    assert ops.LAUNCHES["count"] == 20                                         # 4 + 12 sort + 4 reduce


def test_c3_scale_against_python_int_reference():
    """E = 9.97e6 (C3): model-shaped probabilities with a saturated tail of ties at 1.0f."""
    rng = np.random.default_rng(11)
    E = 9_970_000
    y = (rng.random(E) < 0.18)
    logit = np.where(y, rng.normal(4.0, 3.0, E), rng.normal(-4.0, 3.0, E))
    s = (1.0 / (1.0 + np.exp(-logit))).astype(np.float32)
    s[rng.random(E) < 0.02] = 1.0
    r = _run(s, y.astype(np.float32))
    # numpy runs + Python ints
    u, inv = np.unique(-(s.astype(np.float64)), return_inverse=True)           # decreasing scores
    pos = np.bincount(inv, weights=y, minlength=u.size).astype(np.int64)
    cnt = np.bincount(inv, minlength=u.size).astype(np.int64)
    neg = cnt - pos
    tp = np.cumsum(pos)
    tp_prev = tp - pos
    P, N = int(tp[-1]), int(neg.sum())
    auc = int((neg * (tp_prev + tp)).sum())                                   # < 2^63: exact in int64
    assert r["num_runs"] == u.size and r["num_pos"] == P and r["num_neg"] == N
    assert r["auroc"] == float(Fraction(auc, 2 * P * N))
    fpc = np.cumsum(neg)
    m = pos > 0                                                                # 2^200 fixed point: error < runs * 2^-200
    ap = Fraction(sum((p * t << 200) // (t + f) for p, t, f in zip(pos[m].tolist(), tp[m].tolist(), fpc[m].tolist())),
                  P << 200)
    assert abs(r["average_precision"] - float(ap)) <= 2 * np.spacing(float(ap))


# ---- the training flow -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def flow(tmp_path_factory):
    from pangnn_b200 import ops, setup, train
    setup.reset()
    ops.clear_cache()
    tmp = tmp_path_factory.mktemp("metrics_flow")
    argv = ["--simulate_dataset", "300", "3", "0.5", "10", "3", "--train", "-e", "3", "-b", "32",
            "-o", str(tmp / "runs"), "-m", str(tmp / "absent.pkl"), "--seed", "1"]
    res = train.run(setup.parse(argv), device=DEV)
    yield res
    setup.reset()
    ops.clear_cache()


def test_flow_test_metrics_equal_sklearn(flow):
    t = flow["test"][0]
    g = flow["dataset"].test[0]
    prob, y = t["prob"].double().cpu().numpy(), g.y.cpu().numpy()
    assert abs(t["auroc"] - skm.roc_auc_score(y, prob)) <= 1e-12
    assert abs(t["average_precision"] - skm.average_precision_score(y, prob)) <= 1e-12
    from pangnn_b200 import train
    assert t["youden_threshold"] == train.youden_threshold(t["prob"].cpu(), g.y.cpu())


def test_flow_history_carries_epoch_metrics(flow):
    for h in flow["history"]:
        for k in ("auroc_train", "ap_train", "auroc_val", "ap_val"):
            assert h[k] is not None and np.isfinite(h[k]) and 0.0 <= h[k] <= 1.0, k


def test_flow_baselines(flow):
    from pangnn_b200 import train
    ds = flow["dataset"]
    t = flow["test"][0]
    y = ds.test[0].y.cpu()
    ref = {}
    for name, lab in (("base_labels", ds.base_labels), ("base_labels_raw", ds.base_labels_raw),
                      ("logit_baseline", t["logit_baseline"].cpu().tolist())):
        ref[name] = train.prf(*train.confusion(torch.tensor(lab), y), eps=0.0)
    assert t["baselines"] == ref
