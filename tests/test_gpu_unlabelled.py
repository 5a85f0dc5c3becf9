"""Inference on genomes without a RIBAP table (``pangnn.py -a *.gff -s hits.tsv -r '' -m model.pkl``) on the committed
real-data excerpt, against the same run with ``-r ribap.csv``:

* the dataset: the same graph tensors, baselines and edge order, with ``y`` None;
* the one-GPU CLI (``train.run``): the same logits, predictions and groups file, the same per-edge table but for its
  ``homolog`` column (-1), no curve files;
* the genome-partitioned CLI (an NCCL group of one rank, and two ranks when two GPUs are visible): the same groups and
  per-edge files as the one-GPU unlabelled run.

The model is a seeded initialisation saved as ``model.pkl``.  Its threshold is put in the widest gap between the
middle half of the labelled run's probabilities, so that about half of the edges are predicted positive (the groups
file is not trivial) and no probability lies within rounding of the threshold.
"""
import os
import tempfile

import numpy as np
import pytest
import torch

from tests.helpers import rel_err
from tests.test_gpu_cli_dist import _run, _worker

pytestmark = pytest.mark.gpu

FIX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "parsers")
FILES = ["-a", os.path.join(FIX, "Cga_08-1274-3_RENAMED.gff"), os.path.join(FIX, "Cga_12-4358_RENAMED.gff"),
         "-s", os.path.join(FIX, "hits.tsv")]
RIBAP = ["-r", os.path.join(FIX, "ribap.csv")]
NONE = ["-r", ""]
MODES = {"default": [], "union_skip": ["--union_edge_weights", "--neighbours", "3", "--skip_connections"]}
CURVES = ("roc_curve.csv", "precision_recall_curve.csv")
TOL = 1e-5


def _gap_threshold(prob):
    """Midpoint of the widest gap between consecutive distinct probabilities of the middle half."""
    p = np.unique(prob.astype(np.float64))
    assert p.size >= 8, "the model gives too few distinct probabilities"
    lo, hi = p.size // 4, 3 * p.size // 4
    i = lo + int(np.argmax(p[lo + 1:hi + 1] - p[lo:hi]))
    assert p[i + 1] - p[i] > 1e-5, "no clear gap between the probabilities"
    return float((p[i] + p[i + 1]) / 2)


@pytest.fixture(scope="module", params=list(MODES), ids=list(MODES))
def runs(request):
    """One-GPU inference of a seeded ``model.pkl`` with and without labels, in a temporary directory."""
    from pangnn_b200 import setup
    from pangnn_b200.gnn import AlternateGCN
    extra = MODES[request.param]
    with tempfile.TemporaryDirectory() as tmp:
        model = os.path.join(tmp, "model.pkl")
        setup.reset()
        setup.parse(FILES + extra)                        # the scorer's input width follows --skip_connections
        torch.manual_seed(11)
        torch.save(AlternateGCN("cpu", None, False).state_dict(), model)
        setup.reset()
        base = FILES + extra + ["-m", model]
        probe = _run(base + RIBAP + ["-o", os.path.join(tmp, "probe")], "cuda:0")
        th = _gap_threshold(probe["test"][0]["prob"].cpu().numpy())
        base += ["--binary_threshold", repr(th)]
        dirs = {k: os.path.join(tmp, k) for k in ("labelled", "unlabelled")}
        res = {"labelled": _run(base + RIBAP + ["-o", dirs["labelled"]], "cuda:0"),
               "unlabelled": _run(base + NONE + ["-o", dirs["unlabelled"]], "cuda:0")}
        yield dict(tmp=tmp, base=base, dirs=dirs, res=res, mode=request.param)


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _rows(path):
    return [r.split(",") for r in open(path).read().splitlines()]


def test_dataset_without_labels_equals_the_labelled_graph(runs):
    a, b = runs["res"]["labelled"]["dataset"], runs["res"]["unlabelled"]["dataset"]
    ga, gb = a.test[0], b.test[0]
    assert ga.y is not None and gb.y is None
    assert a.class_balance is not None and b.class_balance is None
    keys = sorted(k for k, v in ga.__dict__.items() if torch.is_tensor(v) and k != "y")
    assert keys == sorted(k for k, v in gb.__dict__.items() if torch.is_tensor(v))
    assert ("union_edge_index" if runs["mode"] == "union_skip" else "neighbour_edge_index") in keys
    for k in keys:
        va, vb = getattr(ga, k), getattr(gb, k)
        assert va.dtype == vb.dtype and torch.equal(va, vb), k
    assert len(a.base_labels) == ga.edge_index.size(1) and a.base_labels == b.base_labels
    assert a.base_labels_raw == b.base_labels_raw
    assert a.gene_str_ids_lst == b.gene_str_ids_lst


def test_cli_inference_without_labels(runs):
    ta, tb = runs["res"]["labelled"]["test"][0], runs["res"]["unlabelled"]["test"][0]
    da, db = runs["dirs"]["labelled"], runs["dirs"]["unlabelled"]
    assert torch.equal(ta["logits"], tb["logits"]) and torch.equal(ta["pred"], tb["pred"])
    assert "f1" in ta and not {"f1", "tp", "loss", "auroc", "baselines"} & set(tb)
    k = int(tb["pred"].sum())
    assert tb["predicted_positive"] == k and 0 < k < tb["pred"].numel()
    groups = _read(os.path.join(da, "holiest_of_all_tables.csv"))
    assert groups and groups == _read(os.path.join(db, "holiest_of_all_tables.csv"))
    ra, rb = _rows(os.path.join(da, "q_score_vs_logit.csv")), _rows(os.path.join(db, "q_score_vs_logit.csv"))
    h = ra[0].index("homolog")
    assert ra[0] == rb[0] and len(ra) == len(rb) == tb["logits"].numel() + 1
    assert {r[h] for r in ra[1:]} <= {"0", "1"} and {r[h] for r in rb[1:]} == {"-1"}
    assert [r[:h] + r[h + 1:] for r in ra] == [r[:h] + r[h + 1:] for r in rb]
    for f in CURVES:
        assert os.path.exists(os.path.join(da, f)) and not os.path.exists(os.path.join(db, f)), f


def _same_outputs(one_gpu_dir, part_dir):
    """Groups file byte for byte; per-edge table equal in every field, the logit to fp32 rounding (the partition
    scores its edges through its own kernels' summation order); no curve files."""
    assert _read(os.path.join(part_dir, "holiest_of_all_tables.csv")) == \
        _read(os.path.join(one_gpu_dir, "holiest_of_all_tables.csv"))
    ra, rb = _rows(os.path.join(one_gpu_dir, "q_score_vs_logit.csv")), _rows(os.path.join(part_dir, "q_score_vs_logit.csv"))
    assert ra[0] == rb[0] and len(ra) == len(rb)
    c = ra[0].index("logit")
    assert [r[:c] + r[c + 1:] for r in ra] == [r[:c] + r[c + 1:] for r in rb]
    la, lb = (np.array([float(r[c]) for r in rows[1:]]) for rows in (ra, rb))
    assert rel_err(lb, la) < TOL
    for f in CURVES:
        assert not os.path.exists(os.path.join(part_dir, f)), f


def test_world1_group_inference_without_labels_matches_one_gpu(runs):
    tmp, part = runs["tmp"], os.path.join(runs["tmp"], "w1")
    _worker(0, 1, os.path.join(tmp, "rdv_w1"), [runs["base"] + NONE + ["-o", part]], tmp)
    out = dict(np.load(os.path.join(tmp, "run0_r0.npz")))
    ref = runs["res"]["unlabelled"]["test"][0]
    assert np.array_equal(out["pred"][np.argsort(out["edge_ids"])], ref["pred"].cpu().numpy().astype(np.int64))
    _same_outputs(runs["dirs"]["unlabelled"], part)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_world2_inference_without_labels_matches_one_gpu(runs):
    import torch.multiprocessing as mp
    tmp, part = runs["tmp"], os.path.join(runs["tmp"], "w2")
    mp.spawn(_worker, args=(2, os.path.join(tmp, "rdv_w2"), [runs["base"] + NONE + ["-o", part]], tmp),
             nprocs=2, join=True)
    _same_outputs(runs["dirs"]["unlabelled"], part)
