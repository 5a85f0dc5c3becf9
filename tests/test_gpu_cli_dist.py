"""``pangnn.py`` through the genome-partitioned driver (pangnn_b200/dist_train.py) against the one-GPU CLI.

* world 1: an NCCL group of one rank runs every part of the partitioned driver on one GPU;
* world 2 (needs 2 GPUs; skipped otherwise): two ranks over NCCL, plus ``--categorical_node`` and ``model.pkl`` files
  exchanged between world 1 and world 2 in both directions.

Each run is compared with ``train.run`` without a process group on the same flags: per-epoch losses, ``model.pkl``,
test logits and predictions, the curve files, ``q_score_vs_logit.csv`` and the ortholog groups.
"""
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest
import torch

from tests.helpers import rel_err

pytestmark = pytest.mark.gpu

SIM = ["--simulate_dataset", "300", "4", "0.5", "10", "3", "--seed", "1"]
TRAIN = ["--train", "--whole_graph_training", "-e", "3"]
UNION = ["--union_edge_weights", "--neighbours", "3", "--skip_connections"]
TOL = 1e-5


def _run(argv, device):
    from pangnn_b200 import ops, setup, train
    setup.reset()
    ops.clear_cache()
    try:
        return train.run(setup.parse(argv), device=device)
    finally:
        setup.reset()
        ops.clear_cache()


def _summary(res):
    """One rank's result as numpy arrays (what a spawned rank sends back)."""
    t = res["test"][0]
    ids = t["edge_ids"] if "edge_ids" in t else torch.arange(t["logits"].numel())
    return dict(edge_ids=ids.cpu().numpy(), logits=t["logits"].float().cpu().numpy(),
                prob=t["prob"].float().cpu().numpy(), pred=t["pred"].cpu().numpy().astype(np.int64),
                train_loss=np.array([h["train_loss"] for h in res["history"]]),
                val_loss=np.array([h["val_loss"] for h in res["history"]]))


def _worker(rank, world, init_file, runs, out_dir):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    try:
        for i, argv in enumerate(runs):
            np.savez(os.path.join(out_dir, f"run{i}_r{rank}.npz"), **_summary(_run(argv, dev)))
    finally:
        dist.destroy_process_group()


def _assemble(outs):
    """Per-rank summaries -> whole-graph arrays indexed by global edge id."""
    ids = np.concatenate([o["edge_ids"] for o in outs])
    assert np.array_equal(np.sort(ids), np.arange(ids.size))
    whole = {}
    for k in ("logits", "prob", "pred"):
        whole[k] = np.empty(ids.size, dtype=outs[0][k].dtype)
        for o in outs:
            whole[k][o["edge_ids"]] = o[k]
    return whole


def _same_predictions(a, b, prob_ref):
    clear = np.abs(prob_ref - 0.5) > 1e-5
    assert np.array_equal(a[clear], b[clear])


def _compare(ref, ref_dir, outs, out_dir, tmp):
    """A partitioned run (per-rank summaries ``outs``, files in ``out_dir``) against the one-GPU run ``ref``."""
    from pangnn_b200 import train
    from oracle import postprocess as opp
    r = _summary(ref)
    for k in ("train_loss", "val_loss"):
        assert len(outs[0][k]) == len(r[k])
        for o in outs:                                       # every rank reports the same global history
            assert np.array_equal(o[k], outs[0][k])
        assert np.all(np.abs(outs[0][k] - r[k]) <= TOL * np.abs(r[k])), k
    if len(r["train_loss"]):
        a = torch.load(os.path.join(ref_dir, "model.pkl"), map_location="cpu")
        b = torch.load(os.path.join(out_dir, "model.pkl"), map_location="cpu")
        assert list(a) == list(b)
        for k in a:
            assert float((a[k] - b[k]).abs().max()) <= 2e-5 * max(float(a[k].abs().max()), 1e-3), k
    whole = _assemble(outs)
    assert rel_err(whole["logits"], r["logits"]) < TOL
    _same_predictions(whole["pred"], r["pred"], r["prob"])
    # curves: byte for byte the one-GPU writer's files of the run's own probabilities on the whole graph
    g = ref["dataset"].test[0]
    check = os.path.join(tmp, "curves_check")
    train.write_curves(SimpleNamespace(y=g.y), {"prob": torch.from_numpy(whole["prob"]).to(g.y.device)}, check)
    for f in ("roc_curve.csv", "precision_recall_curve.csv"):
        assert open(os.path.join(out_dir, f), "rb").read() == open(os.path.join(check, f), "rb").read(), f
    # per-edge table
    ta, tb = (pd.read_csv(os.path.join(d, "q_score_vs_logit.csv")) for d in (ref_dir, out_dir))
    assert list(ta.columns) == list(tb.columns) and len(ta) == len(tb)
    for c in ta.columns:
        if c == "logit":
            assert rel_err(tb[c].to_numpy(), ta[c].to_numpy()) < TOL
        else:
            assert np.array_equal(ta[c].to_numpy(), tb[c].to_numpy()), c
    # ortholog groups: connected components of the run's own predicted edges (oracle)
    ei = g.edge_index.cpu().numpy()
    groups = opp.groups(opp.component_labels(ei[0], ei[1], whole["pred"], int(ref["dataset"].num_genes)))
    text = "".join(f"group_{i}, {', '.join(str(v) for v in grp)}\n" for i, grp in enumerate(groups))
    assert open(os.path.join(out_dir, "holiest_of_all_tables.csv")).read() == text


def _dirs(tmp, name):
    """Outputs under ``tmp/name``, parameters saved as ``tmp/name/model.pkl`` (``-m`` names a file that does not exist:
    training mode)."""
    return ["-o", os.path.join(tmp, name), "-m", os.path.join(tmp, "model.pkl")]


@pytest.mark.parametrize("extra", [[], UNION], ids=["default", "union_skip"])
def test_world1_group_matches_one_gpu_cli(extra):
    with tempfile.TemporaryDirectory() as tmp:
        ref = _run(SIM + TRAIN + extra + _dirs(tmp, "ref"), "cuda:0")
        _worker(0, 1, os.path.join(tmp, "rdv"), [SIM + TRAIN + extra + _dirs(tmp, "part")], tmp)
        out = dict(np.load(os.path.join(tmp, "run0_r0.npz")))
        _compare(ref, os.path.join(tmp, "ref"), [out], os.path.join(tmp, "part"), tmp)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_world2_matches_one_gpu_cli():
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        refs = {name: _run(SIM + TRAIN + extra + _dirs(tmp, f"ref_{name}"), "cuda:0")
                for name, extra in (("default", []), ("union", UNION), ("cat", ["--categorical_node"]))}
        runs = [SIM + TRAIN + _dirs(tmp, "w2_default"), SIM + TRAIN + UNION + _dirs(tmp, "w2_union"),
                SIM + TRAIN + ["--categorical_node"] + _dirs(tmp, "w2_cat"),
                SIM + ["-o", os.path.join(tmp, "w2_infer"), "-m", os.path.join(tmp, "ref_default", "model.pkl")]]
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdv"), runs, tmp), nprocs=2, join=True)
        outs = [[dict(np.load(os.path.join(tmp, f"run{i}_r{r}.npz"))) for r in range(2)] for i in range(len(runs))]
        _compare(refs["default"], os.path.join(tmp, "ref_default"), outs[0], os.path.join(tmp, "w2_default"), tmp)
        _compare(refs["union"], os.path.join(tmp, "ref_union"), outs[1], os.path.join(tmp, "w2_union"), tmp)
        # --categorical_node: the saved [N, 64] table holds every rank's trained rows
        a = torch.load(os.path.join(tmp, "ref_cat", "model.pkl"), map_location="cpu")
        b = torch.load(os.path.join(tmp, "w2_cat", "model.pkl"), map_location="cpu")
        assert a["embedding.weight"].shape == b["embedding.weight"].shape == (1200, 64)
        for k in a:
            assert float((a[k] - b[k]).abs().max()) <= 2e-5 * max(float(a[k].abs().max()), 1e-3), k
        _same_predictions(_assemble(outs[2])["pred"], _summary(refs["cat"])["pred"], _summary(refs["cat"])["prob"])
        # inference at world 2 from the world-1 model.pkl == the world-1 test predictions of that model
        ref = _summary(refs["default"])
        _same_predictions(_assemble(outs[3])["pred"], ref["pred"], ref["prob"])
        # inference at world 1 from the world-2 model.pkl == the world-2 test predictions of that model
        w2 = _assemble(outs[0])
        inf = _summary(_run(SIM + ["-o", os.path.join(tmp, "w1_infer"), "-m", os.path.join(tmp, "w2_default", "model.pkl")],
                            "cuda:0"))
        _same_predictions(inf["pred"], w2["pred"], w2["prob"])
