"""``--edge_split`` on the GPU: the split kernel against the numpy rule, the training scorer with unlabelled edges
(``y < 0``) against fp64 autograd of the masked BCE, ``forward_loss`` with train labels against the oracle model, and
the CLI on one GPU, in inference from its own ``model.pkl`` and in an NCCL group (world 1, and 2 with two GPUs)."""
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests.helpers import GRAD_TOL, VARIANT_FLAGS, assert_close, golden_graph, oracle_model, rel_err
from tests.test_edge_split_host import split_rule
from tests.test_gpu_scorer import NAMES, make, oracle_logits

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


# ------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E", [0, 1, 255, 256, 1000, 100_003])
@pytest.mark.parametrize("seed,val,test", [(0, 0.15, 0.15), (12345678901, 0.01, 0.5), (3, 0.4, 0.0001)])
def test_split_kernel_bit_exact(E, seed, val, test):
    from pangnn_b200.edge_split import split_codes
    rng = np.random.default_rng(E)
    s = rng.integers(0, 2 ** 31, E).astype(np.int32)
    d = rng.integers(0, 2 ** 31, E).astype(np.int32)
    if E >= 4:                                               # the largest ids, in both orders
        s[:4] = [2 ** 31 - 1, 0, 2 ** 31 - 1, 2 ** 31 - 2]
        d[:4] = [0, 2 ** 31 - 1, 2 ** 31 - 2, 2 ** 31 - 1]
    got = split_codes(torch.from_numpy(s).to(DEV), torch.from_numpy(d).to(DEV), seed, val, test).cpu().numpy()
    assert got.dtype == np.int8 and got.shape == (E,)
    assert np.array_equal(got, split_rule(s, d, seed, val, test))


def _scorer_inputs(E, skip, seed):
    N = 700
    h, ei, P, sk, y = make(N, E, skip, seed)
    mask = torch.rand(ei.size(1), generator=torch.Generator().manual_seed(seed + 1)) < 0.4    # held out
    return N, h, ei, P, sk, y, mask


def _train_call(N, h, ei, P, sk, y, pw, scale):
    from pangnn_b200 import ops
    wcat, w1c = ops.split_w1(P["w1"].to(DEV), sk is not None)
    pq = ops.node_linear(h.to(DEV), wcat)
    gs = ops.GraphStruct(ei.to(DEV), N)
    logits = torch.empty(ei.size(1), device=DEV)
    loss_sum = torch.zeros(1, dtype=torch.float64, device=DEV)
    da1, grads = ops.edge_score_train(pq, w1c, P["b1"].to(DEV), P["w2"].to(DEV), P["b2"].to(DEV), P["w3"].to(DEV),
                                      P["b3"].to(DEV), gs, None if sk is None else sk.to(DEV), y=y.to(DEV),
                                      pos_weight=pw, scale=scale, logits=logits, loss_sum=loss_sum)
    return logits, loss_sum, da1, grads.clone()


@pytest.mark.parametrize("E", [129, 33_333])
@pytest.mark.parametrize("skip", [False, True])
def test_scorer_unlabelled_edges(E, skip):
    from pangnn_b200 import ops
    N, h, ei, P, sk, y, mask = _scorer_inputs(E, skip, E)
    E = ei.size(1)
    ym = torch.where(mask, torch.full_like(y, -1.0), y)
    n = int((~mask).sum())
    pw = 2.3
    # logits bit-identical to the all-labelled call; da1 rows of unlabelled edges exactly 0
    z_all, _, _, _ = _train_call(N, h, ei, P, sk, y, pw, 1.0 / E)
    z, loss_sum, da1, _ = _train_call(N, h, ei, P, sk, ym, pw, 1.0 / n)
    assert torch.equal(z, z_all)
    assert bool((da1[mask.to(DEV)] == 0).all())
    # loss and every gradient against fp64 autograd of the masked BCE
    ho = h.double().requires_grad_(True)
    Po = {k: v.double().requires_grad_(True) for k, v in P.items()}
    zo = oracle_logits(ho, ei, Po, None if sk is None else sk.double())
    keep = ~mask
    lo = torch.nn.functional.binary_cross_entropy_with_logits(
        zo[keep], y[keep].double(), pos_weight=torch.tensor(pw, dtype=torch.float64), reduction="sum") / n
    lo.backward()
    hd = h.clone().to(DEV).requires_grad_(True)
    Pd = {k: v.clone().to(DEV).requires_grad_(True) for k, v in P.items()}
    gs = ops.GraphStruct(ei.to(DEV), N)
    ld, zd = ops.EdgeScoreBCEFn.apply(hd, *[Pd[k] for k in NAMES], gs, None if sk is None else sk.to(DEV),
                                      ym.to(DEV), pw, n)
    ld.backward()
    assert abs(ld.item() - lo.item()) <= TOL * abs(lo.item())
    assert abs(float(loss_sum) / n - lo.item()) <= TOL * abs(lo.item())
    assert_close("logits", zd.cpu().numpy(), zo.detach().numpy(), TOL)
    assert_close("dh", hd.grad.cpu().numpy(), ho.grad.numpy(), GRAD_TOL)
    for k in NAMES:
        assert_close(f"d{k}", Pd[k].grad.cpu().numpy(), Po[k].grad.numpy(), GRAD_TOL)


def test_scorer_all_unlabelled_is_zero():
    N, h, ei, P, sk, y, _ = _scorer_inputs(5000, True, 4)
    ym = torch.full_like(y, -1.0)
    z_all, _, _, _ = _train_call(N, h, ei, P, sk, y, 1.7, 1.0)
    z, loss_sum, da1, grads = _train_call(N, h, ei, P, sk, ym, 1.7, 1.0)
    assert torch.equal(z, z_all)
    assert float(loss_sum) == 0.0
    assert bool((da1[:ei.size(1)] == 0).all()) and bool((grads == 0).all())


def test_scorer_chunked_equals_single_launch():
    from pangnn_b200 import ops
    N, h, ei, P, sk, y, mask = _scorer_inputs(40_000, True, 8)
    key, order = torch.sort(ei[0] * N + ei[1])                # (src, dst) sorted: the chunked form's layout
    ei = torch.stack((key // N, key % N))
    sk, y, mask = sk[order], y[order], mask[order]
    ym = torch.where(mask, torch.full_like(y, -1.0), y).to(DEV)
    n = int((~mask).sum())
    wcat, w1c = ops.split_w1(P["w1"].to(DEV), True)
    pq = ops.node_linear(h.to(DEV), wcat).detach()
    out = []
    old = ops.SCORER_CHUNK_EDGES["n"]
    for chunk in (old, 4096):
        ops.SCORER_CHUNK_EDGES["n"] = chunk
        try:
            gs = ops.GraphStruct(ei.to(DEV), N)
            pqd = pq.clone().requires_grad_(True)
            Pd = {k: v.clone().to(DEV).requires_grad_(True) for k, v in P.items() if k != "w1"}
            loss, z = ops.EdgeScoreBCEPQFn.apply(pqd, w1c.detach(), Pd["b1"], Pd["w2"], Pd["b2"], Pd["w3"], Pd["b3"],
                                                 gs, sk.to(DEV), ym, 1.9, 1.0 / n)
            loss.backward()
            out.append([loss.detach(), z, pqd.grad] + [Pd[k].grad for k in ("b1", "w2", "b2", "w3", "b3")])
        finally:
            ops.SCORER_CHUNK_EDGES["n"] = old
    for a, b in zip(*out):
        assert rel_err(b.cpu().numpy(), a.cpu().numpy()) <= 1e-5


# ------------------------------------------------------------------------------------------------
# model: forward_loss with train labels against the oracle model
# ------------------------------------------------------------------------------------------------
@pytest.fixture
def flags():
    from pangnn_b200 import gnn, ops, setup
    setup.reset()
    ops.clear_cache()
    yield setup.args
    gnn.set_operator_layer("function")
    setup.reset()
    ops.clear_cache()


MODEL_CASES = [("c1", "default", {}), ("c1", "union_skip", {}), ("c2", "default", {}), ("c2", "union_skip", {}),
               ("sim5", "union_n4", {}), ("c1", "cosine", {}), ("c1", "default", {"node_dim": 32})]


def _model(variant, flags, extra):
    from pangnn_b200.gnn import AlternateGCN
    from oracle.params import make_state_dict
    for k, v in dict(VARIANT_FLAGS[variant], **extra).items():
        setattr(flags, k, v)
    m = AlternateGCN(DEV, None, False, dims=[flags.node_dim, flags.hidden_dim])
    m.load_state_dict(make_state_dict(flags.node_dim, flags.hidden_dim, flags.skip_connections, seed=1234), strict=True)
    return m.to(DEV)


def _split_of(graph):
    from pangnn_b200.edge_split import EdgeSplit
    return EdgeSplit.build(*graph.edge_index, graph.y, 1, (0.15, 0.15))


@pytest.mark.parametrize("case,variant,extra", MODEL_CASES, ids=[f"{c}-{v}{'-' + str(e) if e else ''}"
                                                                 for c, v, e in MODEL_CASES])
def test_forward_loss_train_labels_match_oracle(golden, flags, case, variant, extra):
    from pangnn_b200.edge_split import TRAIN
    g = golden(case)
    model = _model(variant, flags, extra)
    graph = golden_graph(g, variant, device=DEV)
    sp = _split_of(graph)
    ytr, n = sp.labels(graph.y, TRAIN), sp.count(TRAIN)
    loss, logits = model.forward_loss(graph, sp.class_balance, y=ytr, num_labelled=n)
    loss.backward()
    om, _ = oracle_model(variant, **extra)
    og = golden_graph(g, variant)
    z = om(og)
    keep = (ytr >= 0).cpu()
    lo = torch.nn.functional.binary_cross_entropy_with_logits(
        z[keep], og.y[keep], pos_weight=torch.tensor(sp.class_balance), reduction="sum") / n
    lo.backward()
    assert abs(loss.item() - lo.item()) <= TOL * abs(lo.item())
    assert_close("logits", logits.cpu().numpy(), z.detach().numpy(), TOL)
    ref = dict(om.named_parameters())
    for name, p in model.named_parameters():
        q = ref[name]
        if q.grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert_close(f"grad {name}", p.grad.cpu().numpy(), q.grad.numpy(), GRAD_TOL)


@pytest.mark.parametrize("case,variant", [("c1", "default"), ("c2", "union_skip")])
def test_library_operator_layer_bit_identical(golden, flags, case, variant):
    from pangnn_b200 import gnn, ops
    from pangnn_b200.edge_split import TRAIN
    g = golden(case)
    out = []
    for kind in ("function", "library"):
        gnn.set_operator_layer(kind)
        ops.clear_cache()
        model = _model(variant, flags, {})
        model.fuse_embedding = False                      # the same composition in both spellings
        graph = golden_graph(g, variant, device=DEV)
        sp = _split_of(graph)
        loss, logits = model.forward_loss(graph, sp.class_balance, y=sp.labels(graph.y, TRAIN),
                                          num_labelled=sp.count(TRAIN))
        loss.backward()
        out.append([loss.item(), logits] + [p.grad for p in model.parameters()])
    assert out[0][0] == out[1][0]
    for a, b in zip(out[0][1:], out[1][1:]):
        assert (a is None and b is None) or torch.equal(a, b)


# ------------------------------------------------------------------------------------------------
# CLI
# ------------------------------------------------------------------------------------------------
SIM = ["--simulate_dataset", "300", "4", "0.5", "10", "3", "--seed", "1"]
SPLIT = ["--edge_split", "0.15", "0.15"]
TRAIN_FLAGS = ["--train", "--whole_graph_training", "-e", "3"]
UNION = ["--union_edge_weights", "--neighbours", "3", "--skip_connections"]
STAT_KEYS = ("tn", "fp", "fn", "tp", "precision", "recall", "f1", "loss", "auroc", "average_precision",
             "youden_threshold")


def _run(argv, device=DEV):
    from pangnn_b200 import ops, setup, train
    setup.reset()
    ops.clear_cache()
    try:
        return train.run(setup.parse(argv), device=device)
    finally:
        setup.reset()
        ops.clear_cache()


def _dirs(tmp, name, model=None):
    return ["-o", os.path.join(tmp, name), "-m", model or os.path.join(tmp, "model.pkl")]


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _summary(res):
    t = res["test"][0]
    ids = t["edge_ids"] if "edge_ids" in t else torch.arange(t["logits"].numel())
    return dict(edge_ids=ids.cpu().numpy(), logits=t["logits"].float().cpu().numpy(),
                prob=t["prob"].float().cpu().numpy(), pred=t["pred"].cpu().numpy().astype(np.int64),
                stats=np.array([np.nan if t[k] is None else t[k] for k in STAT_KEYS], dtype=np.float64),
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


def _check_one_gpu(res, out_dir):
    from pangnn_b200 import train
    from pangnn_b200.edge_split import TEST, VAL, EdgeSplit
    whole = res["test"][0]
    g = res["dataset"].test[0]
    sp = EdgeSplit.build(*g.edge_index, g.y, 1, (0.15, 0.15))
    for h in res["history"]:
        assert sum(h["val_confusion"]) == sp.count(VAL)
    t = res["test"][0]
    assert t["tn"] + t["fp"] + t["fn"] + t["tp"] == sp.count(TEST)
    assert torch.equal(t["sel"], sp.codes == TEST)
    assert t["logits"].numel() == g.edge_index.size(1)          # predictions of every edge
    # curve files: the one-GPU writer over the test edges
    sel = sp.codes == TEST
    check = os.path.join(out_dir, "curves_check")
    train.write_curves(SimpleNamespace(y=g.y[sel]), {"prob": whole["prob"][sel]}, check)
    for f in ("roc_curve.csv", "precision_recall_curve.csv"):
        assert _read(os.path.join(out_dir, f)) == _read(os.path.join(check, f)), f
    return sp


@pytest.mark.parametrize("extra", [[], UNION], ids=["default", "union_skip"])
def test_cli_one_gpu_inference_and_world1_group(extra):
    with tempfile.TemporaryDirectory() as tmp:
        ref = _run(SIM + SPLIT + TRAIN_FLAGS + extra + _dirs(tmp, "ref"))
        ref_dir = os.path.join(tmp, "ref")
        _check_one_gpu(ref, ref_dir)
        r = _summary(ref)
        # inference from the saved model.pkl: the same test statistics and output files
        model = os.path.join(ref_dir, "model.pkl")
        inf = _run(SIM + SPLIT + extra + _dirs(tmp, "infer", model))
        i = _summary(inf)
        assert np.array_equal(i["stats"], r["stats"], equal_nan=True)
        for f in ("holiest_of_all_tables.csv", "q_score_vs_logit.csv", "roc_curve.csv", "precision_recall_curve.csv"):
            assert _read(os.path.join(tmp, "infer", f)) == _read(os.path.join(ref_dir, f)), f
        # an NCCL group of one rank: the partitioned driver
        _worker(0, 1, os.path.join(tmp, "rdv"), [SIM + SPLIT + TRAIN_FLAGS + extra + _dirs(tmp, "part")], tmp)
        o = dict(np.load(os.path.join(tmp, "run0_r0.npz")))
        _compare(ref, ref_dir, [o], os.path.join(tmp, "part"), tmp)


def _compare(ref, ref_dir, outs, out_dir, tmp):
    import pandas as pd
    from pangnn_b200 import train
    from pangnn_b200.edge_split import TEST, EdgeSplit
    r = _summary(ref)
    for k in ("train_loss", "val_loss"):
        for o in outs:
            assert np.array_equal(o[k], outs[0][k])
        assert np.all(np.abs(outs[0][k] - r[k]) <= TOL * np.abs(r[k])), k
    a = torch.load(os.path.join(ref_dir, "model.pkl"), map_location="cpu")
    b = torch.load(os.path.join(out_dir, "model.pkl"), map_location="cpu")
    assert list(a) == list(b)
    for k in a:
        assert float((a[k] - b[k]).abs().max()) <= 2e-5 * max(float(a[k].abs().max()), 1e-3), k
    ids = np.concatenate([o["edge_ids"] for o in outs])
    assert np.array_equal(np.sort(ids), np.arange(ids.size))
    whole = {k: np.empty(ids.size, dtype=outs[0][k].dtype) for k in ("logits", "prob", "pred")}
    for o in outs:
        for k in whole:
            whole[k][o["edge_ids"]] = o[k]
    assert rel_err(whole["logits"], r["logits"]) < TOL
    clear = np.abs(r["prob"] - 0.5) > 1e-5
    assert np.array_equal(whole["pred"][clear], r["pred"][clear])
    # test statistics: the counts of the same edges; the rates and ranking metrics to the tolerance
    for o in outs:
        assert np.array_equal(o["stats"], outs[0]["stats"], equal_nan=True)
    s = outs[0]["stats"]
    assert s[:4].sum() == r["stats"][:4].sum()
    assert np.all(np.abs(s[4:] - r["stats"][4:]) <= 1e-3 * np.maximum(np.abs(r["stats"][4:]), 1)), (s, r["stats"])
    # curve files: the one-GPU writer over the test edges of the run's own probabilities
    g = ref["dataset"].test[0]
    sel = (EdgeSplit.build(*g.edge_index, g.y, 1, (0.15, 0.15)).codes == TEST).cpu().numpy()
    check = os.path.join(tmp, "curves_check_part")
    train.write_curves(SimpleNamespace(y=g.y[torch.from_numpy(sel).to(g.y.device)]),
                       {"prob": torch.from_numpy(whole["prob"][sel]).to(g.y.device)}, check)
    for f in ("roc_curve.csv", "precision_recall_curve.csv"):
        assert _read(os.path.join(out_dir, f)) == _read(os.path.join(check, f)), f
    ta, tb = (pd.read_csv(os.path.join(d, "q_score_vs_logit.csv")) for d in (ref_dir, out_dir))
    assert list(ta.columns) == list(tb.columns) and len(ta) == len(tb)
    for c in ta.columns:
        if c == "logit":
            assert rel_err(tb[c].to_numpy(), ta[c].to_numpy()) < TOL
        else:
            assert np.array_equal(ta[c].to_numpy(), tb[c].to_numpy()), c
    if np.array_equal(whole["pred"], r["pred"]):
        f = "holiest_of_all_tables.csv"
        assert _read(os.path.join(out_dir, f)) == _read(os.path.join(ref_dir, f))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_cli_world2_matches_one_gpu():
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        ref = _run(SIM + SPLIT + TRAIN_FLAGS + _dirs(tmp, "ref"))
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdv"), [SIM + SPLIT + TRAIN_FLAGS + _dirs(tmp, "w2")], tmp),
                 nprocs=2, join=True)
        outs = [dict(np.load(os.path.join(tmp, f"run0_r{r}.npz"))) for r in range(2)]
        _compare(ref, os.path.join(tmp, "ref"), outs, os.path.join(tmp, "w2"), tmp)
