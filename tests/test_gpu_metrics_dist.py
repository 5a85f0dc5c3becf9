"""Exact global ranking metrics over two GPUs (NCCL; skipped with fewer): ``metrics.ranking_metrics`` on per-rank
slices and ``DistModel.evaluate`` on the golden graphs, against the single-GPU results."""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle.params import make_state_dict
from tests.conftest import load_golden
from tests.helpers import VARIANT_FLAGS, golden_graph

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")]

CASES = [("sim5", "default"), ("c1", "base"), ("c2", "union_skip")]


def _slices():
    """400 000 scores with heavy ties and a saturated tail at 1.0f; rank 0 gets the first third, rank 1 the rest."""
    rng = np.random.default_rng(5)
    E = 400_000
    y = (rng.random(E) < 0.04).astype(np.float32)
    s = (np.round(rng.random(E) * 200) / 200 + 0.2 * y).astype(np.float32)
    s[rng.random(E) < 0.01] = 1.0
    return s, y, [(s[:E // 3], y[:E // 3]), (s[E // 3:], y[E // 3:])]


def _worker(rank, world, init_file, out_dir):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    try:
        from pangnn_b200 import dist as pd, ops, setup
        from pangnn_b200.gnn import AlternateGCN
        from pangnn_b200.metrics import ranking_metrics
        _, _, parts = _slices()
        s, y = parts[rank]
        res = {"slices": ranking_metrics(torch.from_numpy(s).to(dev), torch.from_numpy(y).to(dev))}
        e = torch.zeros(0, device=dev)
        res["empty_rank"] = ranking_metrics(torch.from_numpy(s).to(dev) if rank else e,
                                            torch.from_numpy(y).to(dev) if rank else e)
        for case, variant in CASES:
            setup.reset()
            ops.clear_cache()
            for k, v in VARIANT_FLAGS[variant].items():
                setattr(setup.args, k, v)
            fl = setup.args
            g = load_golden(case)
            graph = golden_graph(g, variant, device=dev)
            model = AlternateGCN(dev, None, False, dims=[fl.node_dim, fl.hidden_dim])
            model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
            model = model.to(dev)
            pg = pd.PartitionedGraph.from_global(graph, graph.x.size(0), rank, world)
            rec = pd.DistModel(model).evaluate(pg, 0.5, float(g[f"model/{variant}/pos_weight"]))
            res[case] = {k: rec[k] for k in ("tn", "fp", "fn", "tp", "precision", "recall", "f1", "loss", "auroc",
                                             "average_precision", "youden_threshold")}
            res[case]["prob"] = rec["prob"].cpu()
            res[case]["edge_ids"] = pg.scored_edge_ids.cpu()
        torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_ranks():
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdv"), tmp), nprocs=2, join=True)
        yield [torch.load(os.path.join(tmp, f"r{r}.pt")) for r in range(2)]


def test_slices_equal_world1_on_the_concatenation(two_ranks):
    from pangnn_b200.metrics import ranking_metrics
    s, y, _ = _slices()
    ref = ranking_metrics(torch.from_numpy(s).cuda(), torch.from_numpy(y).cuda())
    for r in two_ranks:
        assert r["slices"] == ref
        assert r["empty_rank"] == ranking_metrics(torch.from_numpy(s[len(s) // 3:]).cuda(),
                                                  torch.from_numpy(y[len(y) // 3:]).cuda())


@pytest.mark.parametrize("case,variant", CASES)
def test_dist_evaluate_equals_single_gpu_evaluate(two_ranks, case, variant):
    from pangnn_b200 import ops, setup, train
    from pangnn_b200.gnn import AlternateGCN
    from pangnn_b200.metrics import ranking_metrics
    setup.reset()
    ops.clear_cache()
    for k, v in VARIANT_FLAGS[variant].items():
        setattr(setup.args, k, v)
    fl = setup.args
    g = load_golden(case)
    graph = golden_graph(g, variant, device="cuda:0")
    model = AlternateGCN("cuda:0", None, False, dims=[fl.node_dim, fl.hidden_dim])
    model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
    model = model.to("cuda:0")
    pw = float(g[f"model/{variant}/pos_weight"])
    ref = train.evaluate(model, [graph], 0.5, pw)[0]
    outs = [r[case] for r in two_ranks]
    # the world-2 probabilities, reassembled in global edge order
    prob = torch.empty_like(ref["prob"]).cpu()
    for o in outs:
        prob[o["edge_ids"]] = o["prob"]
    same_prob = torch.equal(prob, ref["prob"].cpu())
    glob = ranking_metrics(prob.cuda(), graph.y)
    for o in outs:
        for k in ("auroc", "average_precision", "youden_threshold"):
            assert o[k] == glob[k], k                                   # exact global metrics of the world-2 probs
            if same_prob:
                assert o[k] == ref[k], k
        if same_prob:
            assert (o["tn"], o["fp"], o["fn"], o["tp"]) == (ref["tn"], ref["fp"], ref["fn"], ref["tp"])
        assert o["tn"] + o["fp"] + o["fn"] + o["tp"] == graph.y.numel()
        assert abs(o["loss"] - ref["loss"]) <= 1e-6 * abs(ref["loss"])
        assert all(o[k] == outs[0][k] for k in ("tn", "fp", "fn", "tp", "loss", "auroc", "average_precision",
                                                "youden_threshold"))
