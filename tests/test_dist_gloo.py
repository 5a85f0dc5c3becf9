"""Host logic of the genome-partitioned multi-GPU path (pangnn_b200/dist.py) on CPU: world_size 2
and 3 over the gloo backend.

The partition algebra — local "own + halo" numbering, halo plans, the grouped exchange and its
transposed backward, gcn_norm across the cut, the global-mean loss and the weight-gradient
all-reduce — is exercised through ``DistModel`` itself; only the CUDA kernels underneath are
replaced by torch-CPU stand-ins defined HERE (test infrastructure; the product has no CPU path).
The result must equal the whole-graph oracle model on the same golden graph.
"""
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.helpers import VARIANT_FLAGS, golden_graph, oracle_model, rel_err
from tests.conftest import load_golden


# ------------------------------------------------------------------------------------------------
# torch-CPU stand-ins for the kernels DistModel calls (same signatures as pangnn_b200.ops)
# ------------------------------------------------------------------------------------------------
class _CpuStruct:
    def __init__(self, edge_index, num_nodes):
        self.edge_index, self.num_nodes, self.num_edges = edge_index, num_nodes, edge_index.size(1)
        self.dst = SimpleNamespace(ei=edge_index, by_dst=True, num_rows=num_nodes)
        self.src = SimpleNamespace(ei=edge_index, by_dst=False, num_rows=num_nodes)


def _cpu_gcn_norm(csr_dst, w):
    ei = csr_dst.ei
    w = torch.ones(ei.size(1)) if w is None else w.float()
    deg = torch.zeros(csr_dst.num_rows).scatter_add_(0, ei[1], w)
    dis = deg.pow(-0.5)
    dis[dis == float("inf")] = 0
    return dis, None


def _cpu_gcn_norm_apply(csr, w, dis):
    ei = csr.ei
    w = torch.ones(ei.size(1)) if w is None else w.float()
    return dis[ei[0]] * w * dis[ei[1]]                      # original edge order in this stand-in


class _CpuAggregate:
    @staticmethod
    def apply(x_ext, bias, csr_dst, val_dst, csr_src, val_src, n_out, act, dx_out=None):
        ei = csr_dst.ei
        out = torch.zeros(n_out, x_ext.size(1)).index_add_(0, ei[1], val_dst.unsqueeze(1) * x_ext[ei[0]])
        if bias is not None:
            out = out + bias
        return torch.nn.functional.elu(out) if act == 1 else out


class _CpuScorer:
    @staticmethod
    def apply(pq, w1c, b1, w2, b2, w3, b3, gs, skip, y, pos_weight, scale, dpq_out=None, unit_grad=False):
        D = 64
        s, d = gs.edge_index[0], gs.edge_index[1]
        a1 = pq[s, :D] + pq[d, D:] + b1
        if skip is not None:
            a1 = a1 + skip.unsqueeze(1) * w1c
        r2 = torch.relu(torch.relu(a1) @ w2.t() + b2)
        z = (r2 @ w3.t()).squeeze(1) + b3
        loss = torch.nn.functional.binary_cross_entropy_with_logits(
            z, y, pos_weight=torch.tensor(float(pos_weight)), reduction="sum")
        return loss * scale, z.detach()


def _cpu_linear(x, weight, bias=None, act=0, extra_rows=0, out_full=None, push=None):
    y = x @ weight.t()
    if bias is not None:
        y = y + bias
    y = torch.nn.functional.elu(y) if act == 1 else y
    if extra_rows:                                           # room for the halo rows (HaloFill)
        y = torch.cat((y, torch.zeros(extra_rows, y.size(1))), dim=0)
    return y


def _cpu_rank1_vectors(csr_dst, val_dst, x, num_rows=None):
    ei, n = csr_dst.ei, csr_dst.num_rows
    xs = x.reshape(-1).float()
    a = torch.zeros(n).index_add_(0, ei[1], val_dst * xs[ei[0]])
    c = torch.zeros(n).index_add_(0, ei[1], val_dst)
    k = n if num_rows is None else num_rows
    return a[:k], c[:k]


class _CpuRankOne:
    @staticmethod
    def apply(a, c, w_e, b_e, weight, bias, act):
        y = a.unsqueeze(1) * (weight @ w_e.reshape(-1)) + c.unsqueeze(1) * (weight @ b_e)
        if bias is not None:
            y = y + bias
        return torch.nn.functional.elu(y) if act == 1 else y


def _patch(ops):
    ops.rank1_vectors = _cpu_rank1_vectors
    ops.RankOneFn = _CpuRankOne
    ops.linear = _cpu_linear
    ops.GraphStruct = _CpuStruct
    ops.gcn_norm = _cpu_gcn_norm
    ops.gcn_norm_apply = _cpu_gcn_norm_apply
    ops.AggregateFn = _CpuAggregate
    ops.EdgeScoreBCEPQFn = _CpuScorer


# ------------------------------------------------------------------------------------------------
def _worker(rank, world, init_file, case, variant, fuse_embedding, out_dir):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        from pangnn_b200 import dist as pd, ops, setup
        from pangnn_b200.gnn import AlternateGCN
        from oracle.params import make_state_dict
        _patch(ops)
        setup.reset()
        for k, v in VARIANT_FLAGS[variant].items():
            setattr(setup.args, k, v)
        fl = setup.args
        g = load_golden(case)
        graph = golden_graph(g, variant)
        N = graph.x.size(0)
        model = AlternateGCN("cpu", None, False, dims=[fl.node_dim, fl.hidden_dim])
        model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
        model.fuse_embedding = fuse_embedding
        pgraph = pd.PartitionedGraph.from_global(graph, N, rank, world)
        dm = pd.DistModel(model)
        pw = float(g[f"model/{variant}/pos_weight"])
        loss, logits = dm.forward_loss(pgraph, pw)
        loss.backward()
        dm.allreduce_grads()
        total = loss.detach().clone().double()
        dist.all_reduce(total)
        grads = {k: p.grad.numpy() for k, p in model.named_parameters() if p.grad is not None}
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), loss=total.numpy(), logits=logits.numpy(),
                 edge_ids=pgraph.scored_edge_ids.numpy(), class_balance=pgraph.class_balance,
                 n_halo=np.array([pgraph.conv.plan.n_halo, pgraph.scored.plan.n_halo]),
                 **{f"grad/{k}": v for k, v in grads.items()})
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case,variant,fuse_embedding", [
    pytest.param(case, variant, fuse, id=f"{case}-{variant}" + ("" if fuse else "-unfused"))
    for fuse in (True, False)
    for case, variant in [("sim5", "default"), ("sim5", "union_skip"), ("c1", "base"), ("c1", "union_n4")]])
def test_partitioned_model_equals_whole_graph(case, variant, fuse_embedding, world):
    g = load_golden(case)
    with tempfile.TemporaryDirectory() as tmp:
        init_file = os.path.join(tmp, "rendezvous")
        mp.spawn(_worker, args=(world, init_file, case, variant, fuse_embedding, tmp), nprocs=world, join=True)
        outs = [np.load(os.path.join(tmp, f"r{r}.npz")) for r in range(world)]
    key = f"model/{variant}"
    ref_logits, ref_loss = g[f"{key}/logits"], float(g[f"{key}/loss"])
    # every scored edge is owned by exactly one rank (the owner of its source)
    ids = np.concatenate([o["edge_ids"] for o in outs])
    assert np.array_equal(np.sort(ids), np.arange(ref_logits.size))
    got = np.empty_like(ref_logits)
    for o in outs:
        got[o["edge_ids"]] = o["logits"]
    assert rel_err(got, ref_logits) < 1e-5
    for o in outs:                                           # same global loss / class balance everywhere
        assert abs(float(o["loss"]) - ref_loss) <= 1e-5 * abs(ref_loss)
        assert abs(float(o["class_balance"]) - float(g[f"{key}/pos_weight"])) < 1e-6 * float(g[f"{key}/pos_weight"])
    for k in [f for f in g.files if f.startswith(f"{key}/grad/")]:
        name = k[len(f"{key}/grad/"):]
        for o in outs:                                       # all-reduced: identical on every rank
            assert rel_err(o[f"grad/{name}"], g[k]) < 1e-4, name


def test_local_numbering_and_bounds():
    from pangnn_b200.dist import balanced_bounds, local_numbering
    assert balanced_bounds(100, 4, 25) == [0, 25, 50, 75, 100]
    assert balanced_bounds(100, 8, 5)[-1] == 100 and len(balanced_bounds(100, 8, 5)) == 9   # 20 genomes / 8
    b = balanced_bounds(4_000_000, 8, 200_000)
    assert all(b[i] < b[i + 1] for i in range(8))
    ei = torch.tensor([[0, 5, 7, 9, 2, 5], [4, 4, 5, 0, 6, 9]])
    keep, halo, loc = local_numbering(ei, 4, 8, "dst")
    assert keep.tolist() == [True, True, True, False, True, False]
    assert halo.tolist() == [0, 2]                           # sorted remote sources
    # own ids -> id - lo ; halo ids -> n_own + rank in halo list
    assert loc.tolist() == [[4, 1, 3, 5], [0, 0, 1, 2]]
    keep, halo, loc = local_numbering(ei, 4, 8, "src")
    assert keep.tolist() == [False, True, True, False, False, True]
    assert halo.tolist() == [9]
    assert loc.tolist() == [[1, 3, 1], [0, 1, 4]]
    keep, halo, loc = local_numbering(ei[:, :0], 0, 4, "dst")           # empty edge set
    assert halo.numel() == 0 and loc.shape == (2, 0)


def test_simulator_slabs_agree_with_the_whole_table():
    """A rank generates only the hits whose QUERY lies in its genomes (+ one boundary genome per
    side); those rows must be exactly the corresponding rows of the full table, so that two ranks
    agree on every edge that crosses their seam."""
    from pangnn_b200.simulate import simulate_hits
    n, G = 60, 6
    full = simulate_hits(n, G, 0.5, 10, 3, seed=7)
    genome_q = full["q"] // n
    for lo, hi in [(0, 2), (1, 4), (3, 6), (-1, 3), (4, 7)]:
        part = simulate_hits(n, G, 0.5, 10, 3, seed=7, genomes=(lo, hi))
        m = (genome_q >= lo) & (genome_q < hi)
        ref = np.stack((full["q"][m], full["t"][m], full["bits"][m]))
        got = np.stack((part["q"], part["t"], part["bits"]))
        assert got.shape == ref.shape
        o1, o2 = np.lexsort(ref[::-1]), np.lexsort(got[::-1])
        assert np.array_equal(ref[:, o1], got[:, o2])
        assert np.array_equal(part["group_of"], full["group_of"])
    # adjacent_only drops nothing that survives the default trivial-case filter
    from oracle import preprocess as op
    adj = simulate_hits(n, G, 0.5, 10, 3, seed=7, adjacent_only=True)
    outs = []
    for s in (full, adj):
        q, t, b = op.dedupe_last(s["q"].astype(np.int64), s["t"].astype(np.int64), s["bits"])
        q, t, b = op.remove_trivial_cases(q, t, b, s["genome_of"])
        outs.append(op.normalize_sim_scores(q, t, b, s["genome_of"]))
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


def _worker_categorical(rank, world, init_file, out_dir):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        from pangnn_b200 import dist as pd, ops, setup
        from pangnn_b200.gnn import AlternateGCN
        _patch(ops)
        setup.reset()
        g = load_golden("sim5")
        graph = golden_graph(g, "default")
        N = graph.x.size(0)
        torch.manual_seed(5)                                  # same initial replica on every rank
        model = AlternateGCN("cpu", N, True, dims=[64, 128])
        init = model.embedding.weight.detach().clone()
        pgraph = pd.PartitionedGraph.from_global(graph, N, rank, world)
        dm = pd.DistModel(model)
        loss, _ = dm.forward_loss(pgraph, 2.0)
        loss.backward()
        if rank == 1:                                         # a rank that lacks a gradient the others have
            model.mlp[4].bias.grad = None
        dm.allreduce_grads()
        with torch.no_grad():
            model.embedding.weight -= 0.5 * model.embedding.weight.grad      # only the owned rows move
        sd = dm.state_dict(pgraph.bounds)
        np.savez(os.path.join(out_dir, f"c{rank}.npz"), table=sd["embedding.weight"].numpy(), init=init.numpy(),
                 bounds=np.asarray(pgraph.bounds),
                 **{f"grad/{k}": p.grad.numpy() for k, p in model.named_parameters()
                    if p.grad is not None and k != "embedding.weight"})
    finally:
        dist.destroy_process_group()


def test_categorical_table_is_gathered_and_bucket_layout_is_rank_independent():
    """ADVICE r1: (1) with --categorical_node every rank trains only its own rows of the embedding table, so the
    checkpoint has to gather the row blocks; (2) the all-reduce bucket must not depend on which gradients
    happen to exist on a rank."""
    world = 2
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker_categorical, args=(world, os.path.join(tmp, "rendezvous"), tmp), nprocs=world, join=True)
        outs = [np.load(os.path.join(tmp, f"c{r}.npz")) for r in range(world)]
    assert np.array_equal(outs[0]["table"], outs[1]["table"])             # complete and identical everywhere
    b = outs[0]["bounds"]
    for r in range(world):                                                # every rank's block was trained
        blk = slice(int(b[r]), int(b[r + 1]))
        assert np.abs(outs[0]["table"][blk] - outs[0]["init"][blk]).max() > 0
    keys = sorted(k for k in outs[0].files if k.startswith("grad/"))
    assert keys == sorted(k for k in outs[1].files if k.startswith("grad/")) and "grad/mlp.4.bias" in keys
    for k in keys:
        assert np.array_equal(outs[0][k], outs[1][k]), k
