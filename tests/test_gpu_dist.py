"""GPU parity of the genome-partitioned path (pangnn_b200/dist.py) through the C ABI.

* world 1 (any box): ``DistModel`` on one partition that owns everything must reproduce the golden
  logits / loss / gradients — this runs the local-numbering, ``AggregateFn`` and pq-scorer kernels.
* world 2 over NCCL (needs 2 GPUs; skipped otherwise): two ranks, halo exchange per layer.
* ``from_simulation``: the partition-local build equals the slice of the whole-graph build.
"""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle.params import make_state_dict
from tests.conftest import load_golden
from tests.helpers import GRAD_TOL, VARIANT_FLAGS, golden_graph, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _setup(variant):
    from pangnn_b200 import ops, setup
    setup.reset()
    ops.clear_cache()
    for k, v in VARIANT_FLAGS[variant].items():
        setattr(setup.args, k, v)
    return setup.args


def _run_rank(rank, world, case, variant, dev, group=None):
    from pangnn_b200 import dist as pd
    from pangnn_b200.gnn import AlternateGCN
    fl = _setup(variant)
    g = load_golden(case)
    graph = golden_graph(g, variant, device=dev)
    model = AlternateGCN(dev, None, False, dims=[fl.node_dim, fl.hidden_dim])
    model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
    model = model.to(dev)
    pg = pd.PartitionedGraph.from_global(graph, graph.x.size(0), rank, world, group=group)
    dm = pd.DistModel(model, group)
    pw = float(g[f"model/{variant}/pos_weight"])
    loss, logits = dm.forward_loss(pg, pw)
    loss.backward()
    dm.allreduce_grads()
    infer = dm(pg)
    out = dict(loss=loss.detach().double().cpu().numpy(), logits=logits.cpu().numpy(), infer=infer.cpu().numpy(),
               edge_ids=pg.scored_edge_ids.cpu().numpy(), class_balance=pg.class_balance)
    out.update({f"grad/{k}": p.grad.cpu().numpy() for k, p in model.named_parameters() if p.grad is not None})
    return out


def _check(outs, case, variant, loss_is_partial):
    g = load_golden(case)
    key = f"model/{variant}"
    ref_logits, ref_loss = g[f"{key}/logits"], float(g[f"{key}/loss"])
    ids = np.concatenate([o["edge_ids"] for o in outs])
    assert np.array_equal(np.sort(ids), np.arange(ref_logits.size))
    got, got_inf = np.empty_like(ref_logits), np.empty_like(ref_logits)
    for o in outs:
        got[o["edge_ids"]] = o["logits"]
        got_inf[o["edge_ids"]] = o["infer"]
    assert rel_err(got, ref_logits) < TOL
    assert rel_err(got_inf, ref_logits) < TOL
    total = sum(float(o["loss"]) for o in outs) if loss_is_partial else float(outs[0]["loss"])
    assert abs(total - ref_loss) <= TOL * abs(ref_loss)
    for k in [f for f in g.files if f.startswith(f"{key}/grad/")]:
        name = k[len(f"{key}/grad/"):]
        for o in outs:
            assert rel_err(o[f"grad/{name}"], g[k]) < GRAD_TOL, name


CASES = [("sim5", "default"), ("sim5", "union_skip"), ("c1", "base"), ("c1", "union_n4"), ("c2", "union_skip")]


@pytest.mark.parametrize("case,variant", CASES)
def test_single_partition_matches_golden(case, variant):
    _check([_run_rank(0, 1, case, variant, "cuda:0")], case, variant, True)


def _nccl_worker(rank, world, init_file, case, variant, out_dir, p2p="1"):
    import torch.distributed as dist
    os.environ["PANGNN_P2P"] = p2p                           # halo transport: NVLink peer memory (default) or NCCL
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    try:
        out = _run_rank(rank, world, case, variant, dev)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **out)
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("case,variant", CASES)
@pytest.mark.parametrize("p2p", ["1", "0"])
def test_two_partitions_match_golden_nccl(case, variant, p2p):
    """world 2, both halo transports: NVLink peer memory (fused GEMM-epilogue push) and NCCL send/recv."""
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_nccl_worker, args=(2, os.path.join(tmp, "rdv"), case, variant, tmp, p2p), nprocs=2, join=True)
        outs = [dict(np.load(os.path.join(tmp, f"r{r}.npz"))) for r in range(2)]
    _check(outs, case, variant, True)


@pytest.mark.parametrize("union", [False, True])
def test_from_simulation_equals_whole_graph_slice(union):
    """Each rank builds its slab alone (world emulated rank by rank on one device, no collectives:
    plans are not needed to compare graphs)."""
    from pangnn_b200 import dist as pd, ops, setup, preprocessing as pp
    from pangnn_b200.simulate import simulate_hits
    fl = _setup("union_skip" if union else "default")
    n, G, world = 300, 6, 3
    s = simulate_hits(n, G, 0.5, 10, 3, seed=3)
    src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"],
                                             num_nodes=n * G, device="cuda:0")
    seen = 0
    for rank in range(world):
        # world=1 plan construction per slab: emulate by building the local pieces directly
        lo, hi = rank * (G // world) * n, (rank + 1) * (G // world) * n
        part = simulate_hits(n, G, 0.5, 10, 3, seed=3, genomes=(lo // n - 1, hi // n + 1), adjacent_only=True)
        ps, pdst, pw_, py = pp.normalize_sim_scores(part["q"], part["t"], part["bits"], part["genome_of"],
                                                    part["group_of"], num_nodes=n * G, device="cuda:0")
        own_src = (src >= lo) & (src < hi)
        m = (ps >= lo) & (ps < hi)
        assert torch.equal(ps[m], src[own_src]) and torch.equal(pdst[m], dst[own_src])
        assert torch.equal(pw_[m], w[own_src]) and torch.equal(py[m], y[own_src])
        own_dst = (dst >= lo) & (dst < hi)
        m2 = (pdst >= lo) & (pdst < hi)
        assert torch.equal(ps[m2], src[own_dst]) and torch.equal(pw_[m2], w[own_dst])
        seen += int(m.sum())
    assert seen == src.numel()


@pytest.mark.parametrize("variant", ["default", "union_skip"])
def test_from_simulation_world1_equals_public_api(variant):
    """The partition-local builder + DistModel on one rank == dataset-style assembly + AlternateGCN."""
    from pangnn_b200 import dist as pd, preprocessing as pp
    from pangnn_b200.data import Data
    from pangnn_b200.gnn import AlternateGCN
    from pangnn_b200.simulate import simulate_hits
    fl = _setup(variant)
    dev = "cuda:0"
    n, G = 400, 4
    pg = pd.PartitionedGraph.from_simulation(n, G, 0.5, 10, 3, 0, 1, dev, seed=5)
    s = simulate_hits(n, G, 0.5, 10, 3, seed=5)
    src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"],
                                             num_nodes=n * G, device=dev)
    ei = torch.stack((src.long(), dst.long()))
    assert torch.equal(pg.scored.edge_index, ei) and torch.equal(pg.y, y)
    nb = pp.neighbour_band(n * G, fl.neighbours, dev)
    x = torch.ones(n * G, 1, device=dev)
    if fl.union_edge_weights:
        graph = Data(x, ei, torch.cat((w, torch.ones(nb.size(1), device=dev))), y)
        graph.union_edge_index = torch.cat((ei, nb), dim=1)
    else:
        graph = Data(x, ei, w, y)
        graph.neighbour_edge_index = nb
    model = AlternateGCN(dev, None, False).to(dev)
    model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
    pw = float(((y == 0).sum() / y.sum()).item())
    assert abs(pg.class_balance - pw) < 1e-6 * pw
    loss_ref, logits_ref = model.forward_loss(graph, pw)
    loss_ref.backward()
    ref_grads = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    model.zero_grad(set_to_none=True)
    loss, logits = pd.DistModel(model).forward_loss(pg, pw)
    loss.backward()
    assert rel_err(logits.cpu().numpy(), logits_ref.cpu().numpy()) < TOL
    assert abs(loss.item() - loss_ref.item()) <= TOL * abs(loss_ref.item())
    for k, p in model.named_parameters():
        if k in ref_grads:
            assert rel_err(p.grad.cpu().numpy(), ref_grads[k].cpu().numpy()) < GRAD_TOL, k
    # host round trip used by bench.py's end-to-end leg
    pg2 = pg.rebuilt_from(pg.to_host_pinned(), dev)
    loss2, logits2 = pd.DistModel(model).forward_loss(pg2, pw)
    assert torch.equal(logits2, logits)


@pytest.mark.parametrize("variant", ["union_skip", "default"])
def test_prefetched_partition_batches_repeat_the_step(variant):
    """PartitionedGraph.prefetch_from: the next batch is copied from pinned host memory and its CSRs are built on
    side streams while the current step runs; every step must be bit-identical to the resident partition's."""
    from pangnn_b200 import dist as pd
    from pangnn_b200.gnn import AlternateGCN
    dev = "cuda:0"
    fl = _setup(variant)
    g = load_golden("c2")
    graph = golden_graph(g, variant, device=dev)
    model = AlternateGCN(dev, None, False, dims=[fl.node_dim, fl.hidden_dim])
    model.load_state_dict(make_state_dict(fl.node_dim, fl.hidden_dim, fl.skip_connections, seed=1234))
    model = model.to(dev)
    pg = pd.PartitionedGraph.from_global(graph, graph.x.size(0), 0, 1)
    dm = pd.DistModel(model)
    pw = float(g[f"model/{variant}/pos_weight"])
    loss0, logits0 = dm.forward_loss(pg, pw)
    host = pg.to_host_pinned()
    main = torch.cuda.current_stream()
    pending = pg.prefetch_from(host, dev, main)
    for i in range(5):
        b, ev = pending
        main.wait_event(ev)
        model.zero_grad()
        loss, logits = dm.forward_loss(b, pw)
        loss.backward()
        pending = pg.prefetch_from(host, dev, main) if i < 4 else None
        assert loss.item() == loss0.item() and torch.equal(logits, logits0)


@pytest.mark.parametrize("union", [False, True])
def test_from_simulation_device_generator_slab_by_slab(union):
    """``from_simulation(device_generator=True)`` generates and normalises one query genome at a time: the table must be
    the one a single pass over all genomes gives (Philox streams are keyed by genome / gene / draw; the candidate sets
    of a query are complete inside its genome's slab) — scored edges, weights, labels bit for bit."""
    from pangnn_b200 import dist as pd, preprocessing as pp
    from pangnn_b200.simulate import simulate_hits_device
    fl = _setup("union_skip" if union else "default")
    dev = torch.device("cuda:0")
    n, G, f = 700, 5, 0.4
    pg = pd.PartitionedGraph.from_simulation(n, G, f, 10, 3, 0, 1, dev, seed=3, device_generator=True)
    s = simulate_hits_device(n, G, f, 10, 3, seed=3, score_means=tuple(fl.simulated_score_means), device=dev)
    src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"], num_nodes=n * G,
                                             device=dev)
    ids = pg.scored_edge_ids
    assert torch.equal(torch.sort(ids).values, torch.arange(src.numel(), device=dev))
    ei = pg.scored.edge_index                                   # world 1: local ids are global ids
    assert torch.equal(ei[0], src.long()[ids]) and torch.equal(ei[1], dst.long()[ids])
    assert torch.equal(pg.y, y[ids])
    if fl.skip_connections:
        assert torch.equal(pg.skip, w[ids])
    assert pg.num_edges_total == src.numel()
