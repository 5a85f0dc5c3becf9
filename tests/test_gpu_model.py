"""GPU parity of the whole model (AlternateGCN drop-in) against the golden vectors minted from the
reference's own src/gnn.py, for every flag variant; plus the model.pkl round trip."""
import io

import numpy as np
import pytest
import torch

from oracle.params import make_state_dict
from tests.helpers import GRAD_TOL, VARIANT_FLAGS, assert_close, golden_graph, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5

CASES = [("minimal", "base"), ("minimal", "default"), ("dummy", "default"), ("dummy", "base"),
         ("dummy", "union_skip"), ("c1", "default"), ("c1", "base"), ("c1", "union_skip"),
         ("c1", "cosine"), ("c1", "union_n4"), ("c2", "default"), ("c2", "union_skip"),
         ("sim5", "default"), ("sim5", "union_skip"), ("sim5", "union_n4"),
         ("sim5_trivial", "default")]


@pytest.fixture
def flags():
    from pangnn_b200 import ops, setup
    setup.reset()
    ops.clear_cache()
    yield setup.args
    setup.reset()
    ops.clear_cache()


def build_model(variant, flags):
    from pangnn_b200.gnn import AlternateGCN
    for k, v in VARIANT_FLAGS[variant].items():
        setattr(flags, k, v)
    m = AlternateGCN(DEV, None, False, dims=[flags.node_dim, flags.hidden_dim])
    m.load_state_dict(make_state_dict(flags.node_dim, flags.hidden_dim, flags.skip_connections,
                                      seed=1234), strict=True)
    return m.to(DEV)


@pytest.mark.parametrize("case,variant", CASES)
@pytest.mark.parametrize("fused_loss", [False, True])
def test_model_matches_golden(golden, flags, case, variant, fused_loss):
    g = golden(case)
    model = build_model(variant, flags)
    graph = golden_graph(g, variant, device=DEV)
    pw = float(g[f"model/{variant}/pos_weight"])
    if fused_loss:
        loss, logits = model.forward_loss(graph, pw)
    else:
        logits = model(graph)
        loss = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(pw, device=DEV))(logits, graph.y)
    loss.backward()
    key = f"model/{variant}"
    assert_close("logits", logits.detach().cpu().numpy(), g[f"{key}/logits"], TOL)
    assert abs(loss.item() - float(g[f"{key}/loss"])) <= TOL * abs(float(g[f"{key}/loss"]))
    # identical thresholded predictions at --binary_threshold 0.5 (away from the decision boundary)
    ref_z = g[f"{key}/logits"]
    far = np.abs(ref_z) > 1e-4
    pred = (torch.sigmoid(logits.detach()) >= 0.5).cpu().numpy()
    assert np.array_equal(pred[far], (1 / (1 + np.exp(-ref_z.astype(np.float64))) >= 0.5)[far])
    for name, p in model.named_parameters():
        gk = f"{key}/grad/{name}"
        if gk not in g.files:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert_close(f"grad {name}", p.grad.cpu().numpy(), g[gk], GRAD_TOL)


def test_state_dict_round_trip_is_reference_layout(flags):
    """model.pkl = AlternateGCN.state_dict() (pangnn.py:128,341): same keys, order and shapes."""
    model = build_model("default", flags)
    buf = io.BytesIO()
    torch.save(model.state_dict(), buf)
    buf.seek(0)
    sd = torch.load(buf, map_location="cpu")
    ref = make_state_dict()
    assert list(sd.keys()) == list(ref.keys())
    for k in ref:
        assert sd[k].shape == ref[k].shape and torch.equal(sd[k], ref[k])


def test_gcnconv_standalone_api(flags):
    """GCNConv(in, out, add_self_loops=False).forward(x, edge_index, edge_weight=None)."""
    from oracle.gcn import GCNConv as OracleConv
    from pangnn_b200.gnn import GCNConv
    torch.manual_seed(0)
    N, E = 300, 2000
    ei = torch.randint(0, N, (2, E))
    x, w = torch.randn(N, 64), torch.rand(E) * 50 + 1
    oc = OracleConv(64, 128)
    dc = GCNConv(64, 128, add_self_loops=False)
    dc.load_state_dict(oc.state_dict(), strict=True)
    dc = dc.to(DEV)
    for ew in (w, None):
        ref = oc(x, ei, ew)
        got = dc(x.to(DEV), ei.to(DEV), ew.to(DEV) if ew is not None else None)
        assert_close("gcnconv", got.detach().cpu().numpy(), ref.detach().numpy(), TOL)


def test_pipelined_h2d_and_prepare_give_the_same_step(golden, flags):
    """Data.to_pipelined (copy stream + per-tensor events) followed by AlternateGCN.prepare must be
    indistinguishable from a plain synchronous transfer."""
    from pangnn_b200 import ops
    from pangnn_b200.data import Data
    g = golden("c2")
    model = build_model("union_skip", flags)
    host = golden_graph(g, "union_skip", device="cpu")
    hd = Data(host.x, host.edge_index, host.edge_attr, host.y)
    hd.union_edge_index = host.union_edge_index
    hd = hd.pin_memory()
    pw = float(g["model/union_skip/pos_weight"])
    loss_a, logits_a = model.forward_loss(hd.to(DEV), pw)
    ops.clear_cache()
    for _ in range(3):                                       # repeated: exercises block reuse across streams
        gp = model.prepare(hd.to_pipelined(DEV))
        loss_b, logits_b = model.forward_loss(gp, pw)
        assert torch.equal(logits_a, logits_b) and loss_a.item() == loss_b.item()
        ops.clear_cache()


@pytest.mark.parametrize("variant", ["union_skip", "default"])
def test_scored_only_batch_is_assembled_on_the_device(golden, flags, variant):
    """A whole-graph batch that arrives as the scored edges only: prepare() generates the band (a8) and the
    union assembly (a11) on the device; the step must be bit-identical to the fully materialised graph."""
    from pangnn_b200 import ops
    from pangnn_b200.data import Data
    g = golden("c2")
    model = build_model(variant, flags)
    full = golden_graph(g, variant, device=DEV)
    pw = float(g[f"model/{variant}/pos_weight"])
    loss_a, logits_a = model.forward_loss(full, pw)
    E = full.edge_index.size(1)
    ops.clear_cache()
    host = Data(full.x.cpu(), full.edge_index.cpu(), full.edge_attr[:E].cpu(), full.y.cpu()).pin_memory()
    for _ in range(2):
        gp = model.prepare(host.to_pipelined(DEV, order=model.transfer_order(scored_only=True)))
        if variant == "union_skip":
            assert torch.equal(gp.union_edge_index, full.union_edge_index) and torch.equal(gp.edge_attr, full.edge_attr)
        else:
            assert torch.equal(gp.neighbour_edge_index, full.neighbour_edge_index)
        loss_b, logits_b = model.forward_loss(gp, pw)
        assert torch.equal(logits_a, logits_b) and loss_a.item() == loss_b.item()
        ops.clear_cache()


@pytest.mark.parametrize("case,variant", [("c2", "union_skip"), ("c2", "default"), ("c1", "base"), ("sim5", "union_n4")])
@pytest.mark.parametrize("ones", [True, False])
def test_fused_embedding_conv_equals_the_two_modules(golden, flags, case, variant, ones):
    """Linear(1, D) + conv_in as one rank-2 update (ops.RankOneFn) against the unfused modules, for x = ones
    (the reference's features) and for arbitrary scalar features: logits, loss and every parameter gradient."""
    g = golden(case)
    model = build_model(variant, flags)
    graph = golden_graph(g, variant, device=DEV)
    if not ones:
        graph.x = torch.randn(graph.x.shape, generator=torch.Generator().manual_seed(3)).to(DEV)
    pw = float(g[f"model/{variant}/pos_weight"])
    out = {}
    for fused in (True, False):
        model.fuse_embedding = fused
        model.zero_grad()
        loss, logits = model.forward_loss(graph, pw)
        loss.backward()
        out[fused] = (loss.item(), logits.cpu().numpy(), {k: p.grad.cpu().numpy().copy() for k, p in model.named_parameters()
                                                          if p.grad is not None})
    fused, ref = out[True], out[False]
    assert abs(fused[0] - ref[0]) <= 2e-6 * abs(ref[0])
    assert rel_err(fused[1], ref[1]) < 5e-6
    assert sorted(fused[2]) == sorted(ref[2])
    for k, v in ref[2].items():
        assert rel_err(fused[2][k], v) < 2e-5, k


@pytest.mark.parametrize("variant", ["union_skip", "default"])
def test_prefetch_loader_overlaps_without_changing_results(golden, flags, variant):
    """PrefetchLoader: batch i+1 is copied and prepared on side streams while step i runs; every step must be
    bit-identical to the step on the resident graph (exercises the allocator hand-over across streams)."""
    from pangnn_b200 import ops
    from pangnn_b200.data import Data, PrefetchLoader
    g = golden("c2")
    model = build_model(variant, flags)
    full = golden_graph(g, variant, device=DEV)
    pw = float(g[f"model/{variant}/pos_weight"])
    E = full.edge_index.size(1)
    host = Data(full.x.cpu(), full.edge_index.cpu(), full.edge_attr[:E].cpu(), full.y.cpu()).pin_memory()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)          # parameters stay put: every step must repeat
    ref = None
    loader = PrefetchLoader([host] * 6, model, DEV)
    for step_no, gp in enumerate(loader):
        opt.zero_grad()
        loss, logits = model.forward_loss(gp, pw)
        loss.backward()
        if step_no % 2 == 0:
            loader.prefetch_next()                           # overlapped start; odd steps use the lazy start
        grads = torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])
        cur = (loss.item(), logits.clone(), grads.clone())
        if ref is None:
            ref = cur
            ops.clear_cache()
            loss_a, logits_a = model.forward_loss(full, pw)
            assert loss_a.item() == cur[0] and torch.equal(logits_a, cur[1])
        else:
            assert cur[0] == ref[0] and torch.equal(cur[1], ref[1]) and torch.equal(cur[2], ref[2])
    assert len(ops._STRUCTS) <= 2


def test_cuda_graph_step_matches_eager(golden, flags):
    """GraphedStep (capture once, replay) walks the same loss trajectory as the eager step."""
    from pangnn_b200.graphs import GraphedStep
    g = golden("c2")
    pw = float(g["model/default/pos_weight"])
    graph = golden_graph(g, "default", device=DEV)
    losses = {}
    for mode in ("eager", "graph"):
        model = build_model("default", flags)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)     # same Adam arithmetic in both modes
        out = []
        if mode == "eager":
            for _ in range(6):
                opt.zero_grad(set_to_none=True)
                loss, _ = model.forward_loss(graph, pw)
                loss.backward()
                opt.step()
                out.append(loss.item())
        else:
            step = GraphedStep(model, graph, opt, pw, warmup=2)       # 2 eager warm-up steps (capture itself runs nothing)
            out = [None, None]
            for _ in range(4):
                out.append(step().item())
        losses[mode] = out
    assert losses["eager"][2:] == losses["graph"][2:]               # same kernels, same order: bit-identical


@pytest.mark.parametrize("case,variant", [("c1", "default"), ("c2", "union_skip"), ("sim5", "union_n4")])
def test_predict_matches_reference_head(golden, flags, case, variant):
    """Fused sigmoid + threshold (src/predict.py:54-55): probabilities to 1e-6, identical predictions wherever the
    reference probability is not within 1e-5 of the threshold."""
    g = golden(case)
    model = build_model(variant, flags)
    graph = golden_graph(g, variant, device=DEV)
    logits, prob, pred = model.predict(graph, 0.5)
    ref_z = torch.as_tensor(g[f"model/{variant}/logits"])
    ref_p = torch.sigmoid(ref_z)
    assert_close("logits", logits.cpu().numpy(), ref_z.numpy(), TOL)
    assert float((prob.cpu() - ref_p).abs().max()) < 2e-6
    clear = (ref_p - 0.5).abs() > 1e-5
    assert torch.equal(pred.cpu()[clear].long(), (ref_p >= 0.5).long()[clear])
    assert pred.dtype == torch.int32 and int(clear.sum()) > 0.99 * ref_p.numel()


def _random_subgraphs(num, union, seed=0, categorical=False):
    from pangnn_b200.data import Data
    rng = np.random.default_rng(seed)
    out = []
    for i in range(num):
        n = int(rng.integers(1, 20))
        e = int(rng.integers(0, 14)) if i % 7 else 0                 # some graphs without scored edges
        u = e + int(rng.integers(0, 16))
        x = torch.ones(n) if categorical else torch.ones(n, 1)
        g = Data(x, torch.from_numpy(rng.integers(0, n, (2, e))), torch.from_numpy(rng.random(u if union else e).astype(np.float32)),
                 torch.from_numpy(rng.integers(0, 2, e).astype(np.float32)))
        if union:
            g.union_edge_index = torch.from_numpy(rng.integers(0, n, (2, u)))
        else:
            g.neighbour_edge_index = torch.from_numpy(rng.integers(0, n, (2, u)))
        g.node_id = torch.from_numpy(rng.integers(0, 10 ** 6, n))
        out.append(g)
    return out


@pytest.mark.parametrize("union", [True, False])
@pytest.mark.parametrize("batch_size", [1, 5, 32, 100, 257])
def test_device_collation_equals_host_collation(union, batch_size):
    """a12 (PyG Batch.from_data_list, SURVEY A.3; pangnn.py:121,152-153) as a device op: DeviceLoader yields the
    same batches, bit for bit and in the same order, as the host collate + H2D of DataLoader -- index offsets,
    `batch`, `ptr`, ragged last batch, graphs without edges."""
    from pangnn_b200.data import DataLoader, DeviceLoader
    graphs = _random_subgraphs(257, union, seed=batch_size)
    host = DataLoader(graphs, batch_size=batch_size, shuffle=True, device=DEV, seed=11)
    dev = DeviceLoader(graphs, batch_size=batch_size, shuffle=True, device=DEV, seed=11)
    assert len(host) == len(dev)
    for epoch in range(2):
        n = 0
        for a, b in zip(host, dev):
            n += 1
            assert sorted(a.keys()) == sorted(b.keys())
            for k in a.keys():
                va, vb = getattr(a, k), getattr(b, k)
                if torch.is_tensor(va):
                    assert va.dtype == vb.dtype and va.shape == vb.shape and torch.equal(va, vb), k
                else:
                    assert va == vb, k
        assert n == len(host)


def test_device_collation_matches_oracle_and_feeds_the_model(flags):
    """The device-collated batch equals the oracle's collate (the restated PyG semantics) and trains the model
    to the same loss as the host-collated one."""
    from oracle import preprocess as op
    from pangnn_b200.data import DeviceLoader, collate
    graphs = _random_subgraphs(64, True, seed=5)
    model = build_model("union_skip", flags)
    loader = DeviceLoader(graphs, batch_size=64, shuffle=False, device=DEV)
    (b,) = list(loader)
    ref = op.collate([{k: getattr(g, k).numpy() for k in ("x", "edge_index", "edge_attr", "y", "union_edge_index", "node_id")}
                      for g in graphs])
    for k, v in ref.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(getattr(b, k).cpu().numpy(), v), k
    hb = collate(graphs).to(DEV)
    la, _ = model.forward_loss(hb, 2.0)
    lb, _ = model.forward_loss(b, 2.0)
    assert la.item() == lb.item()
