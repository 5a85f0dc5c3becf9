"""GPU parity: fused edge scorer (fwd, bwd, fused BCE) vs the oracle's torch-CPU autograd."""
import numpy as np
import pytest
import torch

from oracle.model import bce_with_logits
from tests.helpers import GRAD_TOL, assert_close, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5
D = 64


def make(N, E, skip, seed):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(N, D, generator=g)
    ei = torch.randint(0, N, (2, E), generator=g)
    fin = 2 * D + (1 if skip else 0)
    P = dict(w1=torch.randn(D, fin, generator=g) / fin ** 0.5, b1=torch.randn(D, generator=g) * 0.1,
             w2=torch.randn(D, D, generator=g) / 8, b2=torch.randn(D, generator=g) * 0.1,
             w3=torch.randn(1, D, generator=g) / 8, b3=torch.randn(1, generator=g) * 0.1)
    sk = (torch.rand(E, generator=g) * 80 + 1) if skip else None
    # keep the test inputs away from the ReLU kinks: where a pre-activation is within 1e-4 of zero an
    # fp32 reassociation legitimately flips the derivative, which is not what this test measures
    parts = (h[ei[0]], h[ei[1]]) + ((sk.unsqueeze(1),) if skip else ())
    a1 = torch.cat(parts, 1).double() @ P["w1"].double().t() + P["b1"].double()
    a2 = torch.relu(a1) @ P["w2"].double().t() + P["b2"].double()
    ok = (a1.abs().min(dim=1).values > 1e-4) & (a2.abs().min(dim=1).values > 1e-4)
    if E > 1000:
        ei = ei[:, ok].contiguous()
        sk = sk[ok].contiguous() if skip else None
    y = (torch.rand(ei.size(1), generator=g) < 0.3).float()
    return h, ei, P, sk, y


def oracle_logits(h, ei, P, sk):
    parts = (h[ei[0]], h[ei[1]]) + ((sk.unsqueeze(1),) if sk is not None else ())
    a1 = torch.cat(parts, 1) @ P["w1"].t() + P["b1"]
    a2 = torch.relu(a1) @ P["w2"].t() + P["b2"]
    return (torch.relu(a2) @ P["w3"].t() + P["b3"]).squeeze(-1)


NAMES = ["w1", "b1", "w2", "b2", "w3", "b3"]


@pytest.mark.parametrize("N,E", [(50, 1), (50, 127), (300, 128), (300, 129), (2000, 40_000)])
@pytest.mark.parametrize("skip", [False, True])
def test_scorer_forward_backward(N, E, skip):
    from pangnn_b200 import ops
    h, ei, P, sk, y = make(N, E, skip, E)
    E = ei.size(1)
    ho = h.clone().requires_grad_(True)
    Po = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    zo = oracle_logits(ho, ei, Po, sk)
    dz = torch.randn(E, generator=torch.Generator().manual_seed(1))
    zo.backward(dz)

    hd = h.clone().to(DEV).requires_grad_(True)
    Pd = {k: v.clone().to(DEV).requires_grad_(True) for k, v in P.items()}
    gs = ops.GraphStruct(ei.to(DEV), N)
    zd = ops.EdgeScoreFn.apply(hd, *[Pd[k] for k in NAMES], gs, sk.to(DEV) if skip else None)
    zd.backward(dz.to(DEV))
    assert_close("logits", zd.detach().cpu().numpy(), zo.detach().numpy(), TOL)
    assert_close("dh", hd.grad.cpu().numpy(), ho.grad.numpy(), GRAD_TOL)
    for k in NAMES:
        assert_close(f"d{k}", Pd[k].grad.cpu().numpy(), Po[k].grad.numpy(), GRAD_TOL)


@pytest.mark.parametrize("E,pw", [(1, 1.0), (200, 4.8), (33_333, 0.37)])
@pytest.mark.parametrize("skip", [False, True])
def test_scorer_fused_bce(E, pw, skip):
    from pangnn_b200 import ops
    N = 700
    h, ei, P, sk, y = make(N, E, skip, E + 5)
    E = ei.size(1)
    ho = h.clone().requires_grad_(True)
    Po = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    zo = oracle_logits(ho, ei, Po, sk)
    lo = bce_with_logits(zo, y, pw)
    (lo * 1.7).backward()                                    # non-trivial upstream gradient

    hd = h.clone().to(DEV).requires_grad_(True)
    Pd = {k: v.clone().to(DEV).requires_grad_(True) for k, v in P.items()}
    gs = ops.GraphStruct(ei.to(DEV), N)
    ld, zd = ops.EdgeScoreBCEFn.apply(hd, *[Pd[k] for k in NAMES], gs, sk.to(DEV) if skip else None,
                                      y.to(DEV), pw)
    (ld * 1.7).backward()
    assert abs(ld.item() - lo.item()) <= TOL * abs(lo.item())
    assert_close("logits", zd.cpu().numpy(), zo.detach().numpy(), TOL)
    assert_close("dh", hd.grad.cpu().numpy(), ho.grad.numpy(), GRAD_TOL)
    for k in NAMES:
        assert_close(f"d{k}", Pd[k].grad.cpu().numpy(), Po[k].grad.numpy(), GRAD_TOL)


def test_scorer_extreme_logits_are_finite():
    """Saturated logits (|z| ~ 1e3) must give finite loss / gradients, as torch's formula does."""
    from pangnn_b200 import ops
    N, E = 100, 1000
    h, ei, P, sk, y = make(N, E, False, 9)
    P["w3"] = P["w3"] * 2000
    zo = oracle_logits(h, ei, P, None)
    lo = bce_with_logits(zo, y, 2.0)
    gs = ops.GraphStruct(ei.to(DEV), N)
    Pd = {k: v.to(DEV).requires_grad_(True) for k, v in P.items()}
    ld, zd = ops.EdgeScoreBCEFn.apply(h.to(DEV).requires_grad_(True), *[Pd[k] for k in NAMES], gs,
                                      None, y.to(DEV), 2.0)
    ld.backward()
    assert torch.isfinite(ld) and abs(ld.item() - lo.item()) <= 1e-5 * abs(lo.item())
    assert all(torch.isfinite(Pd[k].grad).all() for k in NAMES)


@pytest.mark.parametrize("mode", [0, 1])
def test_pair_score(mode):
    from pangnn_b200 import ops
    N, E = 400, 5000
    h, ei, *_ = make(N, E, False, 2)
    gs = ops.GraphStruct(ei.to(DEV), N)
    got = ops.edge_pair_score(h.to(DEV), gs, mode).cpu()
    ref = (torch.nn.functional.cosine_similarity(h[ei[0]], h[ei[1]], dim=1) if mode == 0
           else (h[ei[0]] * h[ei[1]]).sum(1))
    assert rel_err(got.numpy(), ref.numpy()) < TOL


@pytest.mark.parametrize("E", [5000, 300_000])
@pytest.mark.parametrize("mode", [0, 1])
def test_pair_score_backward_kernel(mode, E):
    """a17 backward (``pangnn_edge_pair_score_bwd``: two weighted aggregations + a diagonal term) against
    autograd of the reference's formulas (``F.cosine_similarity(z[src], z[dst])``, ``src/gnn.py:206-207``; row-wise
    dot, ``src/gnn.py:77-79``) — sorted and unsorted edge lists, duplicates, isolated nodes."""
    from pangnn_b200 import ops
    N = 400 if E == 5000 else 20_000
    h, ei, *_ = make(N, E, False, 2 + mode)
    ei, E = ei.clone(), ei.size(1)                                      # make() drops edges near a ReLU kink
    ei[:, : E // 20] = ei[:, E // 20: 2 * (E // 20)]                   # duplicate edges
    ei = ei % (N - 7)                                                   # the last 7 nodes have no edge
    g = torch.Generator().manual_seed(E)
    up = torch.randn(E, generator=g)
    hr = h.clone().requires_grad_(True)
    ref = (torch.nn.functional.cosine_similarity(hr[ei[0]], hr[ei[1]], dim=1) if mode == 0
           else (hr[ei[0]] * hr[ei[1]]).sum(1))
    ref.backward(up)
    hd = h.to(DEV).requires_grad_(True)
    got = ops.edge_pair_score(hd, ops.GraphStruct(ei.to(DEV), N), mode)
    got.backward(up.to(DEV))
    assert rel_err(got.detach().cpu().numpy(), ref.detach().numpy()) < TOL
    assert rel_err(hd.grad.cpu().numpy(), hr.grad.numpy()) < TOL
    assert float(hd.grad[N - 7:].abs().max()) == 0.0


def test_scorer_scale_accuracy_vs_fp64():
    """2e6 edges (many tiles per CTA: long tensor-core accumulation chains for dW2): every output and
    gradient of the fused kernel against an fp64 evaluation of the same formulas on the GPU."""
    from pangnn_b200 import ops
    torch.manual_seed(0)
    N, E = 200_000, 2_000_000
    pq = torch.randn(N, 2 * D, device=DEV)
    src = torch.sort(torch.randint(0, N, (E,), device=DEV)).values
    dst = torch.randint(0, N, (E,), device=DEV)
    gs = ops.GraphStruct(torch.stack((src, dst)), N)
    skip = torch.rand(E, device=DEV) * 80 + 1
    y = (torch.rand(E, device=DEV) < 0.2).float()
    w1c, b1, b2 = (torch.randn(D, device=DEV) * 0.1 for _ in range(3))
    b3 = torch.randn(1, device=DEV)
    w2 = torch.randn(D, D, device=DEV) / 8
    w3 = torch.randn(1, D, device=DEV) / 8
    logits = torch.empty(E, device=DEV); loss = torch.zeros(1, dtype=torch.float64, device=DEV)
    pw, scale = 4.0, 1.0 / E
    da1, grads = ops.edge_score_train(pq, w1c, b1, w2, b2, w3, b3, gs, skip, y=y, pos_weight=pw, scale=scale,
                                      logits=logits, loss_sum=loss)
    g = ops.scorer_grads(grads)
    W2, W3 = w2.double(), w3.double().squeeze(0)
    a1 = pq[src, :D].double() + pq[dst, D:].double() + skip[:, None].double() * w1c.double() + b1.double()
    r1 = a1.clamp_min(0)
    a2 = r1 @ W2.t() + b2.double()
    r2 = a2.clamp_min(0)
    z = r2 @ W3 + b3.double()
    yy = y.double()
    lsum = ((1 - yy) * z + (1 + (pw - 1) * yy) * (torch.log1p(torch.exp(-z.abs())) + (-z).clamp_min(0))).sum()
    dz = ((pw * yy + 1 - yy) * torch.sigmoid(z) - pw * yy) * scale
    da2 = dz[:, None] * W3 * (a2 > 0)
    da1_ref = (da2 @ W2) * (a1 > 0)
    rel = lambda got, ref: float((got.double() - ref).abs().max() / ref.abs().max())
    assert rel(logits, z) < 2e-6
    assert abs(float(loss) - float(lsum)) <= 2e-6 * abs(float(lsum))
    # entries whose pre-activation sits within fp32 noise of a ReLU kink may legitimately flip
    ok = ((a1.abs().min(dim=1).values > 1e-5) & (a2.abs().min(dim=1).values > 1e-5))
    assert rel(da1[ok], da1_ref[ok]) < 1e-5
    assert rel(g.dW2, da2.t() @ r1) < 1e-5
    assert rel(g.db2, da2.sum(0)) < 1e-5
    assert rel(g.dw3[0], (dz[:, None] * r2).sum(0)) < 1e-5
    assert rel(g.db1, da1_ref.sum(0)) < 1e-5
    assert rel(g.dw1c, (da1_ref * skip[:, None].double()).sum(0)) < 1e-5


@pytest.mark.parametrize("skew", [False, True])
def test_chunked_scorer_equals_the_single_launch(skew):
    """Scored edges processed in runs of source rows (ops.ScoredChunks; the per-edge spill of a pan-genome-scale
    partition does not fit in one piece): logits identical, loss / node gradients / parameter gradients equal to the
    single-launch form up to the summation order; skewed degrees force the recursive split of a run."""
    from pangnn_b200 import ops
    D, N, E = ops.SCORER_D, 3000, 80_000
    g = torch.Generator().manual_seed(5 + skew)
    src = torch.randint(0, N, (E,), generator=g)
    if skew:
        src[: E // 3] = 17                                      # one source with a third of the edges
    dst = torch.randint(0, N, (E,), generator=g)
    key = src * N + dst
    ei = torch.stack((src, dst))[:, torch.argsort(key, stable=True)].contiguous().to(DEV)
    gs = ops.GraphStruct(ei, N)
    pq = torch.randn(N, 2 * D, generator=g).to(DEV)
    skip = (torch.rand(E, generator=g) * 80 + 1).to(DEV)
    y = (torch.rand(E, generator=g) < 0.2).float().to(DEV)
    w1c, b1, b2 = (torch.randn(D, generator=g).to(DEV) * 0.1 for _ in range(3))
    w2, w3, b3 = (torch.randn(D, D, generator=g) / 8).to(DEV), (torch.randn(1, D, generator=g) / 8).to(DEV), torch.randn(1, generator=g).to(DEV)

    def run(chunk):
        old = ops.SCORER_CHUNK_EDGES["n"]
        ops.SCORER_CHUNK_EDGES["n"] = chunk
        try:
            leaves = [t.clone().requires_grad_(True) for t in (pq, w1c, b1, w2, b2, w3, b3)]
            loss, logits = ops.EdgeScoreBCEPQFn.apply(*leaves, gs, skip, y, 4.0, 1.0 / E, None)
            loss.backward()
            return loss.detach(), logits, [t.grad for t in leaves]
        finally:
            ops.SCORER_CHUNK_EDGES["n"] = old
    l0, z0, g0 = run(1 << 30)
    l1, z1, g1 = run(7000)
    ch = ops.scored_chunks(gs, 7000)
    assert len(ch.runs) > 5 and sum(c1 - c0 for _, _, c0, c1 in ch.runs) == E
    assert torch.equal(z0, z1)
    assert abs(float(l0) - float(l1)) <= 1e-6 * abs(float(l0))
    for a, b in zip(g0, g1):
        assert rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-5


def test_scorer_launch_counts():
    """Kernel launches each scorer path adds to ``ops.LAUNCHES`` (bench.py reports the total as ``gpu_launches``),
    on a small graph in canonical (src, dst) order whose structures and chunks are built beforehand."""
    from pangnn_b200 import ops
    N, E, chunk = 1000, 20_000, 7000
    h, ei, P, sk, y = make(N, E, True, 3)
    order = torch.argsort(ei[0] * N + ei[1], stable=True)
    ei, sk, y = ei[:, order].contiguous().to(DEV), sk[order].to(DEV), y[order].to(DEV)
    gs = ops.GraphStruct(ei, N)
    runs = len(ops.scored_chunks(gs, chunk).runs)
    gs.endpoints32
    assert gs.src.identity_perm and runs > 1
    hd = h.to(DEV).requires_grad_(True)
    Pd = {k: v.to(DEV).requires_grad_(True) for k, v in P.items()}
    wcat, w1c = ops.split_w1(Pd["w1"].detach(), True)
    pq = ops.node_linear(hd.detach(), wcat)
    weights = (w1c,) + tuple(Pd[k].detach() for k in NAMES[1:])
    counts = {}

    def count(name, fn):
        n0 = ops.LAUNCHES["count"]
        out = fn()
        counts[name] = ops.LAUNCHES["count"] - n0
        return out

    z = count("EdgeScoreFn", lambda: ops.EdgeScoreFn.apply(hd, *[Pd[k] for k in NAMES], gs, sk))
    count("EdgeScoreFn backward", z.sum().backward)
    loss, _ = count("EdgeScoreBCEFn", lambda: ops.EdgeScoreBCEFn.apply(hd, *[Pd[k] for k in NAMES], gs, sk, y, 2.0))
    count("EdgeScoreBCEFn backward", loss.backward)
    for name, limit in (("EdgeScoreBCEPQFn", 1 << 30), ("EdgeScoreBCEPQFn chunked", chunk)):
        old = ops.SCORER_CHUNK_EDGES["n"]
        ops.SCORER_CHUNK_EDGES["n"] = limit
        try:
            leaves = [t.clone().requires_grad_(True) for t in (pq,) + weights]
            loss, _ = count(name, lambda: ops.EdgeScoreBCEPQFn.apply(*leaves, gs, sk, y, 2.0, 1.0 / E))
        finally:
            ops.SCORER_CHUNK_EDGES["n"] = old
        count(name + " backward", loss.backward)
    count("edge_score_pq_fwd", lambda: ops.edge_score_pq_fwd(pq, *weights, gs, sk))
    count("edge_score_predict", lambda: ops.edge_score_predict(pq, *weights, gs, sk))
    assert counts == {"EdgeScoreFn": 2, "EdgeScoreFn backward": 7,
                      "EdgeScoreBCEFn": 4, "EdgeScoreBCEFn backward": 5,
                      "EdgeScoreBCEPQFn": 3, "EdgeScoreBCEPQFn backward": 2,
                      "EdgeScoreBCEPQFn chunked": 7 * runs, "EdgeScoreBCEPQFn chunked backward": 0,
                      "edge_score_pq_fwd": 1, "edge_score_predict": 1}, counts
