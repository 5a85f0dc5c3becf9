"""GPU parity: gcn_norm, normalised aggregation and the GCN layer fwd+bwd vs the oracle.
Tolerance: 1e-5 relative to the tensor's scale, fp32 (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from oracle import gcn as ogcn
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


def random_graph(N, E, seed, skew=False):
    rng = np.random.RandomState(seed)
    src = rng.randint(0, N, size=E)
    if skew:                                                 # heavy-tailed in-degree (NegBin-like)
        dst = np.minimum((rng.pareto(1.2, size=E) * N / 50).astype(np.int64), N - 1)
    else:
        dst = rng.randint(0, N, size=E)
    w = rng.uniform(1.0, 81.0, size=E).astype(np.float32)
    w[rng.rand(E) < 0.3] = 81.0
    return np.stack((src, dst)).astype(np.int64), w


@pytest.mark.parametrize("N,E,skew", [(1, 0, False), (7, 3, False), (500, 4000, True),
                                      (20000, 96350, False), (100_000, 1_500_000, True)])
@pytest.mark.parametrize("weighted", [True, False])
def test_gcn_norm(N, E, skew, weighted):
    from pangnn_b200 import ops
    ei, w = random_graph(N, E, 1, skew)
    t_ei = torch.from_numpy(ei).to(DEV)
    t_w = torch.from_numpy(w).to(DEV) if weighted else None
    gs = ops.GraphStruct(t_ei, N)
    ent = gs.norm(t_w, need_src=True)
    ref = ogcn.gcn_norm(torch.from_numpy(ei), torch.from_numpy(w) if weighted else None, N).numpy()
    got_dst = np.empty(E, np.float32); got_dst[gs.dst.perm.cpu().numpy()] = ent["dst"].cpu().numpy()
    got_src = np.empty(E, np.float32); got_src[gs.src.perm.cpu().numpy()] = ent["src"].cpu().numpy()
    if E:
        assert rel_err(got_dst, ref) < TOL
        assert np.array_equal(got_dst, got_src)             # same value in both orientations


@pytest.mark.parametrize("F", [4, 16, 32, 48, 64, 128, 256])
@pytest.mark.parametrize("act,use_bias", [(0, False), (1, True)])
def test_aggregate_matches_oracle(F, act, use_bias):
    from pangnn_b200 import ops
    N, E = 3000, 40000
    ei, w = random_graph(N, E, F, skew=True)
    x = torch.randn(N, F, generator=torch.Generator().manual_seed(F))
    bias = torch.randn(F, generator=torch.Generator().manual_seed(F + 1)) if use_bias else None
    norm = ogcn.gcn_norm(torch.from_numpy(ei), torch.from_numpy(w), N)
    ref = ogcn.gcn_propagate(x, torch.from_numpy(ei), norm)
    if use_bias:
        ref = ref + bias
    if act:
        ref = torch.nn.functional.elu(ref)
    gs = ops.GraphStruct(torch.from_numpy(ei).to(DEV), N)
    ent = gs.norm(torch.from_numpy(w).to(DEV), need_src=False)
    got = ops.gcn_aggregate(gs.dst.rowptr, gs.dst.col, ent["dst"], x.to(DEV), N,
                            bias.to(DEV) if use_bias else None, act)
    assert rel_err(got.cpu().numpy(), ref.numpy()) < TOL


def test_aggregate_strided_views_and_unit_values():
    """Column-slice inputs/outputs (row stride > F) and val == NULL (segment sum of edge rows)."""
    from pangnn_b200 import ops
    N, E = 1000, 9000
    ei, _ = random_graph(N, E, 5)
    gs = ops.GraphStruct(torch.from_numpy(ei).to(DEV), N)
    da1 = torch.randn(E, 64, device=DEV)
    out = torch.zeros(N, 128, device=DEV)
    ops.gcn_aggregate(gs.src.rowptr, gs.src.perm, None, da1, N, out=out[:, :64])
    ops.gcn_aggregate(gs.dst.rowptr, gs.dst.perm, None, da1, N, out=out[:, 64:])
    ref = torch.zeros(N, 128)
    ref[:, :64].index_add_(0, torch.from_numpy(ei[0]), da1.cpu())
    ref[:, 64:].index_add_(0, torch.from_numpy(ei[1]), da1.cpu())
    assert rel_err(out.cpu().numpy(), ref.numpy()) < TOL


@pytest.mark.parametrize("fin,fout", [(64, 128), (128, 128), (128, 64), (16, 32)])
@pytest.mark.parametrize("weighted,act", [(True, 1), (False, 1), (True, 0)])
def test_gcn_layer_forward_backward(fin, fout, weighted, act):
    from pangnn_b200 import ops
    N, E = 2500, 30000
    ei, w = random_graph(N, E, fin + fout, skew=True)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, fin, generator=g)
    W = torch.randn(fout, fin, generator=g) * 0.1
    b = torch.randn(fout, generator=g) * 0.1
    dy = torch.randn(N, fout, generator=g)
    # oracle
    xo, Wo, bo = (t.clone().requires_grad_(True) for t in (x, W, b))
    conv = ogcn.GCNConv(fin, fout)
    out = ogcn.gcn_propagate(xo @ Wo.t(), torch.from_numpy(ei),
                             ogcn.gcn_norm(torch.from_numpy(ei), torch.from_numpy(w) if weighted else None, N)) + bo
    if act:
        out = torch.nn.functional.elu(out)
    out.backward(dy)
    # device
    xd, Wd, bd = (t.clone().to(DEV).requires_grad_(True) for t in (x, W, b))
    got = ops.gcn_layer(xd, Wd, bd, torch.from_numpy(ei).to(DEV),
                        torch.from_numpy(w).to(DEV) if weighted else None, act)
    got.backward(dy.to(DEV))
    assert rel_err(got.detach().cpu().numpy(), out.detach().numpy()) < TOL
    assert rel_err(xd.grad.cpu().numpy(), xo.grad.numpy()) < TOL
    assert rel_err(Wd.grad.cpu().numpy(), Wo.grad.numpy()) < TOL
    assert rel_err(bd.grad.cpu().numpy(), bo.grad.numpy()) < TOL


def test_aggregate_linearity_full_size():
    """Size-independent property at C3-like scale: A(ax + by) == a A(x) + b A(y)."""
    from pangnn_b200 import ops
    N, E, F = 1_000_000, 10_000_000, 64
    g = torch.Generator(device=DEV).manual_seed(0)
    ei = torch.randint(0, N, (2, E), device=DEV, generator=g)
    w = torch.rand(E, device=DEV, generator=g) * 80 + 1
    gs = ops.GraphStruct(ei, N)
    ent = gs.norm(w, need_src=False)
    x = torch.randn(N, F, device=DEV, generator=g)
    y = torch.randn(N, F, device=DEV, generator=g)
    agg = lambda v: ops.gcn_aggregate(gs.dst.rowptr, gs.dst.col, ent["dst"], v, N)
    lhs = agg(2.0 * x - 3.0 * y)
    rhs = 2.0 * agg(x) - 3.0 * agg(y)
    assert float((lhs - rhs).abs().max() / rhs.abs().max()) < 1e-5
    # row sums of A_hat against the norm values (checksum of checksums)
    ones = torch.ones(N, 4, device=DEV)
    rs = ops.gcn_aggregate(gs.dst.rowptr, gs.dst.col, ent["dst"], ones, N)[:, 0]
    assert abs(float(rs.double().sum()) - float(ent["dst"].double().sum())) < 1e-6 * float(ent["dst"].double().sum())


@pytest.mark.parametrize("M,K", [(64, 64), (64, 128), (128, 64), (128, 128)])
@pytest.mark.parametrize("N", [1, 31, 32, 33, 10_000, 300_001])
def test_gemm_tn(M, K, N):
    """dW = A^T B streaming kernel vs an fp64 product."""
    from pangnn_b200 import ops
    g = torch.Generator().manual_seed(N + M + K)
    a = torch.randn(N, M, generator=g)
    b = torch.randn(N, K, generator=g)
    ref = (a.double().t() @ b.double()).numpy()
    got = ops.gemm_tn(a.to(DEV), b.to(DEV)).cpu().numpy()
    assert rel_err(got, ref) < TOL
    # strided operands (column halves of a wider matrix)
    wide = torch.randn(N, 2 * M, generator=g).to(DEV)
    got2 = ops.gemm_tn(wide[:, M:], b.to(DEV)).cpu().numpy()
    assert rel_err(got2, (wide[:, M:].cpu().double().t() @ b.double()).numpy()) < TOL


def test_rank1_first_layer_at_bench_scale():
    """Embedding Linear(1, D) + first GCNConv as one rank-2 update vs the two modules at C3 size (N = 1e6,
    1.7e7 edges, D = 64 -> F = 128): outputs and all five parameter gradients."""
    from pangnn_b200 import ops
    dev = "cuda:0"
    N, E, D, F = 1_000_000, 17_000_000, 64, 128
    g = torch.Generator(device=dev).manual_seed(0)
    ei = torch.stack((torch.randint(0, N, (E,), device=dev, generator=g), torch.randint(0, N, (E,), device=dev, generator=g)))
    w = torch.rand(E, device=dev, generator=g) * 80 + 1
    x = torch.ones(N, 1, device=dev)
    mk = lambda *s: (torch.randn(*s, device=dev, generator=g) * 0.3).requires_grad_(True)
    w_e, b_e, W, b = mk(D, 1), mk(D), mk(F, D), mk(F)
    dy = torch.randn(N, F, device=dev, generator=g)
    y1 = ops.embed_conv(x, w_e, b_e, W, b, ei, w, ops.ACT_ELU)
    y1.backward(dy)
    g1 = [p.grad.clone() for p in (w_e, b_e, W, b)]
    for p in (w_e, b_e, W, b):
        p.grad = None
    e0 = torch.addcmul(b_e, x, w_e.t())
    y2 = ops.gcn_layer(e0, W, b, ei, w, ops.ACT_ELU)
    y2.backward(dy)
    g2 = [p.grad for p in (w_e, b_e, W, b)]
    scale = float(y2.detach().abs().max())
    assert float((y1.detach() - y2.detach()).abs().max()) < 1e-5 * scale
    for a, r in zip(g1, g2):
        assert float((a - r).abs().max()) < 1e-4 * float(r.abs().max())


@pytest.mark.parametrize("F", [32, 64, 128])
def test_identity_segment_sum_equals_the_gathered_one(F):
    """col == NULL in pangnn_gcn_aggregate (rows of x already in CSR order, the scorer's per-edge gradients of a
    canonically ordered edge list) == the same sum through the perm gather, bit for bit; empty rows, long rows."""
    from pangnn_b200 import ops
    N, E = 20_011, 300_000
    g = torch.Generator().manual_seed(F)
    src = torch.sort(torch.randint(0, N, (E,), generator=g)).values
    src[:5000] = 7                                              # one long row
    src = torch.sort(src).values
    dst = torch.randint(0, N, (E,), generator=g)
    key = src * N + dst
    ei = torch.stack((src, dst))[:, torch.argsort(key, stable=True)].contiguous().to(DEV)
    gs = ops.GraphStruct(ei, N)
    assert gs.src.identity_perm and not gs.dst.identity_perm
    rows = torch.randn(E, F, generator=g).to(DEV)
    ref = ops.gcn_aggregate(gs.src.rowptr, gs.src.perm, None, rows, N)
    got = ops.segment_sum_edges(gs.src, rows, N, torch.empty(N, F, device=DEV))
    assert torch.equal(got, ref)
    wide = torch.empty(N, 2 * F, device=DEV)                    # strided output (the dpq halves)
    ops.segment_sum_edges(gs.src, rows, N, wide[:, :F])
    assert torch.equal(wide[:, :F], ref)
