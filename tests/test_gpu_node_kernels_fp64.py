"""The node-side kernels of the training step, one entry point at a time, against fp64 on one GPU.

Whole-model tests (``test_gpu_c3_fp64.py``) say that a step is wrong, not which kernel broke at which shape.  Each
test here calls one kernel at the shapes where its schedule changes -- the persistent block cap, the ``kFlush``
chain cut of ``gemm_tn``, the tile ring of ``node_linear`` -- and compares it with plain torch fp64 written from the definition (dense products, ``index_add_`` over the edge list).
Where a kernel has to be isolated from its fp32 inputs (the CSR values), the reference takes those same fp32 inputs
promoted to fp64.  The halo kernels see only device pointers, so their peer buffers are plain device tensors here.

Bars are either condition-aware (``|got - ref| <= rel * sum |term|``, per element or per column) or bit-exact where
the kernel performs the same roundings as torch.  ``-s`` prints a table per case: the measured error and, where
the bar is element-wise, the largest ratio of error to bar.
"""
import zlib

import pytest
import torch
import torch.nn.functional as tnf

from tests.helpers import Table, bits, check, lib, nan_fill, plain_fp32, ptr, ratio, scale_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24                                 # fp32 unit roundoff
NUM_SMS = 148
CAP_ROWS = 64 * NUM_SMS * 8                    # rank1_bwd / act_bwd_bias: 64-row chunks, persistent cap kNumSMs * 8
ROW_N = [0, 1, 63, 64, 65, CAP_ROWS - 1, CAP_ROWS, CAP_ROWS + 1, 1_000_000]
ROW_F = [4, 64, 96, 128, 256]                  # F = 96: 24 threads per row, TY = 10, 16 threads idle
SHAPES = [(64, 64), (128, 64), (64, 128), (128, 128)]
# Bars (measured on one B200 in profiles/r06_node_kernels_fp64.log; the figures are in DESIGN.md section 2)
COL_REL = 1e-6                                 # column sums: |got - ref| <= COL_REL * sum_r |term_r|
SCALE_REL = 1e-5                               # the project's scale-relative bar
NL_SCALE, NL_ABS = 2e-6, 2e-7                  # node_linear: 3xTF32 + ex2.approx ELU
# gemm_tn: the tensor core truncates when it adds into its fp32 accumulator, so the error drifts one way along a
# chain (16 tiles = 192 tcgen05.mma) where cuBLAS rounds to nearest; one-signed operands show it most.  Measured on
# one B200 against fp64: randn ours <= 4.2e-6 (at most 4.1 x cuBLAS fp32), one-signed ours 1.2-5.5e-6 (cuBLAS fp32
# 0.5-2.2e-6); with the chain left uncut, one-signed 9.2-11e-6 at 32-33 tiles per CTA and 2.1-2.6e-5 at 1e6 rows.
TN_DRIFT = 8e-6                                # every case
TN_FP32 = 6.0                                  # randn: at most this many times cuBLAS fp32's error (floor 2e-6)


def ops():
    from pangnn_b200 import ops as o
    return o


def gen(*seed):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(repr(seed).encode()))


# ------------------------------------------------------------------------------------------------
# graphs given by their row degrees
# ------------------------------------------------------------------------------------------------
def csr_of(deg, g, n_src=None):
    """(rowptr int64, col int32, val fp32 > 0, row of each edge) of a CSR with the given row degrees."""
    deg = torch.as_tensor(deg, dtype=torch.int64, device=DEV)
    N = deg.numel()
    rowptr = torch.zeros(N + 1, dtype=torch.int64, device=DEV)
    rowptr[1:] = deg.cumsum(0)
    E = int(rowptr[-1])
    col = torch.randint(0, max(n_src or N, 1), (E,), generator=g, device=DEV, dtype=torch.int32)
    val = torch.rand(E, generator=g, device=DEV) * 0.5 + 0.01
    rows = torch.repeat_interleave(torch.arange(N, device=DEV), deg)
    return rowptr, col, val, rows


def row_sum64(rows, N, vals):
    """fp64 sum of per-edge values (vector or [E, F]) into their rows."""
    out = torch.zeros((N,) + tuple(vals.shape[1:]), dtype=torch.float64, device=DEV)
    return out.index_add_(0, rows, vals)


# ------------------------------------------------------------------------------------------------
# A. rank-1 first layer (rank1.cu)
# ------------------------------------------------------------------------------------------------
def _spmv_graph(name, g):
    if name == "edgeless":
        return [0] * 100
    if name == "one_row":
        return [37]
    if name == "empty_rows":
        d = torch.randint(0, 21, (5000,), generator=g, device=DEV)
        return d * (torch.rand(5000, generator=g, device=DEV) > 0.3)
    d = torch.randint(0, 9, (1000,), generator=g, device=DEV)               # hub: one row of 150 000 edges
    d[417] = 150_000
    return d


@pytest.mark.parametrize("graph", ["edgeless", "one_row", "empty_rows", "hub"])
def test_csr_spmv2_matches_fp64(graph):
    """a = A x, c = A 1, accumulated in fp64 and rounded once: within half an ulp plus fp64 accumulation."""
    g = gen("spmv2", graph)
    rowptr, col, val, rows = csr_of(_spmv_graph(graph, g), g)
    N = rowptr.numel() - 1
    t = Table(f"csr_spmv2, {graph}: N = {N}, E = {col.numel()}", ["max err/bar"])
    for xname in ("ones", "positive", "mixed"):
        x = {"ones": torch.ones(N, device=DEV), "positive": torch.rand(N, generator=g, device=DEV) + 0.01,
             "mixed": torch.randn(N, generator=g, device=DEV)}[xname]
        a, c = torch.full((N,), float("nan"), device=DEV), torch.full((N,), float("nan"), device=DEV)
        check(lib().pangnn_csr_spmv2(ptr(rowptr), ptr(col), ptr(val), ptr(x), N, ptr(a), ptr(c),
                                     ops()._stream()), "csr_spmv2")
        v64, x64 = val.double(), x.double()[col.long()]
        for name, got, term in (("a", a, v64 * x64), ("c", c, v64)):
            ref, mag = row_sum64(rows, N, term), row_sum64(rows, N, term.abs())
            r = ratio((got.double() - ref).abs(), U * ref.abs() + 1e-12 * mag)
            t.add(f"x {xname}: {name}", r, ok=r <= 1.0, why=f"{name} error {r:.2f} x bar")
    t.check()


@pytest.mark.parametrize("F", ROW_F)
def test_rank1_affine_act_matches_fp64(F):
    """y = act(a u + c v + b), with a row stride ldy > F, pre-activations around 0 and below -20; the padding of
    each row is never written."""
    o = ops()
    g = gen("affine", F)
    N, ldy = 3001, F + 12
    a = torch.randn(N, generator=g, device=DEV)
    c = torch.rand(N, generator=g, device=DEV) * 2
    a[::3] *= 40                                                          # |pre| up to ~100: far below -20
    a[1::7], c[1::7] = 0.0, 0.0                                           # pre = b: around 0
    u, v = torch.randn(F, generator=g, device=DEV), torch.randn(F, generator=g, device=DEV) * 0.5
    b = torch.randn(F, generator=g, device=DEV) * 0.1
    a64, c64, u64, v64, b64 = (t.double() for t in (a, c, u, v, b))
    t = Table(f"rank1_affine_act, F = {F}, N = {N}, ldy = {ldy}", ["max err/bar", "pre < -20"])
    for bias in (None, b):
        for act in (o.ACT_NONE, o.ACT_ELU):
            buf = nan_fill(N, ldy)
            fill = bits(buf).clone()
            check(lib().pangnn_rank1_affine_act(ptr(a), ptr(c), ptr(u), ptr(v), ptr(bias), N, F, act, ptr(buf), ldy,
                                                o._stream()), "rank1_affine_act")
            bb = b64 if bias is not None else torch.zeros_like(b64)
            pre = a64[:, None] * u64 + c64[:, None] * v64 + bb
            ref = torch.where(pre > 0, pre, torch.expm1(pre)) if act == o.ACT_ELU else pre
            bar = 4 * U * ((a64[:, None] * u64).abs() + (c64[:, None] * v64).abs() + bb.abs())
            r = ratio((buf[:, :F].double() - ref).abs(), bar)
            pad_ok = torch.equal(bits(buf)[:, F:], fill[:, F:])
            case = f"bias {'yes' if bias is not None else 'no'}, act {'elu' if act else 'none'}"
            t.add(case, r, int((pre < -20).sum()), ok=r <= 1.0 and pad_ok,
                  why=f"error {r:.2f} x bar" if pad_ok else "padding of a row written")
    t.check()


def _dy(kind, N, F, g):
    return torch.randn(N, F, generator=g, device=DEV) if kind == "randn" else \
        torch.rand(N, F, generator=g, device=DEV) + 0.1


def _elu_out(N, F, g):
    """ELU outputs with the edge values of the derivative: +-0.0, just above -1, tiny of both signs."""
    y = tnf.elu(torch.randn(N, F, generator=g, device=DEV) * 2)
    special = torch.tensor([0.0, -0.0, -1.0 + 2.0 ** -24, -0.99999994, 1e-30, -1e-30, -1e-7, 2.0 ** -126],
                           device=DEV)
    k = min(y.numel(), 8 * 64)
    y.view(-1)[:k] = special.repeat(64)[:k]
    return y


def _col_bar(t, case, got, ref, mag):
    """Per column |got - ref| <= COL_REL * sum |term|, and the scale-relative SCALE_REL."""
    r = ratio((got.double() - ref).abs(), COL_REL * mag)
    e = scale_err(got, ref)
    t.add(case, r, e, ok=r <= 1.0 and e <= SCALE_REL, why=f"column error {r:.2f} x bar, scale-relative {e:.2e}")


@pytest.mark.parametrize("F", ROW_F)
@pytest.mark.parametrize("N", ROW_N)
def test_rank1_bwd_column_sums(N, F):
    """(sum g, sum a g, sum c g) with g = dy * act'(y), around the persistent block cap and at 1e6 rows."""
    o = ops()
    g = gen("rank1_bwd", N, F)
    t = Table(f"rank1_bwd, N = {N}, F = {F}", ["col err/bar", "scale err"])
    a = torch.randn(N, generator=g, device=DEV)
    c = torch.rand(N, generator=g, device=DEV) * 2
    y = _elu_out(N, F, g)
    for kind in ("randn", "one-signed"):
        dy = _dy(kind, N, F, g)
        for act in (o.ACT_NONE, o.ACT_ELU):
            sums = torch.full((3, F), float("nan"), device=DEV)
            ws = o._ws(lib().pangnn_rank1_bwd_workspace_bytes(N, F), DEV)
            check(lib().pangnn_rank1_bwd(ptr(dy), ptr(y), ptr(a), ptr(c), N, F, act, ptr(sums), ptr(ws), ws.numel(),
                                         o._stream()), "rank1_bwd")
            g64 = dy.double() * (torch.where(y > 0, 1.0, y.double() + 1) if act == o.ACT_ELU else 1.0)
            for k, wgt in enumerate((None, a.double()[:, None], c.double()[:, None])):
                term = g64 if wgt is None else wgt * g64
                _col_bar(t, f"{kind}, act {'elu' if act else 'none'}: {('db', 'du', 'dv')[k]}", sums[k],
                         term.sum(0), term.abs().sum(0))
            del g64, term
    t.check()


def _random_graph(N, E, g):
    src = torch.randint(0, N, (E,), generator=g, device=DEV)
    dst = torch.randint(0, N, (E,), generator=g, device=DEV)
    key = torch.argsort(src * N + dst)
    return torch.stack((src[key], dst[key])).contiguous(), torch.rand(E, generator=g, device=DEV) * 80 + 1


def _conv64(gs, weight, h):
    """fp64 A_hat h over the by-destination CSR of ``gs`` and its fp32 gcn_norm values (promoted)."""
    d = gs.dst
    val = gs.norm(weight, need_src=False)["dst"].double()
    rows = torch.repeat_interleave(torch.arange(gs.num_nodes, device=DEV), d.rowptr.diff())
    return row_sum64(rows, gs.num_nodes, val[:, None] * h[d.col.long()])


@pytest.mark.parametrize("F", [32, 64, 128])
@pytest.mark.parametrize("x_kind", ["ones", "scalar"])
def test_embed_conv_autograd_matches_fp64_unfused(x_kind, F):
    """RankOneFn (embed_conv): output and dw_e, db_e, dW, db against fp64 autograd of the unfused
    Linear(1, D) -> GCNConv."""
    o = ops()
    g = gen("rank1_autograd", x_kind, F)
    N, E, D = 20_000, 200_000, 64
    ei, w = _random_graph(N, E, g)
    x = torch.ones(N, 1, device=DEV) if x_kind == "ones" else torch.randn(N, 1, generator=g, device=DEV)
    params = [torch.randn(*s, generator=g, device=DEV) * 0.3 for s in ((D, 1), (D,), (F, D), (F,))]
    dy = torch.randn(N, F, generator=g, device=DEV)
    t = Table(f"rank-1 autograd, x {x_kind}, N = {N}, F = {F}", ["scale err"])
    try:
        ps = [p.clone().requires_grad_(True) for p in params]
        out = o.embed_conv(x, *ps, ei, w, o.ACT_ELU)
        out.backward(dy)
        p64 = [p.double().requires_grad_(True) for p in params]
        w_e, b_e, W, b = p64
        e0 = x.double() @ w_e.t() + b_e
        ref = tnf.elu(_conv64(o.graph_struct(ei, N), w, e0 @ W.t()) + b)
        ref.backward(dy.double())
        for name, got, r in zip(("out", "dw_e", "db_e", "dW", "db"), [out] + [p.grad for p in ps],
                                [ref] + [p.grad for p in p64]):
            e = scale_err(got.detach(), r.detach())
            t.add(f"RankOneFn: {name}", e, ok=e <= SCALE_REL, why=f"{name} {e:.2e}")
    finally:
        o.clear_cache()
    t.check()


# ------------------------------------------------------------------------------------------------
# B. activation backward + bias gradient (act_bwd_bias, gcn.cu)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", ROW_F + [1020, 1024])
@pytest.mark.parametrize("N", ROW_N)
def test_act_bwd_bias_matches_fp64(N, F):
    """g bit-identical to fp32 torch (the same two roundings), dbias per column against fp64; need_g=False gives
    the same dbias."""
    o = ops()
    g = gen("act_bwd", N, F)
    t = Table(f"act_bwd_bias, N = {N}, F = {F}", ["col err/bar", "scale err"])
    y = _elu_out(N, F, g)
    for kind in ("randn", "one-signed"):
        dy = _dy(kind, N, F, g)
        for act in (o.ACT_NONE, o.ACT_ELU):
            gg, db = o.act_bwd_bias(dy, y, act)
            want = dy * torch.where(y > 0, 1, y + 1) if act == o.ACT_ELU else dy
            same = torch.equal(bits(gg), bits(want))
            _, db2 = o.act_bwd_bias(dy, y, act, need_g=False)
            g64 = dy.double() * (torch.where(y > 0, 1.0, y.double() + 1) if act == o.ACT_ELU else 1.0)
            case = f"{kind}, act {'elu' if act else 'none'}"
            _col_bar(t, case, db, g64.sum(0), g64.abs().sum(0))
            if not same:
                t.failures.append(f"{case}: g is not bit-identical to fp32 torch")
            if not torch.equal(bits(db2), bits(db)):
                t.failures.append(f"{case}: need_g=False changes dbias")
            del g64, gg, want
    t.check()


def test_act_bwd_bias_column_slices():
    """y and dy as column slices of wider buffers (row stride > F) give what the contiguous call gives, through
    ops and through the registered operator."""
    o = ops()
    import pangnn_b200.torch_ops  # noqa: F401  (registers torch.ops.pangnn)
    g = gen("act_bwd_slices")
    N, F = 10_001, 64
    wide_y = elu_rows(N, 2 * F + 4, g)
    wide_dy = torch.randn(N, 2 * F + 4, generator=g, device=DEV)
    y, dy = wide_y[:, 4:4 + F], wide_dy[:, F:2 * F]
    g0, db0 = o.act_bwd_bias(dy.contiguous(), y.contiguous(), o.ACT_ELU)
    for name, fn in (("ops", o.act_bwd_bias), ("torch.ops.pangnn", torch.ops.pangnn.act_bwd_bias)):
        for yy, dd in ((y, dy), (y, dy.contiguous()), (y.contiguous(), dy)):
            g1, db1 = fn(dd, yy, o.ACT_ELU)
            assert torch.equal(bits(g1), bits(g0)) and torch.equal(bits(db1), bits(db0)), \
                f"{name}: g off by {scale_err(g1, g0.double()):.2e}, dbias by {scale_err(db1, db0.double()):.2e}"


def elu_rows(N, W, g):
    return tnf.elu(torch.randn(N, W, generator=g, device=DEV) * 2)


def test_act_bwd_bias_misaligned_base():
    """A dense operand whose base is not 16-byte aligned is copied by the wrapper, not handed to the float4 loads."""
    o = ops()
    g = gen("act_bwd_misaligned")
    N, F = 5003, 128
    flat_y = elu_rows(1, N * F + 4, g).view(-1)
    flat_dy = torch.randn(N * F + 4, generator=g, device=DEV)
    y, dy = flat_y[1:1 + N * F].view(N, F), flat_dy[3:3 + N * F].view(N, F)
    assert y.data_ptr() % 16 and dy.data_ptr() % 16
    g0, db0 = o.act_bwd_bias(dy.clone(), y.clone(), o.ACT_ELU)
    g1, db1 = o.act_bwd_bias(dy, y, o.ACT_ELU)
    assert torch.equal(bits(g1), bits(g0)) and torch.equal(bits(db1), bits(db0))


# ------------------------------------------------------------------------------------------------
# C. halo kernels on one GPU (node_linear push epilogue, halo_p2p.cu)
# ------------------------------------------------------------------------------------------------
def three_way_push_maps(g):
    """Push maps of a three-rank genome partition, built as HaloPlan.push_maps builds them: 30 genomes of 1000
    genes, edges between nearby genomes, ``balanced_bounds`` split.  -> (own sizes, ext sizes, maps) where
    maps[s] = [(peer, slot_map int32[own_s], lo, hi)]: the middle rank pushes to two peers, each end rank to one."""
    from pangnn_b200.dist import balanced_bounds, local_numbering
    N, world = 30_000, 3
    src = torch.randint(0, N, (200_000,), generator=g, device=DEV)
    dst = (src + torch.randint(-4000, 4001, src.shape, generator=g, device=DEV)).clamp(0, N - 1)
    ei = torch.stack((src, dst))
    bounds = balanced_bounds(N, world, 1000)
    own = [bounds[r + 1] - bounds[r] for r in range(world)]
    halo = [local_numbering(ei, bounds[r], bounds[r + 1], "dst")[1] for r in range(world)]
    need = [[int(((h >= bounds[o]) & (h < bounds[o + 1])).sum()) for o in range(world)] for h in halo]  # [r][o]
    maps = []
    for s in range(world):
        ms = []
        for p in range(world):
            if p == s or need[p][s] == 0:
                continue
            h = halo[p]
            rows = h[(h >= bounds[s]) & (h < bounds[s + 1])] - bounds[s]
            slot0 = own[p] + sum(need[p][:s])
            m = torch.full((own[s],), -1, dtype=torch.int32, device=DEV)
            m[rows] = torch.arange(slot0, slot0 + rows.numel(), dtype=torch.int32, device=DEV)
            ms.append((p, m, int(rows.min()), int(rows.max()) + 1))
        maps.append(ms)
    ext = [own[r] + halo[r].numel() for r in range(world)]
    return own, ext, maps


def c3_push_maps(g):
    """One rank of 1e6 rows that pushes 1e5 rows at each end, with unmapped rows inside both [lo, hi)."""
    M, H, win = 1_000_000, 100_000, 150_000
    ext = M + 2 * H
    maps = []
    for p, base, slot0 in ((0, 0, M), (2, M - win, M + H)):
        rows = base + torch.sort(torch.randperm(win, generator=g, device=DEV)[:H]).values
        m = torch.full((M,), -1, dtype=torch.int32, device=DEV)
        m[rows] = torch.arange(slot0, slot0 + H, dtype=torch.int32, device=DEV)
        maps.append((p, m, int(rows.min()), int(rows.max()) + 1))
    return [None, M, None], {0: ext, 2: ext}, maps


@pytest.mark.parametrize("n,k", SHAPES)
@pytest.mark.parametrize("case", ["rank0", "rank1", "rank2", "c3"])
def test_node_linear_push_is_bit_exact(case, n, k):
    """node_linear with the fused halo push (bias + ELU, output row stride > n): ``out`` is bit-identical to the
    call without push; every mapped peer row is its source row of ``out``; every other peer element -- unmapped
    rows inside [lo, hi) and the padding columns included -- keeps its NaN-payload fill."""
    o = ops()
    g = gen("push", case, n, k)
    if case == "c3":
        own, ext, maps = c3_push_maps(g)
        M = own[1]
    else:
        r = int(case[-1])
        own, ext, all_maps = three_way_push_maps(g)
        M, maps = own[r], all_maps[r]
        ext = {p: ext[p] for p, *_ in maps}
    assert len(maps) == (2 if case in ("rank1", "c3") else 1) and M % 128
    ld = n + 8
    x = torch.randn(M, k, generator=g, device=DEV) * 2
    w = torch.randn(n, k, generator=g, device=DEV) / k ** 0.5
    bias = torch.randn(n, generator=g, device=DEV) * 0.5
    out_buf = nan_fill(M, ld)
    out_fill = bits(out_buf).clone()
    peers = {p: nan_fill(ext[p], ld) for p, *_ in maps}
    fills = {p: bits(b).clone() for p, b in peers.items()}
    push = [(m, peers[p][:, :n], lo, hi) for p, m, lo, hi in maps]
    o.node_linear(x, w, bias, o.ACT_ELU, out=out_buf[:, :n], push=push)
    ref = o.node_linear(x, w, bias, o.ACT_ELU)
    t = Table(f"node_linear push, {case}: M = {M}, n = {n}, k = {k}", ["pushed", "unmapped<hi"])
    out = out_buf[:, :n]
    if not torch.equal(bits(out), bits(ref)):
        t.failures.append("out differs from the call without push")
    if not torch.equal(bits(out_buf)[:, n:], out_fill[:, n:]):
        t.failures.append("padding of out written")
    for p, m, lo, hi in maps:
        src = torch.nonzero(m >= 0).squeeze(1)
        want = fills[p].clone()
        want[m[src].long(), :n] = bits(out)[src]
        holes = int((m[lo:hi] < 0).sum())
        ok = torch.equal(bits(peers[p]), want)
        t.add(f"peer {p}", src.numel(), holes, ok=ok, why=f"peer {p} buffer differs from the expected pushes")
    assert all(int((m[lo:hi] < 0).sum()) > 0 for _, m, lo, hi in maps), "no unmapped row inside [lo, hi)"
    t.check()


@pytest.mark.parametrize("F", [4, 64, 128, 256])
@pytest.mark.parametrize("n", [0, 1003])
@pytest.mark.parametrize("with_idx", [True, False])
def test_rows_gather_copy_is_bit_exact(with_idx, n, F):
    """dst[k] = src[idx[k]] (or src[k]) with row strides > F on both sides; nothing else of dst changes."""
    o = ops()
    g = gen("gather", with_idx, n, F)
    R = 2000
    src = torch.randn(R, F + 12, generator=g, device=DEV)[:, :F]
    dst_buf = nan_fill(n, F + 8)
    dst = dst_buf[:, 4:4 + F]
    idx = torch.randint(0, R, (n,), generator=g, device=DEV, dtype=torch.int32) if with_idx else None
    want = bits(dst_buf).clone()
    want[:, 4:4 + F] = bits(src[idx.long()] if with_idx else src[:n])
    o.rows_gather_copy(src, idx, dst)
    assert torch.equal(bits(dst_buf), want)


@pytest.mark.parametrize("F", [4, 64, 128, 256])
def test_rows_scatter_add_is_bit_exact(F):
    """dst[idx[k]] += src[k] with unique indices is one fp32 add per element: bit-exact to index_add_; three
    'peers' applied in rank order are bit-exact to the same sequence in torch."""
    o = ops()
    g = gen("scatter", F)
    R = 5000
    dst = torch.randn(R, F + 8, generator=g, device=DEV)[:, :F]
    want = dst.clone()
    for peer in range(3):
        n = (1200, 0, 3001)[peer]
        src = torch.randn(n, F + 4, generator=g, device=DEV)[:, :F] * 10 ** peer
        idx = torch.randperm(R, generator=g, device=DEV)[:n].to(torch.int32)
        o.rows_scatter_add(src, idx, dst)
        want.index_add_(0, idx.long(), src)
        assert torch.equal(bits(dst), bits(want)), f"after peer {peer}"


# ------------------------------------------------------------------------------------------------
# D. tensor-core GEMMs at the shapes of the step
# ------------------------------------------------------------------------------------------------
def _tn_operands(kind, R, M, K, g):
    if kind == "randn":
        return torch.randn(R, M, generator=g, device=DEV), torch.randn(R, K, generator=g, device=DEV)
    # one-signed: ELU-output-like A (shifted to >= 0) against a positive B -- the truncating accumulator drifts
    return (tnf.elu(torch.randn(R, M, generator=g, device=DEV)) + 1.0,
            torch.rand(R, K, generator=g, device=DEV))


def _tn_case(t, case, a, b, one_signed):
    o = ops()
    l0 = o.LAUNCHES["count"]
    got = o.gemm_tn(a, b)
    assert o.LAUNCHES["count"] == l0 + 2, "the tensor-core kernel must be the path taken"
    ref = a.double().t() @ b.double()
    with plain_fp32():
        e32 = scale_err(a.t() @ b, ref)
    e = scale_err(got, ref)
    bar = TN_DRIFT if one_signed else min(TN_DRIFT, max(TN_FP32 * e32, SCALE_REL / 5))
    t.add(case, e, e32, ok=e <= SCALE_REL and e <= bar,
          why=f"e {e:.2e} (cuBLAS fp32 {e32:.2e}; bars {SCALE_REL:.0e}, {bar:.2e})")


@pytest.mark.parametrize("tiles", [15, 16, 17, 32, 33])
@pytest.mark.parametrize("M,K", SHAPES)
def test_gemm_tn_chain_boundaries(M, K, tiles):
    """R = 32 * 148 * c * tiles + d: with c CTAs per SM (3 for every shape, so c = 3 gives each CTA exactly
    ``tiles`` tiles) the per-CTA chain is cut at kFlush = 16 tiles just before, at and after the cut."""
    g = gen("gemm_tn", M, K, tiles)
    t = Table(f"gemm_tn, M = {M}, K = {K}, {tiles} tiles per CTA at c = 3", ["scale err", "cuBLAS fp32"])
    for c in (1, 2, 3):
        for d in (-1, 0, 1):
            R = 32 * NUM_SMS * c * tiles + d
            for kind in ("randn", "one-signed"):
                a, b = _tn_operands(kind, R, M, K, g)
                _tn_case(t, f"c {c}, d {d:+d}, {kind}", a, b, kind == "one-signed")
    t.check()


@pytest.mark.parametrize("M,K", SHAPES)
def test_gemm_tn_million_rows_and_layouts(M, K):
    """R = 1e6 (about 70 tiles per CTA: five chains), column slices of wider operands, and a base that is not
    16-byte aligned, which must reach the library GEMM instead of the kernel's alignment check."""
    o = ops()
    g = gen("gemm_tn_1e6", M, K)
    R = 1_000_000
    t = Table(f"gemm_tn, M = {M}, K = {K}, R = {R}", ["scale err", "cuBLAS fp32"])
    for kind in ("randn", "one-signed"):
        a, b = _tn_operands(kind, R, M, K, g)
        _tn_case(t, kind, a, b, kind == "one-signed")
    wa = torch.randn(R, 2 * M, generator=g, device=DEV)
    wb = torch.randn(R, K + 4, generator=g, device=DEV)
    _tn_case(t, "strided A and B", wa[:, M:], wb[:, 4:], False)
    t.check()
    for a, b in ((wa[:, 1:1 + M], b), (a, wb[:, 1:1 + K])):        # row strides % 4 == 0, base + 4 bytes
        assert a.stride(0) % 4 == 0 and b.stride(0) % 4 == 0 and (a.data_ptr() % 16 or b.data_ptr() % 16)
        l0 = o.LAUNCHES["count"]
        got = o.gemm_tn(a, b)
        assert o.LAUNCHES["count"] == l0, "a misaligned base must not reach the kernel"
        assert scale_err(got, a.double().t() @ b.double()) <= SCALE_REL


NL_M = sorted({128 * (NUM_SMS * t + r) + d for t in (1, 2, 5) for r in (0, 1, 147) for d in (0, 1)}) + [1_000_000]


@pytest.mark.parametrize("w_is_kn", [False, True])
@pytest.mark.parametrize("n,k", SHAPES)
def test_node_linear_tile_schedule(n, k, w_is_kn):
    """M = 128 (148 t + r) + d: 1, 2 or 5 tiles per persistent CTA with r CTAs taking one more, both parities of
    the ring and the accumulator ping-pong, a partial last tile; then 1e6 rows.  ELU with pre-activations across 0
    and far below it."""
    o = ops()
    g = gen("nl", n, k, w_is_kn)
    t = Table(f"node_linear, n = {n}, k = {k}, w_is_kn = {w_is_kn}", ["scale err", "el err/bar"])
    w = torch.randn((k, n) if w_is_kn else (n, k), generator=g, device=DEV) / k ** 0.5
    w64 = w.double() if w_is_kn else w.double().t()
    bias = torch.randn(n, generator=g, device=DEV) * 0.5
    for M in NL_M:
        x = torch.randn(M, k, generator=g, device=DEV) * (torch.rand(M, 1, generator=g, device=DEV) * 3)
        x[::5] *= 10                                                     # pre-activations far below -20
        x64 = x.double()
        rowscale = (x64.abs() @ w64.abs() + bias.double().abs()).max(dim=1, keepdim=True).values
        for bb, act in ((None, o.ACT_NONE), (bias, o.ACT_ELU)):
            l0 = o.LAUNCHES["count"]
            y = o.node_linear(x, w, bb, act, w_is_kn=w_is_kn)
            assert o.LAUNCHES["count"] == l0 + 1, "the tensor-core kernel must be the path taken"
            pre = x64 @ w64 + (bb.double() if bb is not None else 0.0)
            ref = torch.where(pre > 0, pre, torch.expm1(pre)) if act == o.ACT_ELU else pre
            e = scale_err(y, ref)
            r = ratio((y.double() - ref).abs(), NL_SCALE * rowscale + NL_ABS)
            t.add(f"M {M}, act {'elu' if act else 'none'}", e, r, ok=e <= NL_SCALE and r <= 1.0,
                  why=f"scale-relative {e:.2e}, element-wise {r:.2f} x bar")
            del pre, ref, y
        del x, x64, rowscale
    t.check()
