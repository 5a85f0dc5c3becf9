"""Tensor-level wrappers over the C ABI (``include/pangnn_b200.h``) and their autograd glue.

PyTorch is plumbing here: it owns device memory and streams; every kernel on the hot path is ours,
reached through ctypes.  The node GEMMs (K3 in SURVEY.md §2b: ``X @ W^T`` at N x 64..128) are
our tcgen05 3xTF32 kernel (``node_linear``); only shapes outside {64,128}^2 reach the library GEMM.
No fallback: a tensor that is not on a CUDA device raises.
"""
import ctypes as C
from collections import OrderedDict, namedtuple

import torch

from . import _abi

ACT_NONE, ACT_ELU = 0, 1
SCORER_D = 64
NGRADS = 64 * 64 + 64 + 64 + 1 + 64 + 64

# kernel-launch accounting for bench.py ("gpu_launches")
LAUNCHES = {"count": 0}


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _abi.PangnnError("pangnn_b200 ops need CUDA tensors (there is no CPU path)")


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _alias(buf, shape, stride=()):
    """A fresh tensor of ``shape`` (row-major unless ``stride`` is given) over the memory of a persistent buffer,
    from its first element, that is NOT a view of it as far as autograd is concerned: the buffers are reused every
    step, and an in-place (mark_dirty) custom function on a view, or an output that is a view of an input, would
    tie the history of the shared base tensor to unrelated sites and steps."""
    return torch.empty(0, dtype=buf.dtype, device=buf.device).set_(buf.untyped_storage(), buf.storage_offset(),
                                                                   tuple(map(int, shape)), tuple(stride))


# ------------------------------------------------------------------------------------------------
# primitives
# ------------------------------------------------------------------------------------------------
def sort_pairs_u64(keys, vals=None, key_bits=64):
    """Stable LSD radix sort of (int64-viewed-as-u64 keys, int32 vals)."""
    lib = _abi.load()
    _need_cuda(keys, vals)
    n = keys.numel()
    keys = keys.contiguous()
    out_k = torch.empty_like(keys)
    out_v = torch.empty(n, dtype=torch.int32, device=keys.device)
    ws = _ws(lib.pangnn_sort_pairs_workspace_bytes(n), keys.device)
    _abi.check(lib.pangnn_sort_pairs_u64(_p(keys), _p(vals), _p(out_k), _p(out_v), n, key_bits,
                                         _p(ws), ws.numel(), _stream()), "sort_pairs_u64")
    LAUNCHES["count"] += 3 * ((key_bits + 7) // 8)
    return out_k, out_v


def exclusive_scan_u32(x):
    lib = _abi.load()
    _need_cuda(x)
    n = x.numel()
    out = torch.empty_like(x)
    total = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws = _ws(lib.pangnn_scan_workspace_bytes(n), x.device)
    _abi.check(lib.pangnn_exclusive_scan_u32(_p(x), _p(out), n, _p(total), _p(ws), ws.numel(),
                                             _stream()), "exclusive_scan_u32")
    LAUNCHES["count"] += 1
    return out, total


class CSR:
    """One orientation of a graph: ``rowptr`` int64 [N+1], ``col`` int32 [E], ``perm`` int32 [E]
    (CSR slot -> position in the original edge list)."""
    __slots__ = ("rowptr", "col", "perm", "num_rows", "num_edges", "by_dst", "identity_perm")

    def __init__(self, rowptr, col, perm, num_rows, num_edges, by_dst, identity_perm=False):
        self.rowptr, self.col, self.perm = rowptr, col, perm
        self.num_rows, self.num_edges, self.by_dst = num_rows, num_edges, by_dst
        self.identity_perm = identity_perm            # slot i IS edge i (lists that arrive in this CSR's order)


SMALL_CSR_EDGES = 4096        # single-launch CSR build below this size (sort_scan.cu: kSmallCsrMaxE)


def csr_build(edge_index, num_nodes, by_dst=True):
    """COO int64 ``edge_index`` [2,E] -> CSR (rows = destinations if ``by_dst`` else sources)."""
    lib = _abi.load()
    _need_cuda(edge_index)
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise _abi.PangnnError("edge_index must be an int64 tensor of shape [2, E]")
    ei = edge_index.contiguous()
    E, dev = ei.size(1), ei.device
    rowptr = torch.empty(num_nodes + 1, dtype=torch.int64, device=dev)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    perm = torch.empty(E, dtype=torch.int32, device=dev)
    ws = _ws(lib.pangnn_csr_build_workspace_bytes(E), dev)
    _abi.check(lib.pangnn_csr_build(_p(ei), E, num_nodes, 1 if by_dst else 0, _p(rowptr), _p(col),
                                    _p(perm), _p(ws), ws.numel(), _stream()), "csr_build")
    LAUNCHES["count"] += 1 if E <= SMALL_CSR_EDGES else 2 + 3 * _csr_passes(num_nodes, True)
    return CSR(rowptr, col, perm, num_nodes, E, by_dst)


def _csr_passes(num_nodes, both_halves):
    nbits = max(1, (max(num_nodes, 2) - 1).bit_length())
    return ((2 * nbits if both_halves else nbits) + 7) // 8


def csr_from_sorted(edge_index, num_nodes):
    """By-source CSR of an edge list in canonical (src, dst) order, or None when the list is not sorted (one
    check kernel + a 4-byte read; no radix sort)."""
    lib = _abi.load()
    ei = edge_index.contiguous()
    E, dev = ei.size(1), ei.device
    flag = torch.empty(1, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_edges_sorted(_p(ei), E, num_nodes, _p(flag), _stream()), "edges_sorted")
    LAUNCHES["count"] += 1
    flags = int(flag.item())
    if flags & 2:                                        # torch's index ops would raise on such a list
        raise _abi.PangnnError(f"edge_index holds node ids outside [0, {num_nodes})")
    if flags & 1:
        return None
    rowptr = torch.empty(num_nodes + 1, dtype=torch.int64, device=dev)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    perm = torch.empty(E, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_csr_from_sorted(_p(ei), E, num_nodes, _p(rowptr), _p(col), _p(perm), _stream()),
               "csr_from_sorted")
    LAUNCHES["count"] += 1
    return CSR(rowptr, col, perm, num_nodes, E, False, identity_perm=True)


def csr_transpose(csr):
    """CSR of the other orientation from an existing one: same result as ``csr_build`` with ``by_dst``
    flipped (canonical order, same perm) in half the radix passes."""
    lib = _abi.load()
    E, N, dev = csr.num_edges, csr.num_rows, csr.rowptr.device
    rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    perm = torch.empty(E, dtype=torch.int32, device=dev)
    ws = _ws(lib.pangnn_csr_build_workspace_bytes(E), dev)
    _abi.check(lib.pangnn_csr_transpose(_p(csr.rowptr), _p(csr.col), _p(csr.perm), E, N, _p(rowptr), _p(col),
                                        _p(perm), _p(ws), ws.numel(), _stream()), "csr_transpose")
    LAUNCHES["count"] += 2 + 3 * _csr_passes(N, False)
    return CSR(rowptr, col, perm, N, E, not csr.by_dst)


def csr_merge_band(csr, n):
    """CSR of the whole-graph union list ``[sim ; band(n)]`` from the CSR of the sim edges (one merge kernel,
    no sort of the union list); equals ``csr_build`` of the concatenated list."""
    lib = _abi.load()
    E, N, dev = csr.num_edges, csr.num_rows, csr.rowptr.device
    eu = E + int(lib.pangnn_neighbour_band_edges(N, int(n)))
    rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
    col = torch.empty(eu, dtype=torch.int32, device=dev)
    perm = torch.empty(eu, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_csr_merge_band(_p(csr.rowptr), _p(csr.col), _p(csr.perm), E, N, int(n),
                                         1 if csr.by_dst else 0, _p(rowptr), _p(col), _p(perm), _stream()),
               "csr_merge_band")
    LAUNCHES["count"] += 1
    return CSR(rowptr, col, perm, N, eu, csr.by_dst)


def gcn_norm(csr_dst, weight):
    """-> (dis [N], val [E] in ``csr_dst`` order).  ``weight`` in original edge order or None."""
    lib = _abi.load()
    dev = csr_dst.rowptr.device
    if weight is not None:
        _need_cuda(weight)
        weight = weight.contiguous().float()
    dis = torch.empty(csr_dst.num_rows, dtype=torch.float32, device=dev)
    val = torch.empty(csr_dst.num_edges, dtype=torch.float32, device=dev)
    _abi.check(lib.pangnn_gcn_norm(_p(csr_dst.rowptr), _p(csr_dst.col), _p(csr_dst.perm), _p(weight),
                                   csr_dst.num_rows, _p(dis), _p(val), _stream()), "gcn_norm")
    LAUNCHES["count"] += 2
    return dis, val


def gcn_norm_apply(csr, weight, dis):
    lib = _abi.load()
    if weight is not None:
        weight = weight.contiguous().float()
    val = torch.empty(csr.num_edges, dtype=torch.float32, device=dis.device)
    _abi.check(lib.pangnn_gcn_norm_apply(_p(csr.rowptr), _p(csr.col), _p(csr.perm), _p(weight), _p(dis),
                                         csr.num_rows, 1 if csr.by_dst else 0, _p(val), _stream()),
               "gcn_norm_apply")
    LAUNCHES["count"] += 1
    return val


def gcn_aggregate(rowptr, col, val, x, num_rows, bias=None, act=ACT_NONE, out=None):
    """``out[i] = act(sum_{e in row i} val_e * x[col_e] + bias)``; ``x``/``out`` may be column
    slices of wider row-major matrices (row stride is honoured)."""
    lib = _abi.load()
    _need_cuda(x)
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise _abi.PangnnError("x must be a float32 [rows, F] tensor with unit column stride")
    F = x.size(1)
    if out is None:
        out = torch.empty(num_rows, F, dtype=torch.float32, device=x.device)
    elif out.stride(1) != 1 or out.size(1) != F or out.size(0) != num_rows:
        raise _abi.PangnnError("bad output tensor")
    _abi.check(lib.pangnn_gcn_aggregate(_p(rowptr), _p(col), _p(val), _p(x), x.stride(0), num_rows, F,
                                        _p(bias), act, _p(out), out.stride(0), _stream()),
               "gcn_aggregate")
    LAUNCHES["count"] += 1
    return out


def aggregate(gs, ent, x, by_dst, bias=None, act=ACT_NONE, out=None):
    """``A_hat x`` (``by_dst``) or ``A_hat^T x`` over the structure ``gs`` with the normalisation ``ent`` (=
    ``gs.norm(weight, need_src=not by_dst)``)."""
    csr = gs.dst if by_dst else gs.src
    return gcn_aggregate(csr.rowptr, csr.col, ent["dst" if by_dst else "src"], x, gs.num_nodes, bias, act, out)


def segment_sum_edges(csr, rows, num_rows, out):
    """``out[i] = sum of the per-edge ``rows`` of CSR row i`` (the scorer's per-edge gradients back to the nodes).
    A list that arrived in this CSR's order needs no gather: its rows are consecutive (identity columns)."""
    col = None if (csr.identity_perm and rows.size(1) in (32, 64, 128)) else csr.perm
    return gcn_aggregate(csr.rowptr, col, None, rows, num_rows, out=out)


# ------------------------------------------------------------------------------------------------
# scored edges in chunks (SURVEY §8e / DESIGN §6b: the per-edge spill da1 [E, 64] of a pan-genome-scale partition
# does not fit; every sum over edges is linear, so the scorer runs over fixed-size runs of source rows and the node
# gradients are accumulated across them)
# ------------------------------------------------------------------------------------------------
SCORER_CHUNK_EDGES = {"n": 1 << 26}       # edges per scorer launch above which the chunked form is used (17 GB of da1)


def scored_chunk_runs(rowptr, max_edges):
    """Greedy split of the rows of a CSR (host ``rowptr``, numpy int64 [N+1]) into runs of consecutive rows with at most
    ``max_edges`` entries each (a single row longer than that is a run of its own): ``[(r0, r1, c0, c1), ...]`` =
    rows [r0, r1), entries [c0, c1); empty runs are dropped.  Pure host arithmetic (unit-tested without a GPU)."""
    import numpy as np
    rowptr = np.asarray(rowptr, dtype=np.int64)
    N, runs, r0 = rowptr.size - 1, [], 0
    max_edges = max(int(max_edges), 1)
    while r0 < N:
        # largest r1 with rowptr[r1] - rowptr[r0] <= max_edges, at least one row
        r1 = int(np.searchsorted(rowptr, rowptr[r0] + max_edges, side="right")) - 1
        r1 = min(max(r1, r0 + 1), N)
        if rowptr[r1] > rowptr[r0]:
            runs.append((r0, r1, int(rowptr[r0]), int(rowptr[r1])))
        r0 = r1
    return runs


class ScoredChunks:
    """Runs of consecutive SOURCE rows of a canonically ordered scored-edge list with at most ``max_edges`` edges
    each (``scored_chunk_runs``), each with the by-destination CSR of its own edges (``perm`` = position inside the
    chunk).  Built once per structure (one device -> host copy of the row offsets, one sort per chunk)."""

    def __init__(self, gs, max_edges):
        src = gs.src
        if not src.identity_perm:
            raise _abi.PangnnError("the chunked scorer needs the scored edges in canonical (src, dst) order")
        self.runs = scored_chunk_runs(src.rowptr.cpu().numpy(), max_edges)
        self.max_edges = max((c1 - c0 for _, _, c0, c1 in self.runs), default=0)
        self.csr_dst = []
        for (_, _, c0, c1) in self.runs:
            csr = csr_build(gs.edge_index[:, c0:c1].contiguous(), gs.num_nodes, by_dst=True)
            csr.col = None                                       # only rowptr + perm are used (segment sums)
            self.csr_dst.append(csr)


def scored_chunks(gs, max_edges):
    key = ("chunks", int(max_edges))
    ent = gs._norm.get(key)
    if ent is None:
        ent = gs._norm[key] = {"chunks": ScoredChunks(gs, int(max_edges))}
    return ent["chunks"]


def _rows16(t):
    """``t`` as dense rows from a 16-byte aligned base (the row kernels read float4 at ``base + r * F``)."""
    if t is None:
        return None
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def act_bwd_bias(dy, y, act, need_g=True):
    """-> (g = dy * act'(y), dbias = column sums of g)."""
    lib = _abi.load()
    dy, y = _rows16(dy), _rows16(y)
    rows, F = dy.shape
    g = torch.empty_like(dy) if (need_g and act != ACT_NONE) else None
    dbias = torch.empty(F, dtype=torch.float32, device=dy.device)
    ws = _ws(lib.pangnn_act_bwd_bias_workspace_bytes(rows, F), dy.device)
    _abi.check(lib.pangnn_act_bwd_bias(_p(dy), _p(y), rows, F, act, _p(g), _p(dbias), _p(ws),
                                       ws.numel(), _stream()), "act_bwd_bias")
    LAUNCHES["count"] += 2
    return (g if g is not None else dy), dbias


def gemm_tn(a, b):
    """``a.t() @ b`` for tall-skinny operands ([N,M], [N,K], M,K in {64,128}) with our deterministic
    streaming kernel; other shapes and layouts (row strides or bases that are not 16-byte aligned) go to the
    library GEMM."""
    M, K = a.size(1), b.size(1)
    if (M not in (64, 128) or K not in (64, 128) or a.stride(1) != 1 or b.stride(1) != 1
            or a.stride(0) % 4 or b.stride(0) % 4 or a.data_ptr() % 16 or b.data_ptr() % 16
            or a.dtype != torch.float32):
        return torch.mm(a.t(), b)
    lib = _abi.load()
    N = a.size(0)
    c = torch.empty(M, K, dtype=torch.float32, device=a.device)
    ws = _ws(lib.pangnn_gemm_tn_workspace_bytes(N, M, K), a.device)
    _abi.check(lib.pangnn_gemm_tn(_p(a), a.stride(0), _p(b), b.stride(0), N, M, K, _p(c), _p(ws),
                                  ws.numel(), _stream()), "gemm_tn")
    LAUNCHES["count"] += 2
    return c


def _tc_shape(t, w_rows, w_cols):
    return (t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 4 == 0
            and t.data_ptr() % 16 == 0 and w_rows in (64, 128) and w_cols in (64, 128))


def node_linear(x, w, bias=None, act=ACT_NONE, w_is_kn=False, out=None, push=None):
    """``act(x @ w.T + bias)`` (``w`` [n, k]) or ``act(x @ w + bias)`` (``w`` [k, n], ``w_is_kn``) on the
    tcgen05 tensor cores with the 3xTF32 split (fp32-grade).  Shapes outside n, k in {64, 128} (the
    1-wide embedding, odd --node_dim values) go to the library GEMM."""
    _need_cuda(x, w)
    k = w.size(0) if w_is_kn else w.size(1)
    n = w.size(1) if w_is_kn else w.size(0)
    if not _tc_shape(x, n, k) or x.size(1) != k or w.stride(1) != 1 or (bias is not None and bias.data_ptr() % 16):
        if push is not None:
            raise _abi.PangnnError("the fused halo push needs the tensor-core shapes (n, k in {64, 128})")
        y = torch.mm(x, w if w_is_kn else w.t())
        if bias is not None:
            y += bias
        if act == ACT_ELU:
            torch.nn.functional.elu_(y)
        if out is not None:
            out.copy_(y)
            return out
        return y
    lib = _abi.load()
    M = x.size(0)
    if out is None:
        out = torch.empty(M, n, dtype=torch.float32, device=x.device)
    if push is None:
        _abi.check(lib.pangnn_node_linear(_p(x), x.stride(0), M, k, _p(w), w.stride(0), 1 if w_is_kn else 0, n,
                                          _p(bias), act, _p(out), out.stride(0), _stream()), "node_linear")
    else:
        # push = [(slot_map int32[M], peer tensor with the row stride of `out`, lo, hi), ...] (at most two peers)
        (s0, p0, lo0, hi0), (s1, p1, lo1, hi1) = (list(push) + [(None, None, 0, 0), (None, None, 0, 0)])[:2]
        for pt in (p0, p1):
            if pt is not None and pt.stride(0) != out.stride(0):
                raise _abi.PangnnError("peer buffers must have the row stride of the output")
        _abi.check(lib.pangnn_node_linear_push(_p(x), x.stride(0), M, k, _p(w), w.stride(0), 1 if w_is_kn else 0, n,
                                               _p(bias), act, _p(out), out.stride(0), _p(s0), _p(p0), lo0, hi0,
                                               _p(s1), _p(p1), lo1, hi1, _stream()), "node_linear_push")
    LAUNCHES["count"] += 1
    return out


# ------------------------------------------------------------------------------------------------
# graph structure cache
# ------------------------------------------------------------------------------------------------
class GraphStruct:
    """Both CSR orientations of one ``edge_index`` plus int32 endpoint copies; gcn_norm values are
    cached per weight tensor.  The reference recomputes gcn_norm on every GCNConv call
    (``cached=False``); here structure and norm are built once per distinct (edge_index, weight)."""

    def __init__(self, edge_index, num_nodes):
        self.edge_index = edge_index                  # keeps the storage alive (cache key safety)
        self.num_nodes = num_nodes
        self.num_edges = edge_index.size(1)
        self._src = None
        if self.num_edges > SMALL_CSR_EDGES and edge_index.dtype == torch.int64 and edge_index.dim() == 2:
            # canonical (src, dst) order (every table of this package's preprocessing): no sort for the
            # by-source orientation, 3-pass transpose for the other one
            self._src = csr_from_sorted(edge_index, num_nodes)
        self._dst = csr_transpose(self._src) if self._src is not None else csr_build(edge_index, num_nodes, by_dst=True)
        self._ends = None
        self._norm = OrderedDict()
        self._ready = None                            # event of a side stream that built this structure

    def built_on(self, stream, user_stream):
        """Mark everything built so far as produced on ``stream`` (a side stream) for use on ``user_stream``:
        the first use waits for it (``AlternateGCN.prepare`` builds the scored-edge structure beside the step)."""
        ev = torch.cuda.Event()
        ev.record(stream)
        self._ready = ev
        for t in (self._dst, self._src):
            if t is not None:
                for a in (t.rowptr, t.col, t.perm):
                    a.record_stream(user_stream)
        if self._ends is not None:
            for a in self._ends:
                a.record_stream(user_stream)
        for ent in self._norm.values():                       # gcn_norm / rank-1 vectors precomputed by prepare()
            for v in ent.values():
                for a in (v if isinstance(v, tuple) else (v,)):
                    if torch.is_tensor(a) and a.is_cuda:
                        a.record_stream(user_stream)
        return self

    def _sync(self):
        if self._ready is not None:
            torch.cuda.current_stream().wait_event(self._ready)
            self._ready = None

    @property
    def dst(self):
        self._sync()
        return self._dst

    @property
    def src(self):
        self._sync()
        if self._src is None:
            if self.num_edges <= SMALL_CSR_EDGES:             # one single-CTA launch either way
                self._src = csr_build(self.edge_index, self.num_nodes, by_dst=False)
            else:
                self._src = csr_transpose(self._dst)
        return self._src

    @property
    def endpoints32(self):
        self._sync()
        if self._ends is None:
            ei = self.edge_index.to(torch.int32).contiguous()
            self._ends = (ei[0], ei[1])
        return self._ends

    def norm(self, weight, need_src):
        key = None if weight is None else (weight.data_ptr(), weight._version, weight.numel())
        ent = self._norm.get(key)
        if ent is None:
            dis, val_dst = gcn_norm(self.dst, weight)
            # "w" keeps the weight tensor alive: the key holds its address (as _rank1_cached does for x)
            ent = {"w": weight, "dis": dis, "dst": val_dst, "src": None}
            self._norm[key] = ent
            while len(self._norm) > 4:
                self._norm.popitem(last=False)
        if need_src and ent["src"] is None:
            ent["src"] = gcn_norm_apply(self.src, weight, ent["dis"])
        return ent


_STRUCTS = OrderedDict()
_STRUCT_CAP = 8


def _struct_key(edge_index, num_nodes):
    return (edge_index.data_ptr(), edge_index._version, tuple(edge_index.shape),
            tuple(edge_index.stride()), num_nodes, edge_index.device.index)


def graph_struct_union(union_edge_index, num_nodes, sim, n):
    """Structure of a whole-graph union list ``[sim ; band(n)]`` (as ``union_index`` assembles it) derived from
    the structure ``sim`` of its scored edges: both CSR orientations by row-wise merge with the band instead
    of sorting the 1.7x longer union list.  Registered in the cache under ``union_edge_index``."""
    key = _struct_key(union_edge_index, num_nodes)
    gs = _STRUCTS.get(key)
    if gs is None:
        gs = object.__new__(GraphStruct)
        gs.edge_index, gs.num_nodes, gs.num_edges = union_edge_index, num_nodes, union_edge_index.size(1)
        gs._dst = csr_merge_band(sim.dst, n)
        gs._src = csr_merge_band(sim.src, n)
        gs._ends, gs._norm, gs._ready = None, OrderedDict(), None
        assert gs._dst.num_edges == gs.num_edges
        _STRUCTS[key] = gs
        while len(_STRUCTS) > _STRUCT_CAP:
            _STRUCTS.popitem(last=False)
    return gs


def graph_struct(edge_index, num_nodes):
    key = _struct_key(edge_index, num_nodes)
    gs = _STRUCTS.get(key)
    if gs is None:
        gs = GraphStruct(edge_index, num_nodes)
        _STRUCTS[key] = gs
        while len(_STRUCTS) > _STRUCT_CAP:
            _STRUCTS.popitem(last=False)
    else:
        _STRUCTS.move_to_end(key)
    return gs


def clear_cache():
    _STRUCTS.clear()


def cached_structs(graph):
    """The cached structures of a batch's edge lists (whichever of them exist)."""
    out = []
    n = graph.x.size(0)
    for name in ("edge_index", "union_edge_index", "neighbour_edge_index"):
        ei = getattr(graph, name, None)
        if ei is not None:
            gs = _STRUCTS.get(_struct_key(ei, n))
            if gs is not None:
                out.append(gs)
    return out


def drop_structs(graph):
    """Evict a batch's structures (a prefetching loader keeps two batches alive, not the LRU's eight)."""
    n = graph.x.size(0)
    for name in ("edge_index", "union_edge_index", "neighbour_edge_index"):
        ei = getattr(graph, name, None)
        if ei is not None:
            _STRUCTS.pop(_struct_key(ei, n), None)


# ------------------------------------------------------------------------------------------------
# autograd: one GCN layer  y = act( A_hat (x W^T) + b )
# ------------------------------------------------------------------------------------------------
class GCNLayerFn(torch.autograd.Function):
    """Transform-then-aggregate (the reference's order): y = act(A_hat (x W^T) + b).  Used when the
    layer does not widen (out <= in), so the gather runs at the narrower width."""

    @staticmethod
    def forward(ctx, x, weight, bias, gs, edge_weight, act):
        ent = gs.norm(edge_weight, need_src=False)
        h = node_linear(x, weight)                                      # K3: tcgen05 3xTF32
        y = aggregate(gs, ent, h, True, bias, act)
        ctx.gs, ctx.edge_weight, ctx.act = gs, edge_weight, act
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, weight, y if act != ACT_NONE else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, y = ctx.saved_tensors
        gs = ctx.gs
        ent = gs.norm(ctx.edge_weight, need_src=True)
        g, dbias = act_bwd_bias(dy, y, ctx.act)
        dh = aggregate(gs, ent, g, False)                                            # A_hat^T g
        dW = gemm_tn(dh, x) if ctx.needs_input_grad[1] else None
        dx = node_linear(dh, weight, w_is_kn=True) if ctx.needs_input_grad[0] else None
        return dx, dW, (dbias if ctx.has_bias and ctx.needs_input_grad[2] else None), None, None, None


class GCNLayerAggFirstFn(torch.autograd.Function):
    """Aggregate-then-transform: y = act((A_hat x) W^T + b) — the same linear map (A_hat (x W^T) =
    (A_hat x) W^T), chosen when the layer widens (in < out) so that the HBM/L2-bound gather moves
    rows of width `in` instead of `out` (half the bytes for conv_in, 64 -> 128)."""

    @staticmethod
    def forward(ctx, x, weight, bias, gs, edge_weight, act):
        ent = gs.norm(edge_weight, need_src=False)
        ax = aggregate(gs, ent, x, True)
        y = node_linear(ax, weight, bias, act)                          # bias + ELU in the GEMM epilogue
        ctx.gs, ctx.edge_weight, ctx.act = gs, edge_weight, act
        ctx.has_bias = bias is not None
        ctx.save_for_backward(ax, weight, y if act != ACT_NONE else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        ax, weight, y = ctx.saved_tensors
        gs = ctx.gs
        g, dbias = act_bwd_bias(dy, y, ctx.act)
        dW = gemm_tn(g, ax) if ctx.needs_input_grad[1] else None
        dx = None
        if ctx.needs_input_grad[0]:
            ent = gs.norm(ctx.edge_weight, need_src=True)
            dax = node_linear(g, weight, w_is_kn=True)
            dx = aggregate(gs, ent, dax, False)
        return dx, dW, (dbias if ctx.has_bias and ctx.needs_input_grad[2] else None), None, None, None


def rank1_vectors(csr_dst, val_dst, x, num_rows=None):
    """``a = A_hat x``, ``c = A_hat 1`` over the first ``num_rows`` rows of a normalised CSR (``x`` [n] or [n, 1])."""
    lib = _abi.load()
    n = csr_dst.num_rows if num_rows is None else int(num_rows)
    a = torch.empty(n, dtype=torch.float32, device=x.device)
    c = torch.empty(n, dtype=torch.float32, device=x.device)
    xs = x.reshape(-1).contiguous().float()
    _abi.check(lib.pangnn_csr_spmv2(_p(csr_dst.rowptr), _p(csr_dst.col), _p(val_dst), _p(xs), n, _p(a), _p(c),
                                    _stream()), "csr_spmv2")
    LAUNCHES["count"] += 1
    return a, c


class RankOneFn(torch.autograd.Function):
    """``y = act(a u^T + c v^T + b)`` with ``u = W w_e``, ``v = W b_e``: the embedding ``Linear(1, D)`` and the
    first ``GCNConv`` folded together (``rank1.cu``).  Forward is one streaming write of [N, F], backward one
    streaming read of (dY, Y) into three weighted column sums."""

    @staticmethod
    def forward(ctx, a, c, w_e, b_e, weight, bias, act):
        lib = _abi.load()
        N, F = a.numel(), weight.size(0)
        w_e1 = w_e.reshape(-1)
        u, v = torch.mv(weight, w_e1), torch.mv(weight, b_e)
        y = torch.empty(N, F, dtype=torch.float32, device=a.device)
        _abi.check(lib.pangnn_rank1_affine_act(_p(a), _p(c), _p(u), _p(v), _p(bias), N, F, act, _p(y), y.stride(0),
                                               _stream()), "rank1_affine_act")
        LAUNCHES["count"] += 1
        ctx.act, ctx.has_bias = act, bias is not None
        ctx.save_for_backward(a, c, y, w_e1, b_e, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _abi.load()
        a, c, y, w_e1, b_e, weight = ctx.saved_tensors
        N, F = y.shape
        dy = dy.contiguous()
        sums = torch.empty(3, F, dtype=torch.float32, device=y.device)
        ws = _ws(lib.pangnn_rank1_bwd_workspace_bytes(N, F), y.device)
        _abi.check(lib.pangnn_rank1_bwd(_p(dy), _p(y), _p(a), _p(c), N, F, ctx.act, _p(sums), _p(ws), ws.numel(),
                                        _stream()), "rank1_bwd")
        LAUNCHES["count"] += 2
        db, du, dv = sums[0], sums[1], sums[2]
        dW = torch.addr(torch.outer(du, w_e1), dv, b_e)                  # du w_e^T + dv b_e^T
        dw_e = torch.mv(weight.t(), du).unsqueeze(1)
        db_e = torch.mv(weight.t(), dv)
        return None, None, dw_e, db_e, dW, (db if ctx.has_bias else None), None


def _rank1_cached(gs, edge_weight, x):
    ent = gs.norm(edge_weight, need_src=False)
    key = ("rank1", x.data_ptr(), x._version)
    ac = ent.get(key)
    if ac is None:
        for k in [k for k in ent if isinstance(k, tuple) and k[0] == "rank1"]:
            del ent[k]
        ac = ent[key] = rank1_vectors(gs.dst, ent["dst"], x) + (x,)     # x kept alive: the key holds its address
    return ac[0], ac[1]


def embed_conv(x, w_e, b_e, weight, bias, edge_index, edge_weight=None, act=ACT_NONE):
    """``act(GCNConv(Linear(1, D)(x)))`` for scalar node features ``x`` [N, 1] (``src/gnn.py:97,125`` followed by
    the first convolution, ``:129 / :135 / :147``) as one rank-2 update: ``a = A_hat x`` and ``c = A_hat 1`` are
    cached with gcn_norm.  Same parameters, same values (to fp32 rounding) as the two modules."""
    _need_cuda(x, weight, edge_index)
    if x.requires_grad:
        raise _abi.PangnnError("embed_conv: node features are data, not parameters")
    a, c = _rank1_cached(graph_struct(edge_index, x.size(0)), edge_weight, x)
    return RankOneFn.apply(a, c, w_e, b_e, weight, bias, act)


def gcn_layer(x, weight, bias, edge_index, edge_weight=None, act=ACT_NONE):
    """GCNConv(add_self_loops=False) forward (+ optional fused ELU) — ``src/gnn.py:129-165``."""
    _need_cuda(x, weight, edge_index)
    gs = graph_struct(edge_index, x.size(0))
    fn = GCNLayerAggFirstFn if (weight.size(1) < weight.size(0) and weight.size(1) % 4 == 0) else GCNLayerFn
    return fn.apply(x.contiguous(), weight, bias, gs, edge_weight, act)


# ------------------------------------------------------------------------------------------------
# fused edge scorer: one host wrapper per C entry point, the layout of its gradients, the W1 split
# ------------------------------------------------------------------------------------------------
ScorerGrads = namedtuple("ScorerGrads", "dW2 db2 dw3 db3 db1 dw1c")
# offsets of the small gradients in grads[NGRADS] (``pangnn_edge_score_bwd``); read them through scorer_grads
_G_W2, _G_B2, _G_W3, _G_B3, _G_B1, _G_W1C = 0, 4096, 4160, 4224, 4225, 4289


def scorer_grads(grads):
    """Parameter-shaped views of the scorer's small gradients ``grads`` [NGRADS] (``pangnn_edge_score_bwd``):
    dW2 [D, D], db2 [D], dw3 [1, D], db3 [1], db1 [D], dw1c [D]."""
    D = SCORER_D
    return ScorerGrads(grads[_G_W2:_G_W2 + D * D].view(D, D), grads[_G_B2:_G_B2 + D], grads[_G_W3:_G_W3 + D].view(1, D),
                       grads[_G_B3:_G_B3 + 1], grads[_G_B1:_G_B1 + D], grads[_G_W1C:_G_W1C + D])


def split_w1(w1, has_skip):
    """First scorer layer ``W1`` [D, 2D (+1)] hoisted to the nodes: -> (``wcat = [W1[:, :D] ; W1[:, D:2D]]``
    [2D, D], so that ``pq = h wcat^T``; the skip column ``w1c`` [D], or None).  Plain differentiable torch ops."""
    D = SCORER_D
    wcat = torch.cat((w1[:, :D], w1[:, D:2 * D]), dim=0)
    return wcat, (w1[:, 2 * D].contiguous() if has_skip else None)


def _scorer_operands(pq, w1c, b1, w2, b2, w3, b3, gs, skip):
    """-> (the ten leading arguments of every scorer entry point, as tensors that the caller holds until the launch
    is enqueued; the edge count).  ``gs``: the scored-edge structure, or its int32 endpoints ``(src, dst)``."""
    _need_cuda(pq)
    src, dst = gs if isinstance(gs, tuple) else gs.endpoints32
    return (pq.contiguous(), src, dst, skip, w1c, b1, w2.contiguous(), b2, w3.contiguous(), b3), src.numel()


def edge_score_pq_fwd(pq, w1c, b1, w2, b2, w3, b3, gs, skip):
    """Inference form of the scorer on pre-transformed endpoint rows ``pq`` [n_ext, 2D] (layer 1 hoisted,
    ``split_w1``) -> logits."""
    lib = _abi.load()
    args, E = _scorer_operands(pq, w1c, b1, w2, b2, w3, b3, gs, skip)
    logits = torch.empty(E, dtype=torch.float32, device=pq.device)
    _abi.check(lib.pangnn_edge_score_fwd(*map(_p, args), E, None, 1.0, _p(logits), None, None, 0, _stream()),
               "edge_score_fwd")
    LAUNCHES["count"] += 1
    return logits


def edge_score_predict(pq, w1c, b1, w2, b2, w3, b3, gs, skip, threshold=0.5):
    """Inference with the prediction head fused in: -> (logits, prob = sigmoid(logits), pred = prob >= threshold)
    (``pangnn.py:220-221``, ``src/predict.py:54-55``)."""
    lib = _abi.load()
    args, E = _scorer_operands(pq, w1c, b1, w2, b2, w3, b3, gs, skip)
    dev = pq.device
    logits = torch.empty(E, dtype=torch.float32, device=dev)
    prob = torch.empty(E, dtype=torch.float32, device=dev)
    pred = torch.empty(E, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_edge_score_predict(*map(_p, args), E, float(threshold), _p(logits), _p(prob), _p(pred),
                                             _stream()), "edge_score_predict")
    LAUNCHES["count"] += 1
    return logits, prob, pred


def edge_score_train(pq, w1c, b1, w2, b2, w3, b3, gs, skip, *, y=None, pos_weight=1.0, scale=1.0, dlogits=None,
                     logits=None, loss_sum=None, da1=None, grads=None, ws=None):
    """Training form -> (da1 [E, D], the per-edge gradient of layer 1's pre-activation; grads [NGRADS], see
    ``scorer_grads``).  The upstream gradient is ``dlogits`` [E], or with labels ``y`` the fused
    BCE-with-logits(``pos_weight``) times ``scale``, which also writes ``logits`` and adds the loss sum into
    ``loss_sum`` (float64 [1], zeroed by the caller) when they are given.  ``da1`` (at least E rows), ``grads`` and
    the workspace ``ws`` are allocated unless given."""
    lib = _abi.load()
    args, E = _scorer_operands(pq, w1c, b1, w2, b2, w3, b3, gs, skip)
    dev = pq.device
    if da1 is None:
        da1 = torch.empty(E, SCORER_D, dtype=torch.float32, device=dev)
    if grads is None:
        grads = torch.empty(NGRADS, dtype=torch.float32, device=dev)
    if ws is None:
        ws = _ws(lib.pangnn_edge_score_workspace_bytes(E), dev)
    dlogits = None if dlogits is None else dlogits.contiguous()
    y = None if y is None else y.contiguous()
    _abi.check(lib.pangnn_edge_score_bwd(*map(_p, args), E, _p(dlogits), _p(y), float(pos_weight), float(scale),
                                         _p(da1), _p(grads), _p(logits), _p(loss_sum), _p(ws), ws.numel(), _stream()),
               "edge_score_bwd")
    LAUNCHES["count"] += 2 + (loss_sum is not None)
    return da1, grads


def _scorer_common(h, w1, skip):
    if h.size(1) != SCORER_D or w1.size(0) != SCORER_D:
        raise _abi.PangnnError("the fused edge scorer is built for --node_dim 64")
    return split_w1(w1, skip is not None)


def _unpack_scorer_grads(grads, da1, gs, h, wcat, skip, need_h, scale=None):
    """Per-edge gradients -> node gradients by sorted-segment reduction over both orientations of
    the scored-edge graph, then the hoisted layer-1 GEMMs."""
    D = SCORER_D
    N = h.size(0)
    dpq = torch.empty(N, 2 * D, dtype=torch.float32, device=h.device)
    segment_sum_edges(gs.src, da1, N, dpq[:, :D])                                 # edges by source
    segment_sum_edges(gs.dst, da1, N, dpq[:, D:])                                 # edges by target
    dwcat = gemm_tn(dpq, h)                                                        # [2D, D]
    if scale is not None:
        # upstream scalar gradient: folded into the small operands, never into an [N, *] pass
        grads, dwcat, wcat = grads * scale, dwcat * scale, wcat * scale
    g = scorer_grads(grads)
    dw1 = torch.cat((dwcat[:D], dwcat[D:]) + ((g.dw1c.unsqueeze(1),) if skip is not None else ()), dim=1)
    dh = node_linear(dpq, wcat, w_is_kn=True) if need_h else None
    return dh, dw1, g.db1, g.dW2, g.db2, g.dw3, g.db3


class EdgeScoreFn(torch.autograd.Function):
    """logits = MLP(cat(h[src], h[dst] (, skip)))  — ``src/gnn.py:171-177``."""

    @staticmethod
    def forward(ctx, h, w1, b1, w2, b2, w3, b3, gs, skip):
        wcat, w1c = _scorer_common(h, w1, skip)
        pq = node_linear(h, wcat)                                       # hoisted layer 1
        logits = edge_score_pq_fwd(pq, w1c, b1, w2, b2, w3, b3, gs, skip)
        ctx.gs, ctx.skip = gs, skip
        ctx.save_for_backward(h, w1, b1, w2, b2, w3, b3, pq)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        h, w1, b1, w2, b2, w3, b3, pq = ctx.saved_tensors
        gs, skip = ctx.gs, ctx.skip
        wcat, w1c = _scorer_common(h, w1, skip)
        da1, grads = edge_score_train(pq, w1c, b1, w2, b2, w3, b3, gs, skip, dlogits=dlogits)
        return _unpack_scorer_grads(grads, da1, gs, h, wcat, skip, ctx.needs_input_grad[0]) + (None, None)


class EdgeScoreBCEFn(torch.autograd.Function):
    """Fused training form: (loss, logits) = BCEWithLogits(pos_weight)(MLP(...), y), mean reduction
    (``pangnn.py:98,203``).  ONE kernel produces logits, loss and all gradients; backward only
    rescales by the incoming scalar."""

    @staticmethod
    def forward(ctx, h, w1, b1, w2, b2, w3, b3, gs, skip, y, pos_weight):
        wcat, w1c = _scorer_common(h, w1, skip)
        E = gs.num_edges
        pq = node_linear(h, wcat)
        logits = torch.empty(E, dtype=torch.float32, device=h.device)
        loss_sum = torch.zeros(1, dtype=torch.float64, device=h.device)
        da1, grads = edge_score_train(pq, w1c, b1, w2, b2, w3, b3, gs, skip, y=y, pos_weight=pos_weight,
                                      scale=1.0 / max(E, 1), logits=logits, loss_sum=loss_sum)
        ctx.gs, ctx.skip = gs, skip
        ctx.save_for_backward(h, wcat, da1, grads)
        ctx.mark_non_differentiable(logits)
        loss = (loss_sum / max(E, 1)).float().squeeze(0)
        return loss, logits

    @staticmethod
    def backward(ctx, dloss, _dlogits):
        h, wcat, da1, grads = ctx.saved_tensors
        out = _unpack_scorer_grads(grads, da1, ctx.gs, h, wcat, ctx.skip, ctx.needs_input_grad[0],
                                   scale=dloss)
        return out + (None, None, None, None)


class EdgePairScoreFn(torch.autograd.Function):
    """cosine (mode 0, ``src/gnn.py:206-207``) / row-wise dot (mode 1, ``src/gnn.py:77-79``).
    Forward is one warp-per-edge kernel; backward (``pangnn_edge_pair_score_bwd``) is two weighted aggregations
    over the scored-edge graph plus a diagonal term — no per-edge [E, F] gradient rows (``edge_scorer.cu``)."""

    @staticmethod
    def forward(ctx, h, gs, mode):
        lib = _abi.load()
        src, dst = gs.endpoints32
        h = h.contiguous()
        out = torch.empty(gs.num_edges, dtype=torch.float32, device=h.device)
        _abi.check(lib.pangnn_edge_pair_score(_p(h), h.stride(0), h.size(1), _p(src), _p(dst),
                                              gs.num_edges, mode, _p(out), _stream()), "edge_pair_score")
        LAUNCHES["count"] += 1
        ctx.gs, ctx.mode = gs, mode
        ctx.save_for_backward(h, out)
        return out

    @staticmethod
    def backward(ctx, dz):
        lib = _abi.load()
        h, out = ctx.saved_tensors
        gs = ctx.gs
        N, F = h.shape
        if F % 4:                                               # odd --node_dim: the library path
            src, dst = gs.edge_index[0], gs.edge_index[1]
            a, b = h.index_select(0, src), h.index_select(0, dst)
            g = dz.unsqueeze(1)
            if ctx.mode == 1:
                ga, gb = g * b, g * a
            else:
                na = a.norm(dim=1, keepdim=True).clamp_min(1e-8)
                nb = b.norm(dim=1, keepdim=True).clamp_min(1e-8)
                c = out.unsqueeze(1)
                ga, gb = g * (b / (na * nb) - c * a / (na * na)), g * (a / (na * nb) - c * b / (nb * nb))
            return torch.zeros_like(h).index_add_(0, src, ga).index_add_(0, dst, gb), None, None
        dh = torch.empty(N, F, dtype=torch.float32, device=h.device)
        ws = _ws(lib.pangnn_edge_pair_score_bwd_workspace_bytes(gs.num_edges, N, F), h.device)
        s, d = gs.src, gs.dst
        _abi.check(lib.pangnn_edge_pair_score_bwd(_p(h), h.stride(0), F, N, gs.num_edges, _p(s.rowptr), _p(s.col),
                                                  _p(s.perm), _p(d.rowptr), _p(d.col), _p(d.perm),
                                                  _p(dz.contiguous().float()), _p(out), ctx.mode, _p(dh), _p(ws),
                                                  ws.numel(), _stream()), "edge_pair_score_bwd")
        LAUNCHES["count"] += 6
        return dh, None, None


def edge_pair_score(h, gs, mode):
    return EdgePairScoreFn.apply(h, gs, mode)


class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) with all three products on our kernels (node_linear / gemm_tn).  With
    ``extra_rows`` the result is allocated ``extra_rows`` rows taller, or written into ``out_full``
    (rows [M, ...) are left for the caller: the partitioned path receives halo rows straight into
    them; ``out_full`` may live in symmetric memory)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, extra_rows, out_full, push=None):
        x = x.contiguous()
        M, n = x.size(0), weight.size(0)
        if out_full is None:
            y_full = torch.empty(M + extra_rows, n, dtype=torch.float32, device=x.device)
        else:
            # a fresh tensor object over the caller's memory (never the caller's own tensor: returning
            # an input would need mark_dirty and tie this node's history to a reused buffer)
            y_full = _alias(out_full, out_full.shape, out_full.stride())
        y = node_linear(x, weight, bias, act, out=y_full[:M], push=push)
        ctx.act, ctx.has_bias, ctx.M = act, bias is not None, M
        ctx.save_for_backward(x, weight, y if act != ACT_NONE else None)
        return y_full

    @staticmethod
    def backward(ctx, dy_full):
        x, weight, y = ctx.saved_tensors
        dy = dy_full[:ctx.M]
        if ctx.act != ACT_NONE or ctx.has_bias:
            g, dbias = act_bwd_bias(dy, y, ctx.act)
        else:
            g, dbias = dy.contiguous(), None
        dW = gemm_tn(g, x) if ctx.needs_input_grad[1] else None
        dx = node_linear(g, weight, w_is_kn=True) if ctx.needs_input_grad[0] else None
        return dx, dW, (dbias if ctx.has_bias and ctx.needs_input_grad[2] else None), None, None, None, None


def linear(x, weight, bias=None, act=ACT_NONE, extra_rows=0, out_full=None, push=None):
    return LinearFn.apply(x, weight, bias, act, extra_rows, out_full, push)


# ------------------------------------------------------------------------------------------------
# building blocks of the genome-partitioned (multi-GPU) path: see pangnn_b200/dist.py
# ------------------------------------------------------------------------------------------------
class AggregateFn(torch.autograd.Function):
    """y[:n_out] = act(A_hat x_ext + b) on a LOCAL graph whose sources live in "own + halo"
    numbering: forward walks the by-destination CSR (rows = owned nodes), backward walks the
    by-source CSR (rows = own + halo) and returns gradients for every extended row — into
    ``dx_out`` when given (a symmetric-memory buffer whose halo part the owners read over NVLink)."""

    @staticmethod
    def forward(ctx, x_ext, bias, csr_dst, val_dst, csr_src, val_src, n_out, act, dx_out=None):
        y = gcn_aggregate(csr_dst.rowptr, csr_dst.col, val_dst, x_ext.contiguous(), n_out, bias, act)
        ctx.csr_src, ctx.val_src, ctx.act, ctx.n_in = csr_src, val_src, act, x_ext.size(0)
        ctx.has_bias, ctx.dx_out = bias is not None, dx_out
        ctx.save_for_backward(y if act != ACT_NONE else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        if ctx.act != ACT_NONE or ctx.has_bias:
            g, dbias = act_bwd_bias(dy, y, ctx.act)
        else:
            g, dbias = dy.contiguous(), None
        out = None if ctx.dx_out is None else _alias(ctx.dx_out, (ctx.n_in, ctx.dx_out.size(1)))
        dx = gcn_aggregate(ctx.csr_src.rowptr, ctx.csr_src.col, ctx.val_src, g, ctx.n_in, out=out)
        return dx, (dbias if ctx.has_bias else None), None, None, None, None, None, None, None


class EdgeScoreBCEPQFn(torch.autograd.Function):
    """Fused scorer + BCE on pre-transformed endpoint rows ``pq_ext`` [n_ext, 2D] (layer 1 hoisted by
    the caller).  Returns (sum of the per-edge losses * scale, logits).  Backward yields ``dpq_ext``
    (P half reduced by source, Q half by destination — both sorted-segment) and the small grads."""

    @staticmethod
    def forward(ctx, pq, w1c, b1, w2, b2, w3, b3, gs, skip, y, pos_weight, scale, dpq_out=None, unit_grad=False):
        # unit_grad: the caller promises to back-propagate the returned loss as is (``loss.backward()``): the
        # backward then skips the pass that multiplies the [n, 2D] node gradient by the incoming scalar (0.2 ms at
        # C3 on a partition) and checks the promise with an asynchronous device-side assert instead
        ctx.unit_grad = bool(unit_grad)
        E, D, n = gs.num_edges, SCORER_D, pq.size(0)
        weights = (w1c, b1, w2, b2, w3, b3)
        logits = torch.empty(E, dtype=torch.float32, device=pq.device)
        loss_sum = torch.zeros(1, dtype=torch.float64, device=pq.device)
        ctx.gs, ctx.has_skip, ctx.n_ext, ctx.dpq_out = gs, skip is not None, n, dpq_out
        ctx.chunked = E > SCORER_CHUNK_EDGES["n"] and gs.src.identity_perm
        if not ctx.chunked:
            da1, grads = edge_score_train(pq, *weights, gs, skip, y=y, pos_weight=pos_weight, scale=scale,
                                          logits=logits, loss_sum=loss_sum)
            ctx.save_for_backward(da1, grads)
        else:
            # ---- chunked form: one scorer launch per run of source rows, node gradients reduced right away
            lib = _abi.load()
            ch = scored_chunks(gs, SCORER_CHUNK_EDGES["n"])
            dpq = (_alias(dpq_out, (n, 2 * D)) if dpq_out is not None
                   else torch.empty(n, 2 * D, dtype=torch.float32, device=pq.device))
            dpq.zero_()                                         # rows of nodes without scored edges; Q half accumulates
            da1 = torch.empty(ch.max_edges, D, dtype=torch.float32, device=pq.device)
            tmp = torch.empty(n, D, dtype=torch.float32, device=pq.device)
            grads = torch.zeros(NGRADS, dtype=torch.float32, device=pq.device)
            gk = torch.empty(NGRADS, dtype=torch.float32, device=pq.device)
            ws = _ws(lib.pangnn_edge_score_workspace_bytes(ch.max_edges), pq.device)
            src, dst = gs.endpoints32
            y = y.contiguous()
            for (r0, r1, c0, c1), csr_k in zip(ch.runs, ch.csr_dst):
                edge_score_train(pq, *weights, (src[c0:c1], dst[c0:c1]), None if skip is None else skip[c0:c1],
                                 y=y[c0:c1], pos_weight=pos_weight, scale=scale, logits=logits[c0:c1],
                                 loss_sum=loss_sum, da1=da1, grads=gk, ws=ws)
                grads += gk                                     # (the loss is accumulated by the kernel's own reduction)
                # by source: the run's rows are complete inside the chunk (identity columns).  A raw call, because
                # the CSR's offsets are absolute edge positions: the row base is shifted back by c0 rows
                _abi.check(lib.pangnn_gcn_aggregate(_p(gs.src.rowptr[r0:]), None, None,
                                                    C.c_void_p(da1.data_ptr() - c0 * D * 4), D, r1 - r0, D, None, ACT_NONE,
                                                    _p(dpq[r0:r1]), dpq.stride(0), _stream()), "segment_sum(chunk, by source)")
                # by destination: this chunk's share of every node's sum, accumulated in fixed chunk order
                gcn_aggregate(csr_k.rowptr, csr_k.perm, None, da1[:c1 - c0], n, out=tmp)
                dpq[:, D:] += tmp
                LAUNCHES["count"] += 3                          # the raw segment sum and the two accumulations
            ctx.save_for_backward(dpq, grads)
        ctx.mark_non_differentiable(logits)
        return (loss_sum * scale).float().squeeze(0), logits

    @staticmethod
    def backward(ctx, dloss, _dlogits):
        da1, grads = ctx.saved_tensors
        gs, D, n = ctx.gs, SCORER_D, ctx.n_ext
        if ctx.unit_grad:
            torch._assert_async(dloss == 1)                     # misuse guard, no host synchronisation
        if ctx.chunked:                                         # the forward already reduced da1 to the nodes
            dpq = da1
        else:
            dpq = (_alias(ctx.dpq_out, (n, 2 * D)) if ctx.dpq_out is not None
                   else torch.empty(n, 2 * D, dtype=torch.float32, device=da1.device))
            segment_sum_edges(gs.src, da1, n, dpq[:, :D])
            segment_sum_edges(gs.dst, da1, n, dpq[:, D:])
        g = scorer_grads(grads if ctx.unit_grad else grads * dloss)
        if not ctx.unit_grad:
            dpq = dpq * dloss if dloss.requires_grad else dpq.mul_(dloss)
        return (dpq, g.dw1c if ctx.has_skip else None, g.db1, g.dW2, g.db2, g.dw3, g.db3) + (None,) * 7


# ------------------------------------------------------------------------------------------------
# candidate normalisation
# ------------------------------------------------------------------------------------------------
def hits_sort_unique(q, t, bits, num_nodes):
    """(q, t, bits) device hit table -> sorted by (q, t), duplicate pairs collapsed to the last row."""
    lib = _abi.load()
    _need_cuda(q, t, bits)
    n = q.numel()
    q = q.to(torch.int32).contiguous(); t = t.to(torch.int32).contiguous()
    bits = bits.to(torch.float64).contiguous()
    dev = q.device
    qo = torch.empty(n, dtype=torch.int32, device=dev)
    to = torch.empty(n, dtype=torch.int32, device=dev)
    bo = torch.empty(n, dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _ws(lib.pangnn_hits_sort_unique_workspace_bytes(n), dev)
    _abi.check(lib.pangnn_hits_sort_unique(_p(q), _p(t), _p(bits), n, num_nodes, _p(qo), _p(to), _p(bo),
                                           _p(cnt), _p(ws), ws.numel(), _stream()), "hits_sort_unique")
    nbits = max(1, (max(num_nodes, 2) - 1).bit_length())
    LAUNCHES["count"] += 4 + 3 * ((2 * nbits + 7) // 8)
    m = int(cnt.item())
    return qo[:m], to[:m], bo[:m]


def hits_normalize(q, t, bits, genome_of, group_of=None, temp=0.8, eps=1e-8, pseudo=1.0,
                   drop_trivial=True):
    """Sorted unique hit table -> (src, dst, w, y) int32/int32/fp32/fp32, sorted by (src, dst)."""
    lib = _abi.load()
    _need_cuda(q, t, bits, genome_of, group_of)
    n = q.numel()
    dev = q.device
    genome_of = genome_of.to(torch.int32).contiguous()
    if group_of is not None:
        group_of = group_of.to(torch.int32).contiguous()
    src = torch.empty(n, dtype=torch.int32, device=dev)
    dst = torch.empty(n, dtype=torch.int32, device=dev)
    w = torch.empty(n, dtype=torch.float32, device=dev)
    y = torch.empty(n, dtype=torch.float32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _ws(lib.pangnn_hits_normalize_workspace_bytes(n), dev)
    _abi.check(lib.pangnn_hits_normalize(_p(q.contiguous()), _p(t.contiguous()), _p(bits.contiguous()),
                                         n, _p(genome_of), _p(group_of), float(temp), float(eps),
                                         float(pseudo), 1 if drop_trivial else 0, _p(src), _p(dst),
                                         _p(w), _p(y), _p(cnt), _p(ws), ws.numel(), _stream()),
               "hits_normalize")
    LAUNCHES["count"] += 6
    m = int(cnt.item())
    return src[:m], dst[:m], w[:m], y[:m]


def segment_max_labels(q, t, score, genome_of):
    """Max-candidate baseline labels over (query, target-genome) segments of a (q, t)-sorted table
    (``src/helper.py:437-485,494-576``).  ``score`` fp64 or fp32.  -> int32 [n]."""
    lib = _abi.load()
    _need_cuda(q, t, score, genome_of)
    n = q.numel()
    q = q.to(torch.int32).contiguous(); t = t.to(torch.int32).contiguous()
    if score.dtype not in (torch.float32, torch.float64):
        score = score.float()
    score = score.contiguous()
    genome_of = genome_of.to(torch.int32).contiguous()
    label = torch.empty(n, dtype=torch.int32, device=q.device)
    ws = _ws(lib.pangnn_segment_max_labels_workspace_bytes(n), q.device)
    _abi.check(lib.pangnn_segment_max_labels(_p(q), _p(t), _p(score), 1 if score.dtype == torch.float64 else 0, n,
                                             _p(genome_of), _p(label), _p(ws), ws.numel(), _stream()),
               "segment_max_labels")
    LAUNCHES["count"] += 5
    return label


_LABEL_KINDS = {torch.float32: 0, torch.int32: 1, torch.int64: 2, torch.uint8: 3, torch.bool: 3}
METRIC_NAN, METRIC_BAD_LABEL = 1, 2
METRIC_HIST_BINS = 65536


def metric_runs(scores=None, labels=None, runs=None, info=None, hist=None):
    """Distinct-score runs for the ranking metrics (``pangnn_metric_runs``): of (fp32 ``scores``, {0,1} ``labels``),
    or of input ``runs`` [m, 3] (merged, counts of equal keys summed).  -> int64 runs [n, 3] (key, pos, neg) in
    decreasing score order, of which the first ``info[0]`` rows are valid.  ``info`` int64 [6] (device, written):
    runs, P, N, 0, 0, flags; ``hist`` int64 [65536] (device, optional, written): runs per top 16 key bits."""
    lib = _abi.load()
    if runs is not None:
        _need_cuda(runs, info, hist)
        runs = runs.contiguous()
        n, dev, kind = runs.size(0), runs.device, 0
    else:
        _need_cuda(scores, labels, info, hist)
        if scores.dtype != torch.float32:
            raise _abi.PangnnError(f"metric_runs: scores must be float32, not {scores.dtype}")
        if labels.dtype not in _LABEL_KINDS:
            raise _abi.PangnnError(f"metric_runs: unsupported label dtype {labels.dtype}")
        scores, labels = scores.reshape(-1).contiguous(), labels.reshape(-1).contiguous()
        if labels.numel() != scores.numel():
            raise _abi.PangnnError("metric_runs: scores and labels differ in length")
        n, dev, kind = scores.numel(), scores.device, _LABEL_KINDS[labels.dtype]
    if n >= 1 << 32:
        raise _abi.PangnnError(f"metric_runs: {n} scores on one device; the sort takes fewer than 2^32")
    out = torch.empty(n, 3, dtype=torch.int64, device=dev)
    ws = _ws(lib.pangnn_metric_runs_workspace_bytes(n), dev)
    _abi.check(lib.pangnn_metric_runs(_p(scores), _p(labels), kind, _p(runs), n, _p(out), _p(info), _p(hist),
                                      _p(ws), ws.numel(), _stream()), "metric_runs")
    LAUNCHES["count"] += 4 + 3 * 4 if n else 0
    return out


def metric_reduce(runs, params, out=None):
    """``pangnn_metric_reduce`` over the first ``params[0]`` rows of ``runs`` (device int64 params: runs, P, N, TP_0,
    FP_0) -> int64 [8] (device): AUROC numerator (lo, hi), AP numerator (lo, hi), best Youden j (fp64 bits), its
    run's key, runs, AP fixed-point shift."""
    lib = _abi.load()
    _need_cuda(runs, params, out)
    runs = runs.contiguous()
    if out is None:
        out = torch.empty(8, dtype=torch.int64, device=runs.device)
    R = runs.size(0)
    ws = _ws(lib.pangnn_metric_reduce_workspace_bytes(R), runs.device)
    _abi.check(lib.pangnn_metric_reduce(_p(runs), R, _p(params), _p(out), _p(ws), ws.numel(), _stream()),
               "metric_reduce")
    LAUNCHES["count"] += 4 if R else 1
    return out


CURVE_ALL, CURVE_ROC, CURVE_PR = 0, 1, 2
CURVE_FIRST, CURVE_FOLLOWED = 1, 2


def metric_curve(runs, params, bound, mode, out=None):
    """``pangnn_metric_curve`` over the first ``params[0]`` rows of ``runs`` (device int64 params: runs, P, N, TP_0,
    FP_0; ``bound`` int64 [3]: (pos, neg) of the run after the last one, ``CURVE_FIRST | CURVE_FOLLOWED`` flags) with
    ``mode`` ``CURVE_ALL`` / ``CURVE_ROC`` / ``CURVE_PR`` -> (thresholds fp32 [R], TP int64 [R], FP int64 [R],
    count int64 [3]) on the device: the first ``count[0]`` points are the kept runs; ``count[1:3]`` = (pos, neg) of
    the runs.  ``out`` = the same four tensors, preallocated."""
    lib = _abi.load()
    _need_cuda(runs, params, bound)
    runs = runs.contiguous()
    R, dev = runs.size(0), runs.device
    if out is None:
        out = (torch.empty(R, dtype=torch.float32, device=dev), torch.empty(R, dtype=torch.int64, device=dev),
               torch.empty(R, dtype=torch.int64, device=dev), torch.empty(3, dtype=torch.int64, device=dev))
    thr, tp, fp, count = out
    _need_cuda(thr, tp, fp, count)
    if min(thr.numel(), tp.numel(), fp.numel()) < R or count.numel() < 3:
        raise _abi.PangnnError(f"metric_curve: outputs need room for {R} points and count for 3")
    ws = _ws(lib.pangnn_metric_curve_workspace_bytes(R), dev)
    _abi.check(lib.pangnn_metric_curve(_p(runs), R, _p(params), _p(bound), int(mode), _p(thr), _p(tp), _p(fp),
                                       _p(count), _p(ws), ws.numel(), _stream()), "metric_curve")
    LAUNCHES["count"] += 3 if R else 1
    return out


def rows_gather_copy(src, idx, dst):
    """dst[k] = src[idx[k]] (idx int32 or None); ``dst`` may be a PEER tensor (symmetric memory)."""
    lib = _abi.load()
    n = dst.size(0) if idx is None else idx.numel()
    _abi.check(lib.pangnn_rows_gather_copy(_p(src), src.stride(0), _p(idx), n, src.size(1), _p(dst), dst.stride(0),
                                           _stream()), "rows_gather_copy")
    LAUNCHES["count"] += 1


def rows_scatter_add(src, idx, dst):
    """dst[idx[k]] += src[k] (idx unique); ``src`` may be a PEER tensor (symmetric memory)."""
    lib = _abi.load()
    n = src.size(0) if idx is None else idx.numel()
    _abi.check(lib.pangnn_rows_scatter_add(_p(src), src.stride(0), _p(idx), n, src.size(1), _p(dst), dst.stride(0),
                                           _stream()), "rows_scatter_add")
    LAUNCHES["count"] += 1


# ------------------------------------------------------------------------------------------------
# data-parallel gradient average over peer memory (csrc/grad_reduce.cu)
# ------------------------------------------------------------------------------------------------
GRAD_REDUCE_MAX_TENSORS, GRAD_REDUCE_MAX_RANKS = 32, 8


def _ptr_array(ptrs):
    arr = (C.c_void_p * max(len(ptrs), 1))(*ptrs)
    return arr, C.cast(arr, C.c_void_p)


def _grad_table(grads, numels):
    """(keep-alive, grads**, numels*) host tables: ``grads`` are fp32 dense CUDA tensors or None (NULL)."""
    for g in grads:
        if g is not None and (not g.is_cuda or g.dtype != torch.float32 or not g.is_contiguous()):
            raise _abi.PangnnError("grad_push / grad_reduce need dense fp32 CUDA gradients")
    gp = _ptr_array([g.data_ptr() if g is not None else None for g in grads])
    nn = (C.c_int64 * max(len(numels), 1))(*[int(n) for n in numels])
    return (gp[0], nn), gp[1], C.cast(nn, C.c_void_p)


def grad_bucket_floats(numels):
    """Floats one bucket half needs for tensors of ``numels`` elements (each tensor starts on a 4-float boundary)."""
    nn = (C.c_int64 * max(len(numels), 1))(*[int(n) for n in numels])
    return int(_abi.load().pangnn_grad_bucket_floats(C.cast(nn, C.c_void_p), len(numels)))


def grad_push(grads, numels, bucket, half_floats, peer_signals, rank, ctrl):
    """Pack ``grads`` into half ``ctrl[0] & 1`` of ``bucket`` (this rank's, 2 * ``half_floats`` floats) and signal
    ``ctrl[0] + 1`` into slot ``rank`` of every ``peer_signals`` array (data pointers, one per rank, in rank order)."""
    keep, gp, nn = _grad_table(grads, numels)
    sig_keep, sp = _ptr_array(list(peer_signals))
    _abi.check(_abi.load().pangnn_grad_push(gp, nn, len(grads), _p(bucket), int(half_floats), sp, len(peer_signals),
                                            int(rank), _p(ctrl), _stream()), "grad_push")
    LAUNCHES["count"] += 1


def grad_reduce(grads, numels, peer_buckets, half_floats, signal, rank, ctrl, timeout_s=120.0):
    """Wait for every rank's signal of this call, then ``grads = (b_0 + ... + b_{W-1}) * fp32(1 / W)`` in rank order
    over half ``ctrl[0] & 1`` of the ``peer_buckets`` (data pointers, in rank order); None entries are skipped.  A wait
    longer than ``timeout_s`` leaves ``1 + rank of the missing peer`` in ``ctrl[3]`` instead."""
    keep, gp, nn = _grad_table(grads, numels)
    buck_keep, bp = _ptr_array(list(peer_buckets))
    _abi.check(_abi.load().pangnn_grad_reduce(gp, nn, len(grads), bp, int(half_floats), _p(signal), len(peer_buckets),
                                              int(rank), _p(ctrl), int(timeout_s * 1e9), _stream()), "grad_reduce")
    LAUNCHES["count"] += 1


def neighbour_band(num_nodes, n, device="cuda", out=None):
    """Whole-graph neighbour band ``[2, Eb]`` int64 (``src/dataset.py:351-366``) from one closed-form
    kernel, no host sync.  ``out`` = ``(src_row, dst_row)`` writes into existing int64 storage (the tail of
    a union edge list)."""
    lib = _abi.load()
    eb = int(lib.pangnn_neighbour_band_edges(int(num_nodes), int(n)))
    if out is None:
        nb = torch.empty(2, eb, dtype=torch.int64, device=device)
        out = (nb[0], nb[1])
    else:
        nb = None
    assert all(o.is_cuda and o.dtype == torch.int64 and o.is_contiguous() and o.numel() == eb for o in out)
    _abi.check(lib.pangnn_neighbour_band(int(num_nodes), int(n), _p(out[0]), _p(out[1]), _stream()), "neighbour_band")
    LAUNCHES["count"] += 1
    return nb


def union_index(edge_index, num_nodes, n):
    """``[sim ; nb]`` edge list of the whole-graph union assembly (``src/dataset.py:373-378``) on the device:
    the band is generated straight into the tail of the union list."""
    lib = _abi.load()
    E = edge_index.size(1)
    eb = int(lib.pangnn_neighbour_band_edges(int(num_nodes), int(n)))
    union = torch.empty(2, E + eb, dtype=torch.int64, device=edge_index.device)
    union[:, :E].copy_(edge_index)
    neighbour_band(num_nodes, n, out=(union[0, E:], union[1, E:]))
    return union


def union_weights(edge_weight, num_union_edges):
    """``[w ; 1...]`` (``src/dataset.py:379-381``)."""
    E = edge_weight.numel()
    uw = torch.empty(num_union_edges, dtype=torch.float32, device=edge_weight.device)
    uw[:E].copy_(edge_weight)
    uw[E:].fill_(1.0)
    return uw


# ------------------------------------------------------------------------------------------------
# a12: batch collation on the device
# ------------------------------------------------------------------------------------------------
class _CollateAttr(C.Structure):
    _fields_ = [("src", C.c_void_p), ("seg_ptr", C.c_void_p), ("dst", C.c_void_p), ("src_row_stride", C.c_int64),
                ("dst_row_stride", C.c_int64), ("rows", C.c_int32), ("elem_bytes", C.c_int32), ("kind", C.c_int32),
                ("width", C.c_int32)]


_COLLATE_COPY, _COLLATE_INDEX, _COLLATE_FILL = 0, 1, 2
COLLATE_MAX_ATTRS = 12


class PackedGraphs:
    """The graphs of a split packed back to back on the device, one arena per tensor attribute, so that a batch
    is assembled by ``pangnn_collate`` (two launches) instead of ~10 ``torch.cat`` on the host + one H2D per
    attribute.  ``collate(ids)`` returns the same attribute bag as ``pangnn_b200.data.collate`` of the same
    graphs moved to the device (PyG ``Batch.from_data_list`` semantics, SURVEY A.3), bit for bit."""

    def __init__(self, graphs, device):
        import numpy as np
        self._np = np
        graphs = list(graphs)
        if not graphs:
            raise ValueError("no graphs to pack")
        self.device = torch.device(device)
        self.num_graphs = len(graphs)
        keys = [k for k, v in graphs[0].__dict__.items() if v is not None and not k.startswith("_")]
        self.tensor_keys = [k for k in keys if torch.is_tensor(getattr(graphs[0], k))]
        self.other_keys = [k for k in keys if k not in self.tensor_keys]
        self.other = {k: [getattr(g, k) for g in graphs] for k in self.other_keys}
        if len(self.tensor_keys) + 1 > COLLATE_MAX_ATTRS:
            raise ValueError(f"at most {COLLATE_MAX_ATTRS - 1} tensor attributes per graph")

        def table(sizes):
            ptr = np.zeros(len(sizes) + 1, dtype=np.int64)
            np.cumsum(np.asarray(sizes, dtype=np.int64), out=ptr[1:])
            return ptr, torch.from_numpy(ptr).to(self.device)

        self.node_ptr, self.node_ptr_dev = table([g.x.size(0) for g in graphs])
        self.attrs = {}
        for k in self.tensor_keys:
            vals = [getattr(g, k) for g in graphs]
            v0 = vals[0]
            if v0.element_size() not in (4, 8):
                raise ValueError(f"attribute {k}: only 4- and 8-byte element types are packed")
            if "index" in k:
                if v0.dim() != 2 or v0.size(0) != 2 or v0.dtype != torch.int64:
                    raise ValueError(f"attribute {k}: index attributes must be int64 [2, e]")
                packed = torch.cat(vals, dim=-1).contiguous().to(self.device)
                ptr, ptr_dev = table([v.size(-1) for v in vals])
                ent = dict(kind=_COLLATE_INDEX, rows=2, width=1, tail=(), stride=packed.size(1))
            else:
                packed = torch.cat(vals, dim=0).contiguous().to(self.device)
                ptr, ptr_dev = table([v.size(0) for v in vals])
                width = 1
                for d in v0.shape[1:]:
                    width *= d
                ent = dict(kind=_COLLATE_COPY, rows=1, width=max(width, 1), tail=tuple(v0.shape[1:]), stride=0)
            ent.update(packed=packed, ptr=ptr, ptr_dev=ptr_dev, dtype=v0.dtype, esize=v0.element_size())
            self.attrs[k] = ent
        self._describe()

    @classmethod
    def from_packed(cls, attrs, node_ptr, device):
        """From arenas that already exist on the device: ``attrs[name] = (packed tensor, host offset table)``
        (``[2, total]`` int64 for ``*index*`` attributes, ``[total, ...]`` otherwise) — the output of
        ``pangnn_b200.subgraphs.extract``."""
        import numpy as np
        self = object.__new__(cls)
        self._np, self.device = np, torch.device(device)
        self.node_ptr = np.asarray(node_ptr, dtype=np.int64)
        self.node_ptr_dev = torch.from_numpy(self.node_ptr).to(self.device)
        self.num_graphs = self.node_ptr.size - 1
        self.tensor_keys, self.other_keys, self.other, self.attrs = list(attrs), [], {}, {}
        for k, (packed, ptr) in attrs.items():
            ptr = np.asarray(ptr, dtype=np.int64)
            assert ptr.size == self.num_graphs + 1 and packed.is_cuda and packed.is_contiguous()
            if "index" in k:
                assert packed.dim() == 2 and packed.size(0) == 2 and packed.dtype == torch.int64
                ent = dict(kind=_COLLATE_INDEX, rows=2, width=1, tail=(), stride=packed.size(1))
            else:
                width = 1
                for d in packed.shape[1:]:
                    width *= d
                ent = dict(kind=_COLLATE_COPY, rows=1, width=max(width, 1), tail=tuple(packed.shape[1:]), stride=0)
            ent.update(packed=packed, ptr=ptr, ptr_dev=torch.from_numpy(ptr).to(self.device), dtype=packed.dtype,
                       esize=packed.element_size())
            self.attrs[k] = ent
        self._describe()
        return self

    def _describe(self):
        n = len(self.tensor_keys) + 1
        self._desc = (_CollateAttr * n)()
        for i, k in enumerate(self.tensor_keys):
            a, d = self.attrs[k], self._desc[i]
            d.src, d.seg_ptr = a["packed"].data_ptr(), a["ptr_dev"].data_ptr()
            d.src_row_stride, d.rows, d.elem_bytes, d.kind, d.width = a["stride"], a["rows"], a["esize"], a["kind"], a["width"]
        d = self._desc[n - 1]                                   # `batch`: slot of every node; its offsets are `ptr`
        d.src, d.seg_ptr, d.src_row_stride, d.rows, d.elem_bytes, d.kind, d.width = \
            None, self.node_ptr_dev.data_ptr(), 0, 1, 8, _COLLATE_FILL, 1
        self._n = n

    def sizes(self, ids):
        """Host arithmetic: ``({attribute: entries of the collated batch}, nodes)`` for the graphs ``ids``."""
        tot = {k: int((self.attrs[k]["ptr"][ids + 1] - self.attrs[k]["ptr"][ids]).sum()) for k in self.tensor_keys}
        return tot, int((self.node_ptr[ids + 1] - self.node_ptr[ids]).sum())

    def collate_into(self, ids, ids_dev, dst, batch_vec):
        """``collate`` into caller-owned tensors ``dst[attribute]`` (at least as large as the batch; ``[2, width]``
        index attributes may be wider: their row stride is honoured) and ``batch_vec`` — the static buffers of a
        captured CUDA graph (``pangnn_b200.graphs.GraphedBatchStep``).  Entries past the batch are left untouched."""
        lib = _abi.load()
        B = int(len(ids))
        off = torch.empty(self._n, B + 1, dtype=torch.int64, device=self.device)
        for i, k in enumerate(self.tensor_keys):
            t = dst[k]
            self._desc[i].dst = t.data_ptr()
            self._desc[i].dst_row_stride = t.size(1) if self.attrs[k]["rows"] == 2 else 0
        self._desc[self._n - 1].dst = batch_vec.data_ptr()
        _abi.check(lib.pangnn_collate(C.cast(self._desc, C.c_void_p), self._n, self._n - 1, _p(ids_dev), B, _p(off),
                                      _stream()), "collate")
        LAUNCHES["count"] += 2
        return off

    def collate(self, ids, ids_dev):
        """``ids``: numpy int array of graph ids (host copy, for the output sizes); ``ids_dev``: the same ids as
        an int32 device tensor."""
        from .data import Data
        np, lib = self._np, _abi.load()
        B = int(len(ids))
        out = Data()
        off = torch.empty(self._n, B + 1, dtype=torch.int64, device=self.device)
        keep = [off]
        for i, k in enumerate(self.tensor_keys):
            a = self.attrs[k]
            total = int((a["ptr"][ids + 1] - a["ptr"][ids]).sum())
            shape = (2, total) if a["rows"] == 2 else (total,) + a["tail"]
            t = torch.empty(shape, dtype=a["dtype"], device=self.device)
            self._desc[i].dst, self._desc[i].dst_row_stride = t.data_ptr(), total if a["rows"] == 2 else 0
            out.__dict__[k] = t
        nodes = int((self.node_ptr[ids + 1] - self.node_ptr[ids]).sum())
        batch = torch.empty(nodes, dtype=torch.int64, device=self.device)
        self._desc[self._n - 1].dst = batch.data_ptr()
        assert ids_dev.is_cuda and ids_dev.dtype == torch.int32 and ids_dev.numel() == B and ids_dev.is_contiguous()
        _abi.check(lib.pangnn_collate(C.cast(self._desc, C.c_void_p), self._n, self._n - 1, _p(ids_dev), B, _p(off),
                                      _stream()), "collate")
        LAUNCHES["count"] += 2
        for k in self.other_keys:
            out.__dict__[k] = [self.other[k][int(i)] for i in ids]
        out.batch, out.ptr, out.num_graphs = batch, off[self._n - 1], B
        return out


def connected_components(src, dst, num_nodes, select=None, max_rounds=64):
    """Component label (smallest node id of the component) of every node over the edges ``(src, dst)`` with
    ``select != 0`` (all edges when ``select`` is None): hook + pointer-jumping rounds until nothing changes."""
    lib = _abi.load()
    _need_cuda(src, dst, select)
    src, dst = src.to(torch.int32).contiguous(), dst.to(torch.int32).contiguous()
    sel = select.to(torch.int32).contiguous() if select is not None else None
    labels = torch.empty(num_nodes, dtype=torch.int32, device=src.device)
    changed = torch.zeros(1, dtype=torch.int32, device=src.device)
    _abi.check(lib.pangnn_components_init(_p(labels), num_nodes, _stream()), "components_init")
    LAUNCHES["count"] += 1
    for _ in range(max_rounds):
        _abi.check(lib.pangnn_components_round(_p(src), _p(dst), _p(sel), src.numel(), _p(labels), num_nodes,
                                               _p(changed), _stream()), "components_round")
        LAUNCHES["count"] += 2
        if int(changed.item()) == 0:
            return labels
    raise _abi.PangnnError("connected_components did not converge")


# ------------------------------------------------------------------------------------------------
# MMseqs2 hit table parsed on the device (SURVEY §8f rank 2)
# ------------------------------------------------------------------------------------------------
def fnv1a64(strings):
    """FNV-1a 64-bit hashes of a list of ASCII / UTF-8 strings (numpy, one pass per character position) — the
    hash ``parse_tsv.cu`` computes over the id fields."""
    import numpy as np
    enc = [s.encode("utf-8") for s in strings]
    n = len(enc)
    lens = np.fromiter((len(b) for b in enc), dtype=np.int64, count=n)
    width = int(lens.max()) if n else 0
    # fixed-width byte matrix, zero padded (numpy 'S' arrays strip trailing NULs only on item access)
    mat = np.array(enc, dtype=f"S{max(width, 1)}").view(np.uint8).reshape(n, max(width, 1)) if n else \
        np.zeros((0, 1), dtype=np.uint8)
    h = np.full(n, 0xcbf29ce484222325, dtype=np.uint64)
    prime = np.uint64(0x100000001b3)
    with np.errstate(over="ignore"):
        for j in range(width):
            live = lens > j
            h[live] = (h[live] ^ mat[live, j].astype(np.uint64)) * prime
    return h


class GeneIdTable:
    """Sorted hash table of the known gene ids on the device: hash -> node id (position in ``gene_str_ids_lst``)."""

    def __init__(self, gene_ids, device):
        import numpy as np
        h = fnv1a64(gene_ids)
        order = np.argsort(h, kind="stable")
        hs = h[order]
        if hs.size > 1 and bool((hs[1:] == hs[:-1]).any()):
            raise _abi.PangnnError("gene ids collide under FNV-1a 64 (or are duplicated)")
        self.num_ids = len(gene_ids)
        self.hash = torch.from_numpy(hs.view(np.int64)).to(device)
        self.pos = torch.from_numpy(order.astype(np.int32)).to(device)


def parse_hits_tsv(text, table, score_col=15):
    """``text``: uint8 device tensor holding the TSV file.  -> (q, t, bits) of every data line in file order:
    int32 node ids (-1 = id not in ``table``), float64 scores; blank and ``#`` lines are dropped."""
    lib = _abi.load()
    _need_cuda(text)
    text = text.contiguous()
    n, dev = text.numel(), text.device
    if n == 0:
        z = torch.zeros(0, dtype=torch.int32, device=dev)
        return z, z.clone(), torch.zeros(0, dtype=torch.float64, device=dev)
    ws = _ws(lib.pangnn_parse_hits_tsv_workspace_bytes(n), dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_tsv_line_index(_p(text), n, None, 0, _p(cnt), _p(ws), ws.numel(), _stream()), "tsv_line_index")
    newlines = int(cnt.item())
    lines = newlines + (0 if int(text[-1].item()) == 10 else 1)
    line_start = torch.empty(newlines + 1, dtype=torch.int64, device=dev)
    _abi.check(lib.pangnn_tsv_line_index(_p(text), n, _p(line_start), newlines + 1, _p(cnt), _p(ws), ws.numel(),
                                         _stream()), "tsv_line_index")
    q = torch.empty(lines, dtype=torch.int32, device=dev)
    t = torch.empty(lines, dtype=torch.int32, device=dev)
    bits = torch.empty(lines, dtype=torch.float64, device=dev)
    _abi.check(lib.pangnn_tsv_parse_hits(_p(text), n, _p(line_start), lines, newlines, score_col, _p(table.hash),
                                         _p(table.pos), table.num_ids, _p(q), _p(t), _p(bits), _stream()),
               "tsv_parse_hits")
    LAUNCHES["count"] += 8
    data = q != -2
    return q[data], t[data], bits[data]



def _line_index(text):
    """-> (line_start int64 [newlines + 1], lines, newlines) of a uint8 device text (``pangnn_tsv_line_index``)."""
    lib = _abi.load()
    n, dev = text.numel(), text.device
    ws = _ws(lib.pangnn_parse_hits_tsv_workspace_bytes(n), dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    _abi.check(lib.pangnn_tsv_line_index(_p(text), n, None, 0, _p(cnt), _p(ws), ws.numel(), _stream()), "tsv_line_index")
    newlines = int(cnt.item())
    lines = newlines + (0 if int(text[-1].item()) == 10 else 1)
    line_start = torch.empty(newlines + 1, dtype=torch.int64, device=dev)
    _abi.check(lib.pangnn_tsv_line_index(_p(text), n, _p(line_start), newlines + 1, _p(cnt), _p(ws), ws.numel(),
                                         _stream()), "tsv_line_index")
    LAUNCHES["count"] += 6
    return line_start, lines, newlines


GFF_RECORD, GFF_COMPLETE, GFF_START, GFF_GENE_ID, GFF_COMPLEX = 1, 2, 4, 8, 16


def parse_gff(text, start_gene="hemB"):
    """GFF3 bytes (uint8 device tensor) -> per-gene device tensors ``(id_hash int64 (FNV-1a 64 bit pattern), id_off int64,
    id_len int32)`` in the reference's gene order (``src/preprocessing.py:329-367``): records rotated to the first
    one whose attribute mentions ``start_gene``, incomplete records dropped, ids that do not look like
    ``[A-Z]+_[0-9]+`` dropped.  One kernel over the lines + a scan / compaction of the flags."""
    lib = _abi.load()
    _need_cuda(text)
    text = text.contiguous()
    n, dev = text.numel(), text.device
    empty = (torch.zeros(0, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int64, device=dev),
             torch.zeros(0, dtype=torch.int32, device=dev))
    if n == 0:
        return empty
    line_start, lines, newlines = _line_index(text)
    flags = torch.empty(lines, dtype=torch.int32, device=dev)
    id_off = torch.empty(lines, dtype=torch.int64, device=dev)
    id_len = torch.empty(lines, dtype=torch.int32, device=dev)
    id_hash = torch.empty(lines, dtype=torch.int64, device=dev)
    sg = torch.tensor(list(start_gene.encode()), dtype=torch.uint8, device=dev)
    _abi.check(lib.pangnn_gff_parse_lines(_p(text), n, _p(line_start), lines, newlines, _p(sg), sg.numel(), _p(flags),
                                          _p(id_off), _p(id_len), _p(id_hash), _stream()), "gff_parse_lines")
    LAUNCHES["count"] += 1
    if bool((flags & GFF_COMPLEX).any()):
        raise _abi.PangnnError("GFF attribute with 'ID=' inside the id field: not handled by the device parser")
    rec = (flags & GFF_RECORD) != 0
    rank = torch.cumsum(rec.long(), 0) - 1                       # record index, as pandas numbers the rows
    R = int(rec.sum().item())
    starts = rank[rec & ((flags & GFF_START) != 0)]
    start = int(starts[0].item()) if starts.numel() else 1      # src/preprocessing.py:347-350
    keep = rec & ((flags & GFF_COMPLETE) != 0) & ((flags & GFF_GENE_ID) != 0)
    rot = torch.where(rank >= start, rank - start, rank + (R - start))       # position after the rotation
    order = torch.argsort(rot[keep], stable=True)
    return id_hash[keep][order], id_off[keep][order], id_len[keep][order]


def gather_strings(text_host, off, length):
    """Byte ranges of a host uint8 array -> list of str (vectorised: one fixed-width gather, one decode)."""
    import numpy as np
    off, length = np.asarray(off, dtype=np.int64), np.asarray(length, dtype=np.int64)
    if off.size == 0:
        return []
    width = int(length.max())
    idx = off[:, None] + np.arange(width, dtype=np.int64)[None, :]
    mat = text_host[np.minimum(idx, text_host.size - 1)]
    mat = np.where(np.arange(width)[None, :] < length[:, None], mat, 0).astype(np.uint8)
    return np.char.decode(mat.view(f"S{width}").reshape(-1), "utf-8").tolist()


def gene_id_table_from_hashes(id_hash, device):
    """``GeneIdTable`` from FNV-1a 64 hashes computed on the device (gene i = position i)."""
    t = object.__new__(GeneIdTable)
    key = id_hash ^ torch.tensor(-2 ** 63, dtype=torch.int64, device=id_hash.device)   # unsigned order as signed order
    order = torch.argsort(key, stable=True)
    hs = id_hash[order]
    if hs.numel() > 1 and bool((hs[1:] == hs[:-1]).any()):
        raise _abi.PangnnError("gene ids collide under FNV-1a 64 (or are duplicated)")
    t.num_ids, t.hash, t.pos = int(id_hash.numel()), hs.contiguous(), order.to(torch.int32).contiguous()
    return t


def lookup_columns(text, table, col_slot, num_slots):
    """Node id of the gene named in every kept column of every line of a tab-separated device text.
    -> (out int32 [lines, num_slots]: node id | -1 unknown | -2 missing, line_flag int32 [lines])."""
    lib = _abi.load()
    _need_cuda(text)
    text = text.contiguous()
    n, dev = text.numel(), text.device
    line_start, lines, newlines = _line_index(text)
    out = torch.empty(lines, num_slots, dtype=torch.int32, device=dev)
    flag = torch.empty(lines, dtype=torch.int32, device=dev)
    cs = torch.as_tensor(col_slot, dtype=torch.int32, device=dev).contiguous()
    _abi.check(lib.pangnn_tsv_lookup_columns(_p(text), n, _p(line_start), lines, newlines, _p(cs), cs.numel(), num_slots,
                                             _p(table.hash), _p(table.pos), table.num_ids, _p(out), _p(flag), _stream()),
               "tsv_lookup_columns")
    LAUNCHES["count"] += 1
    return out, flag
