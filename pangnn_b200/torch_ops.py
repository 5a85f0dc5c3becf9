"""``torch.library`` registration of the hot-path operators over the same C ABI (``include/pangnn_b200.h``).

``BASELINE.json:north_star`` asks for "a thin C-ABI PyTorch custom-op layer": the kernels are reached through
``ctypes`` (``_abi.py``), and this module makes them first-class PyTorch operators — ``torch.ops.pangnn.*`` with
schemas, fake (meta) implementations for shape propagation / tracing, and autograd formulas
(``register_autograd``) — so that code written against the reference's module API (``GCNConv.forward``,
``AlternateGCN.forward``; ``src/gnn.py:100-177``) can be traced, ``opcheck``-ed and captured like any other
PyTorch program.  ``ops.py`` keeps the ``torch.autograd.Function`` spelling of the same compositions (less
dispatcher overhead per call, which matters for the reference's ``-b 32`` regime); both call the same kernels in
the same order and are bit-identical (``tests/test_gpu_torch_ops.py``).

Operators (all tensors CUDA; structure tensors as produced by ``ops.GraphStruct``):

* ``pangnn::node_linear(x, weight, bias?, act, w_is_kn) -> y``                       K3: ``act(x W^T + b)``
* ``pangnn::gcn_propagate(x, bias?, rowptr_dst, col_dst, val_dst?, rowptr_src, col_src, val_src?, n_out, act) -> y``
  ``act(A_hat x + b)``: PyG ``GCNConv.propagate`` + bias (+ELU); backward walks the by-source CSR
* ``pangnn::gcn_norm(rowptr, col, perm, weight?, num_rows) -> (dis, val)``             PyG ``gcn_norm``
* ``pangnn::edge_score(pq, src, dst, skip?, w1c?, b1, w2, b2, w3, b3) -> logits``     ``src/gnn.py:171-177`` (inference)
* ``pangnn::edge_score_bce(pq, src, dst, skip?, w1c?, b1, w2, b2, w3, b3, y, pos_weight, scale, rowptr_src,
  perm_src, rowptr_dst, perm_dst) -> (loss, logits, da1, grads)``                     fused scorer + BCE(pos_weight)
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import ops

D = ops.SCORER_D


# ------------------------------------------------------------------------------------------------
# node_linear
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("pangnn::node_linear", mutates_args=())
def node_linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], act: int, w_is_kn: bool) -> Tensor:
    return ops.node_linear(x.contiguous(), weight, bias, act, w_is_kn=w_is_kn)


@node_linear.register_fake
def _(x, weight, bias, act, w_is_kn):
    return x.new_empty(x.size(0), weight.size(1) if w_is_kn else weight.size(0))


def _node_linear_setup(ctx, inputs, output):
    x, weight, bias, act, w_is_kn = inputs
    ctx.act, ctx.has_bias, ctx.w_is_kn = act, bias is not None, w_is_kn
    ctx.save_for_backward(x, weight, output if act != ops.ACT_NONE else None)


def _node_linear_backward(ctx, dy):
    x, weight, y = ctx.saved_tensors
    if ctx.w_is_kn:
        raise NotImplementedError("pangnn::node_linear: autograd is defined for weight [out, in] (w_is_kn = False)")
    if ctx.act != ops.ACT_NONE or ctx.has_bias:
        g, dbias = torch.ops.pangnn.act_bwd_bias(dy.contiguous(), y, ctx.act)
    else:
        g, dbias = dy.contiguous(), None
    dW = torch.ops.pangnn.gemm_tn(g, x) if ctx.needs_input_grad[1] else None
    dx = torch.ops.pangnn.node_linear(g, weight, None, ops.ACT_NONE, True) if ctx.needs_input_grad[0] else None
    return dx, dW, (dbias if ctx.has_bias and ctx.needs_input_grad[2] else None), None, None


node_linear.register_autograd(_node_linear_backward, setup_context=_node_linear_setup)


@torch.library.custom_op("pangnn::act_bwd_bias", mutates_args=())
def act_bwd_bias(dy: Tensor, y: Optional[Tensor], act: int) -> Tuple[Tensor, Tensor]:
    g, db = ops.act_bwd_bias(dy, y, act)
    return (g.clone() if g is dy else g), db             # an output must not alias an input


@act_bwd_bias.register_fake
def _(dy, y, act):
    return torch.empty_like(dy), dy.new_empty(dy.size(1))


@torch.library.custom_op("pangnn::gemm_tn", mutates_args=())
def gemm_tn(a: Tensor, b: Tensor) -> Tensor:
    return ops.gemm_tn(a, b)


@gemm_tn.register_fake
def _(a, b):
    return a.new_empty(a.size(1), b.size(1))


# ------------------------------------------------------------------------------------------------
# gcn_norm / gcn_propagate
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("pangnn::gcn_norm", mutates_args=())
def gcn_norm(rowptr: Tensor, col: Tensor, perm: Tensor, weight: Optional[Tensor], num_rows: int) -> Tuple[Tensor, Tensor]:
    csr = ops.CSR(rowptr, col, perm, num_rows, col.numel(), True)
    return ops.gcn_norm(csr, weight)


@gcn_norm.register_fake
def _(rowptr, col, perm, weight, num_rows):
    return rowptr.new_empty(num_rows, dtype=torch.float32), col.new_empty(col.numel(), dtype=torch.float32)


@torch.library.custom_op("pangnn::gcn_aggregate", mutates_args=())
def gcn_aggregate(rowptr: Tensor, col: Tensor, val: Optional[Tensor], x: Tensor, num_rows: int,
                  bias: Optional[Tensor], act: int) -> Tensor:
    return ops.gcn_aggregate(rowptr, col, val, x.contiguous(), num_rows, bias, act)


@gcn_aggregate.register_fake
def _(rowptr, col, val, x, num_rows, bias, act):
    return x.new_empty(num_rows, x.size(1))


@torch.library.custom_op("pangnn::gcn_propagate", mutates_args=())
def gcn_propagate(x: Tensor, bias: Optional[Tensor], rowptr_dst: Tensor, col_dst: Tensor, val_dst: Optional[Tensor],
                  rowptr_src: Tensor, col_src: Tensor, val_src: Optional[Tensor], n_out: int, act: int) -> Tensor:
    return ops.gcn_aggregate(rowptr_dst, col_dst, val_dst, x.contiguous(), n_out, bias, act)


@gcn_propagate.register_fake
def _(x, bias, rowptr_dst, col_dst, val_dst, rowptr_src, col_src, val_src, n_out, act):
    return x.new_empty(n_out, x.size(1))


def _propagate_setup(ctx, inputs, output):
    x, bias, _, _, _, rowptr_src, col_src, val_src, _, act = inputs
    ctx.act, ctx.has_bias, ctx.n_in = act, bias is not None, x.size(0)
    ctx.save_for_backward(rowptr_src, col_src, val_src, output if act != ops.ACT_NONE else None)


def _propagate_backward(ctx, dy):
    rowptr_src, col_src, val_src, y = ctx.saved_tensors
    if ctx.act != ops.ACT_NONE or ctx.has_bias:
        g, dbias = torch.ops.pangnn.act_bwd_bias(dy.contiguous(), y, ctx.act)
    else:
        g, dbias = dy.contiguous(), None
    dx = torch.ops.pangnn.gcn_aggregate(rowptr_src, col_src, val_src, g, ctx.n_in, None, ops.ACT_NONE)
    return (dx, (dbias if ctx.has_bias else None)) + (None,) * 8


gcn_propagate.register_autograd(_propagate_backward, setup_context=_propagate_setup)


# ------------------------------------------------------------------------------------------------
# edge scorer
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("pangnn::edge_score", mutates_args=())
def edge_score(pq: Tensor, src: Tensor, dst: Tensor, skip: Optional[Tensor], w1c: Optional[Tensor], b1: Tensor,
               w2: Tensor, b2: Tensor, w3: Tensor, b3: Tensor) -> Tensor:
    return ops.edge_score_pq_fwd(pq, w1c, b1, w2, b2, w3, b3, (src, dst), skip)


@edge_score.register_fake
def _(pq, src, dst, skip, w1c, b1, w2, b2, w3, b3):
    return pq.new_empty(src.numel())


@torch.library.custom_op("pangnn::edge_score_bce", mutates_args=())
def edge_score_bce(pq: Tensor, src: Tensor, dst: Tensor, skip: Optional[Tensor], w1c: Optional[Tensor], b1: Tensor,
                   w2: Tensor, b2: Tensor, w3: Tensor, b3: Tensor, y: Tensor, pos_weight: float, scale: float,
                   rowptr_src: Tensor, perm_src: Tensor, rowptr_dst: Tensor, perm_dst: Tensor
                   ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (sum of the per-edge losses * scale, logits, da1 [E, 64], small gradients [NGRADS]); the last two are
    what the backward consumes (the fused kernel produces every gradient in the forward pass)."""
    logits = torch.empty(src.numel(), dtype=torch.float32, device=pq.device)
    loss_sum = torch.zeros(1, dtype=torch.float64, device=pq.device)
    da1, grads = ops.edge_score_train(pq, w1c, b1, w2, b2, w3, b3, (src, dst), skip, y=y, pos_weight=pos_weight,
                                      scale=scale, logits=logits, loss_sum=loss_sum)
    return (loss_sum * scale).float().squeeze(0), logits, da1, grads


@edge_score_bce.register_fake
def _(pq, src, dst, skip, w1c, b1, w2, b2, w3, b3, y, pos_weight, scale, rowptr_src, perm_src, rowptr_dst, perm_dst):
    E = src.numel()
    return pq.new_empty(()), pq.new_empty(E), pq.new_empty(E, D), pq.new_empty(ops.NGRADS)


def _score_bce_setup(ctx, inputs, output):
    pq, _, _, skip = inputs[:4]
    rowptr_src, perm_src, rowptr_dst, perm_dst = inputs[13:17]
    _, _, da1, grads = output
    ctx.n, ctx.has_skip = pq.size(0), skip is not None
    ctx.save_for_backward(da1, grads, rowptr_src, perm_src, rowptr_dst, perm_dst)


def _score_bce_backward(ctx, dloss, _dlogits, _dda1, _dgrads):
    da1, grads, rowptr_src, perm_src, rowptr_dst, perm_dst = ctx.saved_tensors
    n = ctx.n
    # per-node gradients of the two pq halves: sorted-segment sums of da1 over both orientations
    dp = torch.ops.pangnn.gcn_aggregate(rowptr_src, perm_src, None, da1, n, None, ops.ACT_NONE)
    dq = torch.ops.pangnn.gcn_aggregate(rowptr_dst, perm_dst, None, da1, n, None, ops.ACT_NONE)
    dpq = torch.cat((dp, dq), dim=1) * dloss
    g = ops.scorer_grads(grads * dloss)
    return (dpq, None, None, None, g.dw1c if ctx.has_skip else None, g.db1, g.dW2, g.db2, g.dw3, g.db3) + (None,) * 7


edge_score_bce.register_autograd(_score_bce_backward, setup_context=_score_bce_setup)


# ------------------------------------------------------------------------------------------------
# the reference's module API spelled with the registered operators
# ------------------------------------------------------------------------------------------------
def gcn_conv(x, weight, bias, edge_index, edge_weight=None, act=ops.ACT_NONE):
    """``GCNConv(add_self_loops=False).forward`` (+ optional fused ELU), ``src/gnn.py:129-165``: gcn_norm once per
    (structure, weights) from the structure cache, then ``node_linear`` and ``gcn_propagate`` in the order of
    ``ops.aggregate_first``, as ``ops.gcn_layer``."""
    gs = ops.graph_struct(edge_index, x.size(0))
    ent = gs.norm(edge_weight, need_src=True)
    d, s = gs.dst, gs.src
    csr = (d.rowptr, d.col, ent["dst"], s.rowptr, s.col, ent["src"], gs.num_nodes)
    P = torch.ops.pangnn
    if ops.aggregate_first(weight):
        return P.node_linear(P.gcn_propagate(x, None, *csr, ops.ACT_NONE), weight, bias, act, False)
    return P.gcn_propagate(P.node_linear(x, weight, None, ops.ACT_NONE, False), bias, *csr, act)


def score_edges_bce(h, w1, b1, w2, b2, w3, b3, edge_index, skip, y, pos_weight, num_labelled=None):
    """``criterion(mlp(cat(h[src], h[dst] (, skip))), y)`` (``src/gnn.py:171-177``, ``pangnn.py:98,203``), mean
    reduction: -> (loss, logits).  Layer 1 of the MLP is hoisted to the nodes (``pq = h [W1a ; W1b]^T``).
    ``num_labelled``: the number of edges with ``y >= 0`` (held-out edges carry ``y = -1``, ``edge_split``), the
    divisor of the mean and the kernel's ``scale``; None = every edge."""
    gs = ops.graph_struct(edge_index, h.size(0))
    src, dst = gs.endpoints32
    wcat, w1c = ops.split_w1(w1, skip is not None)
    P = torch.ops.pangnn
    pq = P.node_linear(h, wcat, None, ops.ACT_NONE, False)
    n = max(gs.num_edges if num_labelled is None else int(num_labelled), 1)
    loss, logits, _, _ = P.edge_score_bce(pq, src, dst, skip, w1c, b1, w2, b2, w3, b3, y, float(pos_weight),
                                          1.0 / n, gs.src.rowptr, gs.src.perm, gs.dst.rowptr, gs.dst.perm)
    return loss, logits.detach()
