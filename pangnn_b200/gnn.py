"""Model layer: drop-in for the reference's ``src/gnn.py`` module API on the CUDA kernels.

* ``GCNConv(in, out, add_self_loops=False)`` — same constructor / ``forward(x, edge_index,
  edge_weight=None)`` / parameter names (``bias`` then ``lin.weight``) as
  ``torch_geometric.nn.GCNConv`` as the reference uses it (``src/gnn.py:100-102,129-165``).
* ``AlternateGCN(device, dataset, categorical_nodes, dims=[64, 128])`` — same constructor,
  ``forward(graph) -> logits``, ``decode``, ``cosine_sim`` and ``state_dict()`` layout as
  ``src/gnn.py:84-207`` (SURVEY.md A.5); reads the global flags inside ``forward`` like the
  reference does.
"""
import math

import torch
from torch import nn

from . import ops
from .setup import args


_SIDE_STREAMS = {}

# Which spelling of the operators the modules below call: "function" = the torch.autograd.Function compositions
# of ops.py (default: least host overhead), "library" = the torch.library operators of torch_ops.py
# (``torch.ops.pangnn.*``: schemas, fake impls, registered autograd).  Same kernels, same order, bit-identical.
OPERATOR_LAYER = {"kind": "function"}


def set_operator_layer(kind):
    if kind not in ("function", "library"):
        raise ValueError("operator layer is 'function' or 'library'")
    OPERATOR_LAYER["kind"] = kind


def _side_stream(device):
    key = torch.device(device).index
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


class _Lin(nn.Module):
    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        a = math.sqrt(6.0 / (in_channels + out_channels))          # PyG 'glorot'
        nn.init.uniform_(self.weight, -a, a)


class GCNConv(nn.Module):
    def __init__(self, in_channels, out_channels, add_self_loops=False, **kw):
        super().__init__()
        if add_self_loops:
            raise NotImplementedError("the reference only uses add_self_loops=False")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.bias = nn.Parameter(torch.zeros(out_channels))        # registered before `lin` (A.1)
        self.lin = _Lin(in_channels, out_channels)

    def forward(self, x, edge_index, edge_weight=None, _act=ops.ACT_NONE):
        if OPERATOR_LAYER["kind"] == "library":
            from . import torch_ops
            return torch_ops.gcn_conv(x.contiguous(), self.lin.weight, self.bias, edge_index, edge_weight, _act)
        return ops.gcn_layer(x, self.lin.weight, self.bias, edge_index, edge_weight, _act)


class AlternateGCN(nn.Module):
    def __init__(self, device, dataset, categorical_nodes, dims=[64, 128]):
        super().__init__()
        self.device = device
        node_embedding_dim, hidden_dim = dims
        if categorical_nodes:
            # The reference crashes here (len() of a list of graphs, float indices; SURVEY.md F6).
            # Defined behaviour (A.6): one embedding row per gene of the whole graph, indexed by
            # the gene's global position.
            num = dataset if isinstance(dataset, int) else int(getattr(dataset, "num_genes", 0) or len(dataset.x))
            self.embedding = nn.Embedding(num, node_embedding_dim)
        else:
            self.embedding = nn.Linear(1, node_embedding_dim)
        self.conv_in = GCNConv(node_embedding_dim, hidden_dim, add_self_loops=False)
        self.conv_hidden = GCNConv(hidden_dim, hidden_dim, add_self_loops=False)
        self.conv_out = GCNConv(hidden_dim, node_embedding_dim, add_self_loops=False)
        self.linear_out = nn.Linear(hidden_dim, node_embedding_dim)
        self.activation_fct = nn.ELU()
        self.mlp = nn.Sequential(
            nn.Linear(node_embedding_dim * 2 + (1 if args.skip_connections else 0), node_embedding_dim),
            nn.ReLU(),
            nn.Linear(node_embedding_dim, node_embedding_dim),
            nn.ReLU(),
            nn.Linear(node_embedding_dim, 1))
        self.epoch = 0
        self._categorical = bool(categorical_nodes)
        self.fuse_embedding = True        # Linear(1, D) + conv_in as one rank-2 update when x is [N, 1]

    # -- node embeddings after the convolutions (src/gnn.py:125-166) ------------------------------
    def embed(self, graph):
        ELU = ops.ACT_ELU
        if (not self._categorical and graph.x.dim() == 2 and graph.x.size(1) == 1 and self.fuse_embedding
                and OPERATOR_LAYER["kind"] == "function"
                and self.conv_in.out_channels % 4 == 0 and self.conv_in.out_channels <= 256):
            # scalar node features: Linear(1, D) + conv_in collapse into one rank-2 update (ops.RankOneFn)
            ei = graph.union_edge_index if args.union_edge_weights else graph.edge_index
            emb, cin = self.embedding, self.conv_in
            nodes = ops.embed_conv(graph.x, emb.weight, emb.bias, cin.lin.weight, cin.bias, ei, graph.edge_attr, ELU)
            return self._embed_tail(graph, nodes)
        if self._categorical:
            idx = graph.x if graph.x.dtype == torch.long else (
                graph.node_id if hasattr(graph, "node_id") else
                torch.arange(graph.x.size(0), device=graph.x.device))
            node_embeddings = self.embedding(idx)
        elif graph.x.dim() == 2 and graph.x.size(1) == 1:
            # Linear(1, D) (src/gnn.py:97,125) is an outer product: x w^T + b as ONE broadcast elementwise pass
            # instead of a K = 1 library GEMM (0.18 ms at N = 1e6) — same values, same parameters
            node_embeddings = torch.addcmul(self.embedding.bias, graph.x, self.embedding.weight.t())
        else:
            node_embeddings = self.embedding(graph.x)
        ei = graph.union_edge_index if args.union_edge_weights else graph.edge_index
        nodes = self.conv_in(node_embeddings, ei, graph.edge_attr, _act=ELU)
        return self._embed_tail(graph, nodes)

    def _embed_tail(self, graph, nodes):
        """The layers after ``conv_in`` + ELU (``src/gnn.py:131-166``)."""
        ELU = ops.ACT_ELU
        if args.union_edge_weights:
            for _ in range(max(args.neighbours - 2, 1)):
                nodes = self.conv_hidden(nodes, graph.union_edge_index, graph.edge_attr, _act=ELU)
            nodes = self.conv_out(nodes, graph.union_edge_index, None, _act=ELU)
        elif args.base_model:
            nodes = self.activation_fct(self.linear_out(nodes))
        else:
            nodes = self.conv_out(nodes, graph.neighbour_edge_index, None, _act=ELU)
        return nodes

    def _skip(self, graph):
        # literal slice of the reference, src/gnn.py:173 (A.4: union graphs slice the union weights)
        if not args.skip_connections:
            return None
        return graph.edge_attr[:graph.edge_index.size(1)].contiguous().float()

    def _use_fused_mlp(self, nodes):
        return "mlp" in args.decoder and nodes.size(1) == ops.SCORER_D

    def forward(self, graph):
        nodes = self.embed(graph)
        gs = ops.graph_struct(graph.edge_index, nodes.size(0))
        link_predictions = None
        if "mlp" in args.decoder:
            if self._use_fused_mlp(nodes):
                m = self.mlp
                link_predictions = ops.EdgeScoreFn.apply(
                    nodes, m[0].weight, m[0].bias, m[2].weight, m[2].bias, m[4].weight, m[4].bias,
                    gs, self._skip(graph))
            else:
                src, dst = graph.edge_index[0], graph.edge_index[1]
                parts = (nodes[src], nodes[dst]) + ((self._skip(graph).unsqueeze(1),)
                                                    if args.skip_connections else ())
                link_predictions = self.mlp(torch.cat(parts, dim=1)).squeeze(-1)
        if "cosine" in args.decoder:
            link_predictions = self.cosine_sim(nodes, graph.edge_index)
        if "dot" in args.decoder:
            link_predictions = self.decode(nodes, graph.edge_index)
        return link_predictions

    @torch.no_grad()
    def predict(self, graph, threshold=None):
        """``model.eval(); sigmoid(model(batch)) >= threshold`` of the reference (``src/predict.py:29-55``,
        ``pangnn.py:220-221``) with sigmoid and threshold fused into the scorer kernel:
        -> (logits, probabilities, int32 predictions)."""
        th = args.binary_threshold if threshold is None else threshold
        nodes = self.embed(graph)
        if not self._use_fused_mlp(nodes) or args.decoder != "mlp":
            logits = self.forward(graph)
            prob = torch.sigmoid(logits)
            return logits, prob, (prob >= th).to(torch.int32)
        gs = ops.graph_struct(graph.edge_index, nodes.size(0))
        m = self.mlp
        skip = self._skip(graph)
        wcat, w1c = ops.split_w1(m[0].weight, skip is not None)
        pq = ops.node_linear(nodes, wcat)
        return ops.edge_score_predict(pq, w1c, m[0].bias, m[2].weight, m[2].bias, m[4].weight, m[4].bias, gs, skip, th)

    @staticmethod
    def transfer_order(scored_only=False):
        """Host-to-device order for ``Data.to_pipelined`` under the current flags: the first convolution's
        structure and weights first, the scored-edge list and labels (needed last, by the scorer) last."""
        if scored_only:
            return ("edge_index", "edge_attr", "x", "y")
        if args.union_edge_weights:
            return ("union_edge_index", "edge_attr", "x", "edge_index", "y")
        return ("edge_index", "edge_attr", "x", "neighbour_edge_index", "y")

    def prepare(self, graph):
        """Build (and cache) the CSR structures of a batch as its tensors arrive.  With a batch from
        ``Data.to_pipelined(device, order=model.transfer_order())`` the convolution structure is sorted while
        the rest is still on the PCIe bus, and (union mode) the scored-edge structure is built on a side
        stream underneath the convolution layers: the scorer is the first kernel that waits for it.
        Optional: ``forward`` builds on demand otherwise.

        A whole-graph batch may arrive as the SCORED edges only (``x, edge_index [2,E], edge_attr [E], y``
        with neither ``union_edge_index`` nor ``neighbour_edge_index``): the neighbour band (a8,
        ``src/dataset.py:351-366``) and the union assembly (a11, ``:373-381``) are then done here on the
        device instead of travelling over PCIe (the band is a function of N and ``--neighbours`` alone)."""
        wait = getattr(graph, "wait", lambda *a: graph)
        ready = getattr(graph, "_ready", None) or {}
        n = graph.x.size(0)
        main = torch.cuda.current_stream()
        if args.union_edge_weights:
            if getattr(graph, "union_edge_index", None) is None:            # a8 + a11 on the device
                wait("edge_index")
                sim = ops.graph_struct(graph.edge_index, n)
                graph.union_edge_index = ops.union_index(graph.edge_index, n, args.neighbours)
                ops.graph_struct_union(graph.union_edge_index, n, sim, args.neighbours)   # merge, not sort
                sim.endpoints32
                wait(*[k for k in ("edge_attr", "x", "y") if k in ready])
                graph.edge_attr = ops.union_weights(graph.edge_attr, graph.union_edge_index.size(1))
                return graph
            wait("union_edge_index")
            ops.graph_struct(graph.union_edge_index, n).src
            if "mlp" in args.decoder:
                side = _side_stream(graph.x.device)
                side.wait_stream(main)                                      # allocator: blocks handed over in order
                with torch.cuda.stream(side):
                    if ready.get("edge_index") is not None:
                        side.wait_event(ready["edge_index"])
                    gs = ops.graph_struct(graph.edge_index, n)
                    gs.src, gs.endpoints32
                    gs.built_on(side, main)
                graph.edge_index.record_stream(side)
            wait(*[k for k in ("edge_attr", "x", "y") if k in ready])
            return graph
        wait("edge_index")
        gs = ops.graph_struct(graph.edge_index, n)
        gs.src, gs.endpoints32
        if not args.base_model:
            if getattr(graph, "neighbour_edge_index", None) is None:        # a8 on the device
                graph.neighbour_edge_index = ops.neighbour_band(n, args.neighbours, graph.edge_index.device)
            wait("neighbour_edge_index")
            ops.graph_struct(graph.neighbour_edge_index, n).src
        wait()
        return graph

    def forward_loss(self, graph, pos_weight):
        """Fused training form of ``criterion(model(batch), batch.y)`` (``pangnn.py:200-203``):
        returns ``(loss, logits)`` with logits detached; one kernel for scorer + loss + gradients."""
        if not self._use_fused_mlp_flag():
            logits = self.forward(graph)
            loss = torch.nn.functional.binary_cross_entropy_with_logits(
                logits, graph.y, pos_weight=torch.as_tensor(float(pos_weight), device=logits.device))
            return loss, logits.detach()
        nodes = self.embed(graph)
        gs = ops.graph_struct(graph.edge_index, nodes.size(0))
        m = self.mlp
        if OPERATOR_LAYER["kind"] == "library":
            from . import torch_ops
            return torch_ops.score_edges_bce(nodes, m[0].weight, m[0].bias, m[2].weight, m[2].bias, m[4].weight,
                                             m[4].bias, graph.edge_index, self._skip(graph), graph.y, float(pos_weight))
        return ops.EdgeScoreBCEFn.apply(
            nodes, m[0].weight, m[0].bias, m[2].weight, m[2].bias, m[4].weight, m[4].bias,
            gs, self._skip(graph), graph.y, float(pos_weight))

    def _use_fused_mlp_flag(self):
        return args.decoder == "mlp" and self.mlp[2].weight.size(0) == ops.SCORER_D

    def decode(self, z, edge_index):
        # The reference's `z[src] @ z[dst]` is shape-broken (SURVEY.md F6); the intended row-wise
        # dot product is MyGCN.decode, src/gnn.py:77-79.
        return ops.edge_pair_score(z, ops.graph_struct(edge_index, z.size(0)), 1)

    def cosine_sim(self, z, edge_index):
        return ops.edge_pair_score(z, ops.graph_struct(edge_index, z.size(0)), 0)
