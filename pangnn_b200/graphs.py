"""CUDA-graph replay of a static-shape training step.

A whole-graph step over a small pan-genome (BASELINE.json configs[0..1]: the graph lives in L2) is
~90 kernel launches of a few microseconds each — launch-latency-bound, not bandwidth-bound.  When the
same graph is stepped repeatedly (whole-graph epochs, ``pangnn.py:167-238`` with one batch), the step is
captured once and replayed: one launch per step, no Python between kernels.
"""
import torch


class GraphedStep:
    """``loss = GraphedStep(model, graph, optimizer, pos_weight)()`` replays one fused
    forward + BCE loss + backward + optimizer step.  The graph tensors must not be reallocated; parameter
    and optimizer state are updated in place exactly as by the eager step.  ``optimizer`` must be built
    with ``capturable=True`` (Adam)."""

    def __init__(self, model, graph, optimizer, pos_weight, warmup=3):
        self.model, self.graph, self.opt, self.pw = model, graph, optimizer, float(pos_weight)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                       # warm-up off the capturing stream: lazy inits, CSR cache
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.cuda_graph = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=True)
        with torch.cuda.graph(self.cuda_graph):
            self.loss = self._eager()

    def _eager(self):
        self.opt.zero_grad(set_to_none=True)
        loss, self.logits = self.model.forward_loss(self.graph, self.pw)
        loss.backward()
        self.opt.step()
        return loss

    def __call__(self):
        self.cuda_graph.replay()
        return self.loss


class GraphedBatchStep:
    """The reference's own training regime — ``-b 32`` batches of per-ortholog-group sub-graphs, ~300 scored edges
    and ~60 small launches per step (``pangnn.py:180-222``; SURVEY F7) — is bound by Python / autograd dispatch, not
    by the device.  This replays the whole step (CSR builds, gcn_norm, forward, BCE(pos_weight) loss, backward,
    Adam) as ONE CUDA graph per size bucket:

    * a batch is copied into static buffers padded to a bucket ``(nodes, edges per edge list)`` rounded up to
      ``node_quantum`` / ``edge_quantum``; pad nodes are isolated, pad edges are self loops on the last pad node
      (they only ever touch that node's row), and the loss is the masked sum ``sum_e mask_e bce(z_e, y_e) / E`` with
      ``1 / E`` in device memory — so the real rows, logits, loss and gradients are those of the eager step up to the
      summation order of the loss;
    * the first batch of a bucket captures its graph (forward + backward + optimizer step, after a side-effect-free
      warm-up), later batches of that bucket are a handful of small copies + one graph launch.

    ``optimizer`` must be ``torch.optim.Adam(..., capturable=True)``; its learning rate is baked into the captured
    graphs (a scheduler that replaces ``param_group['lr']`` is not seen by them).  Batches whose edge lists exceed the
    single-launch CSR build (4096 edges) fall back to the eager step.

    ``reduce_grads`` (data-parallel training, ``dist.GradReducer``) runs between ``loss.backward()`` and
    ``opt.step()`` of the eager step and of the captured graph, never in the capture's warm-up: ranks capture their
    buckets at different times, and a collective there would put their reductions out of step.

        stepper = GraphedBatchStep(model, optimizer, dataset.class_balance)
        for batch in DeviceLoader(dataset.train, batch_size=32, ...):
            loss, logits = stepper(batch)
    """

    def __init__(self, model, optimizer, pos_weight, node_quantum=64, edge_quantum=128, max_buckets=128,
                 reduce_grads=None):
        from . import ops
        self.model, self.opt, self.pw = model, optimizer, float(pos_weight)
        self.reduce_grads = reduce_grads
        self.nq, self.eq, self.max_buckets = int(node_quantum), int(edge_quantum), int(max_buckets)
        self.buckets = {}
        self.stats = {"captures": 0, "replays": 0, "eager": 0}
        self._small = ops.SMALL_CSR_EDGES
        dev = next(model.parameters()).device
        self._pw_t = torch.tensor(self.pw, device=dev)
        # Adam's state must exist before the first capture: one step with zero gradients leaves every parameter
        # untouched (update = 0 / (sqrt(0) + eps)); the step counters are put back to 0 afterwards
        if not any(len(optimizer.state.get(p, {})) for g in optimizer.param_groups for p in g["params"]):
            for g in optimizer.param_groups:
                for p in g["params"]:
                    if p.requires_grad:
                        p.grad = torch.zeros_like(p)
            optimizer.step()
            for st in optimizer.state.values():
                if torch.is_tensor(st.get("step")):
                    st["step"].zero_()
            optimizer.zero_grad(set_to_none=True)

    # -- padding ----------------------------------------------------------------------------------------------
    @staticmethod
    def _tensor_keys(batch):
        return [k for k, v in batch.__dict__.items() if torch.is_tensor(v) and k not in ("batch", "ptr")]

    def _bucket_key(self, batch):
        up = lambda v, q: (int(v) + q - 1) // q * q
        n = batch.x.size(0)
        key = [("#nodes", up(n + 1, self.nq))]                      # at least one pad node
        for k in self._tensor_keys(batch):
            v = batch.__dict__[k]
            if k == "x" or (v.dim() >= 1 and v.size(0) == n and "index" not in k and k not in ("y", "edge_attr")):
                continue                                            # node-sized: follows #nodes
            key.append((k, up(v.size(-1) if "index" in k else v.size(0), self.eq)))
        return tuple(key)

    def _alloc(self, key, batch):
        from .data import Data
        sizes = dict(key)
        nb, n = sizes["#nodes"], batch.x.size(0)
        g = Data()
        for k in self._tensor_keys(batch):
            v = batch.__dict__[k]
            if k in sizes:
                shape = (2, sizes[k]) if "index" in k else (sizes[k],) + tuple(v.shape[1:])
            else:
                shape = (nb,) + tuple(v.shape[1:])
            g.__dict__[k] = torch.zeros(shape, dtype=v.dtype, device=v.device)
        g._mask = torch.zeros(sizes["y"], dtype=torch.float32, device=batch.y.device)
        g._inv = torch.zeros(1, dtype=torch.float32, device=batch.y.device)
        return g

    def _load(self, g, key, batch):
        sizes = dict(key)
        nb, n = sizes["#nodes"], batch.x.size(0)
        pad_node = nb - 1
        for k in self._tensor_keys(batch):
            v, s = batch.__dict__[k], g.__dict__[k]
            if "index" in k:
                m = v.size(1)
                s[:, :m].copy_(v)
                s[:, m:].fill_(pad_node)                            # self loops on the last pad node
            elif k in sizes:
                m = v.size(0)
                s[:m].copy_(v)
                s[m:].fill_(1.0 if k == "edge_attr" else 0)
            else:                                                   # node-sized (x, node_id)
                s[:n].copy_(v)
                s[n:].fill_(1.0 if k == "x" else 0)
        E = batch.y.size(0)
        g._mask[:E].fill_(1.0)
        g._mask[E:].zero_()
        g._inv.fill_(1.0 / max(E, 1))

    # -- the step ---------------------------------------------------------------------------------------------
    def _loss(self, g):
        logits = self.model(g)
        per = torch.nn.functional.binary_cross_entropy_with_logits(logits, g.y, pos_weight=self._pw_t, reduction="none")
        return (per * g._mask).sum() * g._inv.squeeze(0), logits

    def _capture(self, g):
        from . import ops
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        self.opt.zero_grad(set_to_none=True)
        with torch.cuda.stream(side):                               # warm-up WITHOUT the optimizer step: lazy inits only
            for _ in range(2):
                ops.clear_cache()
                loss, _ = self._loss(g)
                loss.backward()
                self.opt.zero_grad(set_to_none=True)
                del loss
        ops.clear_cache()                                           # the structure builds belong INTO the graph
        cg = torch.cuda.CUDAGraph()
        # captured on the warm-up stream: the parameters' AccumulateGrad nodes were created on it (a node kept alive
        # from an earlier backward on another stream — e.g. by a loss tensor the caller still holds — would break the
        # capture: drop such references before the first call).  Private memory pool per bucket: buckets are replayed
        # in any order.
        with torch.cuda.graph(cg, stream=side):
            self.opt.zero_grad(set_to_none=True)
            loss, logits = self._loss(g)
            loss.backward()
            if self.reduce_grads is not None:
                self.reduce_grads()
            self.opt.step()
        torch.cuda.current_stream().wait_stream(side)
        ops.clear_cache()
        self.stats["captures"] += 1
        return cg, loss, logits.detach()

    def _eager(self, batch):
        self.opt.zero_grad(set_to_none=True)
        loss, logits = self.model.forward_loss(batch, self.pw)
        loss.backward()
        if self.reduce_grads is not None:
            self.reduce_grads()
        self.opt.step()
        self.stats["eager"] += 1
        return loss.detach(), logits

    def step_ids(self, packed, ids, ids_dev):
        """The step for the graphs ``ids`` of a device-resident split (``DeviceLoader.iter_ids()``): the batch is
        collated by ``pangnn_collate`` STRAIGHT into the bucket's static buffers (one multi-tensor copy restores the
        padding first), so a step is ~6 launches: restore, collate (2), mask, 1 / E, graph replay.
        -> (loss, logits of the batch's scored edges)."""
        up = lambda v, q: (int(v) + q - 1) // q * q
        tot, n = packed.sizes(ids)
        E = tot["y"]
        key = (("#nodes", up(n + 1, self.nq)),) + tuple(
            (k, up(m, self.eq)) for k, m in tot.items() if "index" in k or k in ("y", "edge_attr"))
        if any("index" in k and m > self._small for k, m in key) or \
                (key not in self.buckets and len(self.buckets) >= self.max_buckets):
            b = packed.collate(ids, ids_dev)
            self.last_y = b.y
            return self._eager(b)
        ent = self.buckets.get(key)
        fresh = ent is None
        if fresh:
            sizes = dict(key)
            nb = sizes["#nodes"]
            from .data import Data
            g = Data()
            for k in packed.tensor_keys:
                a = packed.attrs[k]
                rows = sizes.get(k, nb)
                shape = (2, rows) if a["rows"] == 2 else (rows,) + tuple(a["tail"])
                fillv = (nb - 1) if a["rows"] == 2 else (1.0 if k in ("x", "edge_attr") else 0)
                g.__dict__[k] = torch.full(shape, fillv, dtype=a["dtype"], device=packed.device)
            g._mask = torch.zeros(sizes["y"], dtype=torch.float32, device=packed.device)
            g._inv = torch.zeros(1, dtype=torch.float32, device=packed.device)
            g._batch_vec = torch.zeros(nb, dtype=torch.int64, device=packed.device)
            g._statics = [g.__dict__[k] for k in packed.tensor_keys] + [g._mask]
            g._templates = [t.clone() for t in g._statics]
        else:
            g = ent[0]
            torch._foreach_copy_(g._statics, g._templates)          # padding (and a zero mask) back in place
        packed.collate_into(ids, ids_dev, {k: g.__dict__[k] for k in packed.tensor_keys}, g._batch_vec)
        g._mask[:E].fill_(1.0)
        g._inv.fill_(1.0 / max(E, 1))
        if fresh:
            cg, loss, logits = self._capture(g)
            ent = self.buckets[key] = (g, cg, loss, logits)
        g, cg, loss, logits = ent
        cg.replay()
        self.stats["replays"] += 1
        self.last_y = g.y[:E]                                       # labels of this batch (valid until the next call)
        return loss, logits[:E]

    def __call__(self, batch):
        key = self._bucket_key(batch)
        if any(k != "#nodes" and "index" in k and m > self._small for k, m in key) or \
                (key not in self.buckets and len(self.buckets) >= self.max_buckets):
            return self._eager(batch)
        ent = self.buckets.get(key)
        if ent is None:
            g = self._alloc(key, batch)
            self._load(g, key, batch)
            cg, loss, logits = self._capture(g)                     # capture does not execute: replay below
            ent = self.buckets[key] = (g, cg, loss, logits)
        else:
            self._load(ent[0], key, batch)
        g, cg, loss, logits = ent
        cg.replay()
        self.stats["replays"] += 1
        return loss, logits[:batch.y.size(0)]
