"""Genome-partitioned multi-GPU execution of the panGNN model (SURVEY.md §8e — new in this
implementation; the reference's only parallelism is implicit DDP through ``accelerate``).

Partition: node ids are genome-major (``src/dataset.py:72,90,101``), so rank r owns the contiguous id
range ``[lo_r, hi_r)`` — a block of genomes — together with

  * the rows (DESTINATIONS) of every convolution graph that fall in its range, and
  * the scored edges whose SOURCE it owns.

One exchange per layer: the layer input rows of remote sources ("halo") are fetched from their
owners with one grouped NCCL send/recv (``batch_isend_irecv``; with the default trivial-case filter
the simulated sim graph only joins adjacent genomes (SURVEY F11), so the halo is the two boundary
genomes, not the whole node set).  The exchange runs at the narrower of the layer's two widths.
Backward is the transposed plan: gradients of halo rows travel back to their owners and are added in
fixed rank order (deterministic; unique indices per peer, no atomics).  The ~54 k weight gradients
are summed with one flat all-reduce per step.  The loss is the global mean: every rank scales its
partial sum by ``1 / E_total``.

Everything below the exchange is the single-GPU code path (same CSR build, gcn_norm, aggregation
and fused scorer kernels) applied to the local "own + halo" numbering.

Two transports for the exchange:
  * NCCL grouped send/recv (``HaloPlan._exchange``) — always available, also used over gloo in the CPU tests;
  * NVLink peer memory (``P2P``; default on CUDA when torch symmetric memory is available, ``PANGNN_P2P=0``
    turns it off): the extended activation buffers live in symmetric memory, every rank STORES the rows
    its peers need straight into their buffers (``pangnn_rows_gather_copy`` on a peer pointer, or the
    epilogue of the producing GEMM), gradients of halo rows are LOADED from the peers' buffers and added
    in rank order (``pangnn_rows_scatter_add``); ONE device-side barrier per exchange orders producers and
    consumers (the buffers alternate between two sets by step parity, ``_sym``).  No packing, no staging
    copies, no NCCL kernel on the data path.
"""
import os

import torch
import torch.distributed as dist

from . import ops
from .setup import args


# ------------------------------------------------------------------------------------------------
# NVLink peer-memory transport
# ------------------------------------------------------------------------------------------------
class P2P:
    """Symmetric-memory buffers of one process group: ``buffer(key, rows, F)`` returns the local
    [rows, F] fp32 tensor and its handle (``hdl.get_buffer(peer, ...)`` maps a peer's copy,
    ``hdl.barrier()`` is a stream-ordered barrier across the group).  Allocation is collective: every
    rank must request the same keys in the same order with the same ``rows`` (callers pass the maximum
    over ranks)."""

    _instances = {}

    def __init__(self, group=None):
        import torch.distributed._symmetric_memory as symm
        self.symm, self.group = symm, (group if group is not None else dist.group.WORLD)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.bufs = {}

    @classmethod
    def get(cls, group=None):
        """The shared context of ``group`` or None when the transport is unavailable / disabled."""
        if os.environ.get("PANGNN_P2P", "1") == "0" or not dist.is_initialized() or not torch.cuda.is_available():
            return None
        if dist.get_backend(group) != "nccl" or dist.get_world_size(group) < 2:
            return None
        key = id(group) if group is not None else 0
        if key not in cls._instances:
            try:                                               # trial allocation: every rank fails or succeeds alike
                ctx = cls(group)
                dev = torch.device("cuda", torch.cuda.current_device())
                _, hdl = ctx.buffer("probe", 8, 4, dev)
                hdl.barrier()
                ok = torch.ones(1, device=dev)
            except Exception as e:                             # no symmetric memory / no peer access on this box
                setup_log = __import__("logging").getLogger("pangnn")
                setup_log.warning(f"NVLink peer-memory transport unavailable ({type(e).__name__}: {e}); using NCCL send/recv")
                ctx, ok = None, torch.zeros(1, device=torch.device("cuda", torch.cuda.current_device()))
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)      # agree: all ranks or none
            cls._instances[key] = ctx if float(ok.item()) > 0 else None
        return cls._instances[key]

    def buffer(self, key, rows, F, device):
        ent = self.bufs.get((key, F))
        if ent is None or ent[0].size(0) < rows:
            t = self.symm.empty(int(rows), int(F), dtype=torch.float32, device=device)
            ent = (t, self.symm.rendezvous(t, self.group))
            self.bufs[(key, F)] = ent
        return ent

    def peer(self, hdl, p, rows, F):
        return hdl.get_buffer(p, (int(rows), int(F)), torch.float32)


# ------------------------------------------------------------------------------------------------
# data-parallel gradient average
# ------------------------------------------------------------------------------------------------
class GradReducer:
    """``reducer()`` replaces every gradient of ``params`` by its mean over the ranks of ``group``: the all-reduce
    DDP runs behind ``accelerator.backward`` (``pangnn.py:207``) in data-parallel training.  Call it between
    ``loss.backward()`` and ``optimizer.step()``, eagerly or inside a CUDA-graph capture, the same number of times
    on every rank.  A gradient that is None stays None.

    The bucket is laid out from ``params``, which must be the same list on every rank (which parameters receive a
    gradient depends on the flags alone).  Over NVLink peer memory (``P2P``) the reduction is ``ops.grad_push`` +
    ``ops.grad_reduce``: every rank packs its gradients into its own symmetric bucket and sums every peer's in rank
    order, so the result is bitwise the same on every rank.  Otherwise (``PANGNN_P2P=0``, no symmetric memory,
    gloo) it is one flat ``dist.all_reduce`` times ``1 / W``.  In a group of one rank it does nothing."""

    def __init__(self, params, group=None, timeout_s=120.0):
        self.params, self.group, self.timeout_s = [p for p in params if p.requires_grad], group, float(timeout_s)
        self.numels = [p.numel() for p in self.params]
        init = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if init else 1
        self.rank = dist.get_rank(group) if init else 0
        self.scale = float(torch.tensor(1.0 / self.world, dtype=torch.float32))          # fp32(1 / W)
        self.p2p = None
        if self.world > 1 and self.params and self.params[0].is_cuda and len(self.params) <= ops.GRAD_REDUCE_MAX_TENSORS \
                and self.world <= ops.GRAD_REDUCE_MAX_RANKS:
            self.p2p = P2P.get(group)
        if self.p2p is not None:
            dev = self.params[0].device
            self.half = ops.grad_bucket_floats(self.numels)
            self.bucket, hb = self.p2p.buffer("grad_bucket", 2, self.half, dev)
            sig, hs = self.p2p.buffer("grad_signal", 1, ops.GRAD_REDUCE_MAX_RANKS, dev)
            sig.zero_()
            self.signal = sig.view(torch.int32)
            self.ctrl = torch.zeros(4, dtype=torch.int32, device=dev)              # epoch, two tickets, status
            peers = range(self.world)
            self.peer_buckets = [self.p2p.peer(hb, p, 2, self.half).data_ptr() if p != self.rank else
                                 self.bucket.data_ptr() for p in peers]
            self.peer_signals = [self.p2p.peer(hs, p, 1, ops.GRAD_REDUCE_MAX_RANKS).data_ptr() if p != self.rank else
                                 sig.data_ptr() for p in peers]
            hs.barrier()                                        # every rank's zeroed signals before any push

    def __call__(self):
        if self.world == 1:
            return
        grads = [p.grad for p in self.params]
        if self.p2p is not None:
            ops.grad_push(grads, self.numels, self.bucket, self.half, self.peer_signals, self.rank, self.ctrl)
            ops.grad_reduce(grads, self.numels, self.peer_buckets, self.half, self.signal, self.rank, self.ctrl,
                            self.timeout_s)
            return
        flat = torch.cat([(g if g is not None else torch.zeros_like(p)).reshape(-1) for p, g in zip(self.params, grads)])
        dist.all_reduce(flat, group=self.group)
        flat.mul_(self.scale)
        off = 0
        for g, n in zip(grads, self.numels):
            if g is not None:
                g.copy_(flat[off:off + n].view_as(g))
            off += n

    def check(self):
        """Raise if a peer-memory reduction gave up waiting (reads the status word: one host synchronisation, so
        call it where the host waits anyway, e.g. once per epoch)."""
        if self.p2p is not None:
            st = int(self.ctrl[3].item())
            if st:
                raise RuntimeError(f"rank {self.rank}: the gradient average timed out after {self.timeout_s:g} s "
                                   f"waiting for rank {st - 1}")


# ------------------------------------------------------------------------------------------------
# halo plans
# ------------------------------------------------------------------------------------------------
class HaloPlan:
    """Who sends which of its owned rows to whom.  ``halo_ids`` (sorted global ids of the remote rows
    this rank needs) is grouped by owner because owners are contiguous ranges."""

    def __init__(self, n_own, halo_ids, bounds, rank, world, group=None):
        self.n_own, self.rank, self.world, self.group = n_own, rank, world, group
        self.n_halo = int(halo_ids.numel())
        dev = halo_ids.device
        b = torch.as_tensor(bounds, device=dev, dtype=halo_ids.dtype)
        owner = torch.searchsorted(b, halo_ids, right=True) - 1
        need = torch.bincount(owner, minlength=world).to(torch.int64)             # rows I need from o
        self.recv_splits = need.tolist()
        if world > 1:
            table = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
            dist.all_gather(table, need, group=group)
            table = torch.stack(table)                                            # [r, o]
        else:
            table = need.view(1, 1)
        self.send_splits = table[:, rank].tolist()                                # rows r needs from me
        # tell every owner WHICH rows: send my id slices, receive theirs
        want = [torch.empty(n, dtype=halo_ids.dtype, device=dev) for n in self.send_splits]
        self._exchange(list(halo_ids.split(self.recv_splits)), want)
        lo = int(bounds[rank])
        self.send_idx = (torch.cat(want) - lo) if want else torch.zeros(0, dtype=torch.long, device=dev)
        self.send_idx = self.send_idx.long()
        # ---- peer-memory transport: where my rows land in each peer's extended buffer
        tab = table.tolist()                                                      # [r][o] rows r needs from o
        own = [int(bounds[r + 1]) - int(bounds[r]) for r in range(world)]
        self.n_ext_max = max(own[r] + sum(tab[r]) for r in range(world))          # symmetric buffer rows
        # my rows occupy [peer_slot0[p], + send_splits[p]) of peer p's buffer (its halo ids are sorted, owners in rank order)
        self.peer_slot0 = [own[p] + sum(tab[p][:rank]) for p in range(world)]
        self.send_off = [sum(self.send_splits[:p]) for p in range(world)]
        self.send_idx32 = self.send_idx.to(torch.int32)
        self.p2p = P2P.get(group) if halo_ids.is_cuda else None

    def _exchange(self, send_list, recv_list):
        """send_list[p] -> peer p, recv_list[p] <- peer p (grouped, skips empty and self)."""
        opsl = []
        for p in range(self.world):
            if p == self.rank:
                continue
            if recv_list[p].numel():
                opsl.append(dist.P2POp(dist.irecv, recv_list[p], p, group=self.group))
            if send_list[p].numel():
                opsl.append(dist.P2POp(dist.isend, send_list[p].contiguous(), p, group=self.group))
        if opsl:
            for w in dist.batch_isend_irecv(opsl):
                w.wait()

    # -- NVLink peer-memory transport ---------------------------------------------------------------
    def push_maps(self):
        """[(peer, slot_map int32[n_own], lo, hi)] for the fused GEMM-epilogue push: slot_map[row] = destination row
        in that peer's extended buffer, -1 where the peer does not need the row.  None when more than two
        peers need rows of mine (the epilogue carries two maps; such plans use the standalone push)."""
        if not hasattr(self, "_push_maps"):
            peers = [p for p in range(self.world) if p != self.rank and self.send_splits[p] > 0]
            if len(peers) > 2:
                self._push_maps = None
            else:
                maps = []
                for p in peers:
                    o, n = self.send_off[p], self.send_splits[p]
                    m = torch.full((self.n_own,), -1, dtype=torch.int32, device=self.send_idx.device)
                    m[self.send_idx[o:o + n]] = torch.arange(self.peer_slot0[p], self.peer_slot0[p] + n,
                                                             dtype=torch.int32, device=m.device)
                    rows = self.send_idx[o:o + n]
                    maps.append((p, m, int(rows.min().item()), int(rows.max().item()) + 1))
                self._push_maps = maps
        return self._push_maps

    def p2p_push(self, ext, hdl):
        """``ext`` [>= n_own + n_halo, F] is this rank's symmetric buffer with valid owned rows: store the
        rows every peer needs into that peer's buffer (barrier after: every halo row has landed; the peer has
        consumed the previous content of this buffer set — see ``_sym``)."""
        F = ext.size(1)
        for p in range(self.world):                            # (no barrier before: double-buffered sites, see _sym)
            n = self.send_splits[p]
            if p == self.rank or n == 0:
                continue
            peer = self.p2p.peer(hdl, p, self.n_ext_max, F)
            o = self.send_off[p]
            ops.rows_gather_copy(ext, self.send_idx32[o:o + n], peer[self.peer_slot0[p]:self.peer_slot0[p] + n])
        hdl.barrier()

    def p2p_pull_add(self, d_ext, hdl):
        """``d_ext`` [>= n_own + n_halo, F] symmetric: add, into my owned rows, the gradients every peer
        computed for them (its halo part), peer by peer in rank order."""
        F = d_ext.size(1)
        hdl.barrier()
        for p in range(self.world):
            n = self.send_splits[p]
            if p == self.rank or n == 0:
                continue
            peer = self.p2p.peer(hdl, p, self.n_ext_max, F)
            o = self.send_off[p]
            ops.rows_scatter_add(peer[self.peer_slot0[p]:self.peer_slot0[p] + n], self.send_idx32[o:o + n], d_ext)
        # (no barrier after: the peers overwrite this set two steps from now, behind other barriers — see _sym)

    def gather(self, rows_own, out=None):
        """[n_own, F] -> halo rows [n_halo, F] in ``halo_ids`` order (received into ``out`` if given)."""
        F = rows_own.shape[1:]
        send = rows_own.index_select(0, self.send_idx)
        halo = out if out is not None else torch.empty((self.n_halo,) + tuple(F), dtype=rows_own.dtype,
                                                       device=rows_own.device)
        self._exchange(list(send.split(self.send_splits)), list(halo.split(self.recv_splits)))
        return halo

    def scatter_add(self, halo_rows, out_own):
        """Transposed exchange: contributions computed for halo rows go back to their owners and are
        added to ``out_own`` peer by peer in rank order."""
        F = halo_rows.shape[1:]
        recv = torch.empty((int(self.send_idx.numel()),) + tuple(F), dtype=halo_rows.dtype,
                           device=halo_rows.device)
        self._exchange(list(halo_rows.contiguous().split(self.recv_splits)), list(recv.split(self.send_splits)))
        off = 0
        for p in range(self.world):
            n = self.send_splits[p]
            if n:
                out_own.index_add_(0, self.send_idx[off:off + n], recv[off:off + n])
            off += n
        return out_own


# Exchange buffers alternate between two sets by step parity (``next_step()``; a backward uses the set of its own
# forward).  With a single set every exchange needed TWO device barriers — "the peer has consumed the previous
# content" before the stores, "every row has landed" after them; with two sets the first is implied by the other
# barriers of the previous step (a rank that is storing into set s of step t has passed a barrier that every peer
# entered after its last read of set s in step t-2), so each exchange keeps one: 4 per step instead of 8.
_STEP = {"parity": 0}


def next_step():
    _STEP["parity"] ^= 1


def _sym(plan, kind, site, F, device):
    """Symmetric buffer of an exchange site (forward activations / backward gradients) for the current step parity."""
    return plan.p2p.buffer(f"{kind}:{site}:{_STEP['parity']}", plan.n_ext_max, F, device)


class HaloGather(torch.autograd.Function):
    """x_own [n_own, F] -> x_ext [n_own + n_halo, F]; backward = transposed exchange.  ``site`` names
    the exchange (one symmetric buffer pair per site in peer-memory mode)."""

    @staticmethod
    def forward(ctx, x_own, plan, site="g"):
        ctx.plan, ctx.site = plan, site
        if plan.n_halo == 0 and plan.world == 1:
            return x_own
        if plan.p2p is not None and x_own.size(1) % 4 == 0:
            ext, hdl = _sym(plan, "fwd", site, x_own.size(1), x_own.device)
            ext[:plan.n_own].copy_(x_own)
            plan.p2p_push(ext, hdl)
            return ops._alias(ext, (plan.n_own + plan.n_halo, ext.size(1)))
        return torch.cat((x_own, plan.gather(x_own)), dim=0)

    @staticmethod
    def backward(ctx, d_ext):
        plan = ctx.plan
        if plan.n_halo == 0 and plan.world == 1:
            return d_ext, None, None
        if plan.p2p is not None and d_ext.size(1) % 4 == 0:
            buf = _p2p_backward(plan, ctx.site, d_ext)
            return ops._alias(buf, (plan.n_own, buf.size(1))), None, None
        d_own = d_ext[:plan.n_own].clone()
        plan.scatter_add(d_ext[plan.n_own:], d_own)
        return d_own, None, None


def _p2p_backward(plan, site, d_ext):
    """Halo-gradient return over peer memory.  ``d_ext`` normally IS the site's symmetric gradient buffer
    (the aggregation / scorer backward wrote into it); otherwise it is copied there first."""
    buf, hdl = _sym(plan, "bwd", site, d_ext.size(1), d_ext.device)
    n = plan.n_own + plan.n_halo
    if d_ext.data_ptr() != buf.data_ptr():
        buf[:n].copy_(d_ext[:n])
    plan.p2p_pull_add(buf, hdl)
    return ops._alias(buf, (n, buf.size(1)))


class HaloFill(torch.autograd.Function):
    """In-place form of ``HaloGather`` for a producer that already left room: ``x_full`` is
    [>= n_own + n_halo, F] with valid owned rows; the halo rows are received straight into its tail
    (no concatenation copy) — over NCCL, or, when ``x_full`` is the site's symmetric buffer, by the
    peers' stores.  Backward adds the returned halo gradients into the owned rows of the incoming
    gradient in place — that tensor is produced by the aggregation backward for this consumer alone."""

    @staticmethod
    def forward(ctx, x_full, plan, site="f", pushed=False):
        ctx.plan, ctx.site = plan, site
        ctx.mark_dirty(x_full)
        if pushed:                                              # the producing GEMM stored the halo rows itself
            _sym(plan, "fwd", site, x_full.size(1), x_full.device)[1].barrier()
            return x_full
        if plan.p2p is not None and x_full.size(1) % 4 == 0:
            ext, hdl = _sym(plan, "fwd", site, x_full.size(1), x_full.device)
            if x_full.data_ptr() != ext.data_ptr():
                ext[:plan.n_own].copy_(x_full[:plan.n_own])
            plan.p2p_push(ext, hdl)
            if x_full.data_ptr() != ext.data_ptr():
                x_full[plan.n_own:plan.n_own + plan.n_halo].copy_(ext[plan.n_own:plan.n_own + plan.n_halo])
            return x_full
        if plan.n_halo:
            plan.gather(x_full[:plan.n_own], out=x_full[plan.n_own:plan.n_own + plan.n_halo])
        return x_full

    @staticmethod
    def backward(ctx, d_full):
        plan = ctx.plan
        d_full = d_full.contiguous()
        if plan.p2p is not None and d_full.size(1) % 4 == 0 and plan.world > 1:
            return _p2p_backward(plan, ctx.site, d_full), None, None, None
        if plan.n_halo or plan.world > 1:
            plan.scatter_add(d_full[plan.n_own:plan.n_own + plan.n_halo], d_full[:plan.n_own])
        return d_full, None, None, None


# ------------------------------------------------------------------------------------------------
# local graphs
# ------------------------------------------------------------------------------------------------
def balanced_bounds(num_nodes, world, genome_size=None):
    """Contiguous id ranges; whole genomes per rank when ``genome_size`` divides evenly, otherwise a
    plain contiguous split (C4: 20 genomes on 8 GPUs)."""
    if genome_size and (num_nodes // genome_size) % world == 0:
        per = (num_nodes // genome_size) // world * genome_size
        return [r * per for r in range(world)] + [num_nodes]
    return [(num_nodes * r) // world for r in range(world)] + [num_nodes]


def local_numbering(edge_index, lo, hi, anchor="dst"):
    """Edges whose ``anchor`` endpoint is owned -> (mask, sorted halo ids, edge_index in own + halo
    numbering).  Pure index arithmetic (also exercised by the CPU gloo tests).  Written to keep the peak at the
    input plus ~2.5x the output (the partition build of a pan-genome-scale rank is memory-bound): the kept edges are
    gathered once into the result and renumbered in place."""
    a = edge_index[1] if anchor == "dst" else edge_index[0]
    keep = (a >= lo) & (a < hi)
    del a
    out = edge_index[:, keep].contiguous()                                        # [2, E'] — becomes the result
    n_own = hi - lo
    own_row, other_row = (out[1], out[0]) if anchor == "dst" else (out[0], out[1])
    outside = (other_row < lo) | (other_row >= hi)
    halo_ids = torch.unique(other_row[outside])                                    # sorted
    own_row.sub_(lo)                                                              # the anchor endpoint is owned
    if halo_ids.numel():
        pos = torch.searchsorted(halo_ids, other_row[outside])
        other_row.sub_(lo)
        other_row[outside] = pos.add_(n_own)
    else:
        other_row.sub_(lo)
    return keep, halo_ids, out


class LocalGraph:
    """The part of one edge set a rank needs: edges whose ``anchor`` endpoint ('dst' for convolution
    graphs, 'src' for the scored edges) is owned, renumbered to own + halo ids.  ``edge_index`` may
    be the global edge list or any superset of the rank's edges, in GLOBAL ids."""

    def __init__(self, edge_index, bounds, rank, world, anchor="dst", edge_weight=None, group=None):
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        self.n_own = hi - lo
        self.edge_mask, self.halo_ids, self.edge_index = local_numbering(edge_index, lo, hi, anchor)
        self.plan = HaloPlan(self.n_own, self.halo_ids, bounds, rank, world, group)
        self.n_ext = self.n_own + self.plan.n_halo
        self.edge_weight = edge_weight[self.edge_mask].contiguous() if edge_weight is not None else None
        self.edge_order = None
        if self.edge_index.size(1):
            # The local list is kept in canonical (src, dst) order of the LOCAL ids (halo ids do not preserve the
            # global order): every later batch of this partition then gets its by-source CSR by head detection and
            # the other orientation by a 3-pass transpose instead of a 5-pass sort (as whole graphs do at N = 1), the
            # scorer's by-source gradients are a gather-free segment sum and its edges can be processed in chunks.
            # ``edge_order`` = the permutation applied after ``edge_mask`` (per-edge tensors of the scored list —
            # labels, skip weights, global edge ids — follow it).
            order = torch.argsort(self.edge_index[0] * self.n_ext + self.edge_index[1], stable=True)
            self.edge_order = order
            self.edge_index = self.edge_index[:, order].contiguous()
            if self.edge_weight is not None:
                self.edge_weight = self.edge_weight[order].contiguous()
        self._gs = None
        self._norm = {}

    @property
    def gs(self):
        """Both CSR orientations of the local graph (built on first use, on the device)."""
        if self._gs is None:
            self._gs = ops.GraphStruct(self.edge_index, self.n_ext)
        return self._gs

    def rebuilt(self, edge_index, edge_weight):
        """Same partition metadata (halo ids, exchange plan), fresh device tensors: the CSR and
        gcn_norm caches start empty (what a new batch costs)."""
        lg = object.__new__(LocalGraph)
        lg.__dict__.update(self.__dict__)
        lg.edge_index, lg.edge_weight, lg._gs, lg._norm = edge_index, edge_weight, None, {}
        return lg

    def norm(self, weighted=True):
        """gcn_norm on the partition: degrees of owned rows are complete locally; ``dis`` of halo
        sources comes from their owners (one exchange, cached)."""
        key = bool(weighted)
        if key not in self._norm:
            w = self.edge_weight if weighted else None
            dis_loc, _ = ops.gcn_norm(self.gs.dst, w)
            dis_own = dis_loc[:self.n_own].contiguous()
            dis_ext = torch.cat((dis_own, self.plan.gather(dis_own.unsqueeze(1)).squeeze(1)))
            self._norm[key] = (ops.gcn_norm_apply(self.gs.dst, w, dis_ext),
                               ops.gcn_norm_apply(self.gs.src, w, dis_ext))
        return self._norm[key]


class PartitionedGraph:
    """What ``DistModel`` consumes: the local pieces of the whole-graph ``Data`` object.
    All edge lists are in GLOBAL ids and may be supersets of what the rank needs.  ``y`` may be None (a graph without
    labels, for inference only): ``self.y`` and ``class_balance`` are then None."""

    def __init__(self, bounds, rank, world, x_own, conv_ei, conv_w, nb_ei, scored_ei, scored_w, y,
                 group=None):
        self.rank, self.world, self.bounds, self.group = rank, world, bounds, group
        b = (bounds, rank, world)
        self.n_own = bounds[rank + 1] - bounds[rank]
        self.x = x_own
        self.conv = LocalGraph(conv_ei, *b, anchor="dst", edge_weight=conv_w, group=group)
        self.nb = LocalGraph(nb_ei, *b, anchor="dst", group=group) if nb_ei is not None else None
        self.scored = LocalGraph(scored_ei, *b, anchor="src", group=group)
        m = self.scored.edge_mask
        self.y = self.pick(y) if y is not None else None
        self.skip = self.pick(scored_w).float() if args.skip_connections else None
        self.scored_edge_ids = self.pick(torch.arange(m.numel(), device=m.device))
        pos = float(self.y.sum().item()) if self.y is not None else 0.0
        cnt = torch.tensor([float(self.scored_edge_ids.numel()), pos], dtype=torch.float64, device=m.device)
        if world > 1:
            dist.all_reduce(cnt, group=group)
        self.num_edges_total = int(cnt[0].item())
        self.class_balance = float((cnt[0] - cnt[1]) / cnt[1]) if self.y is not None else None   # src/dataset.py:346

    def pick(self, t):
        """Per-edge tensor of the scored list given to the constructor -> the rows of this rank's scored edges, in
        their local order (the order of ``y``, ``skip`` and the logits)."""
        m, o = self.scored.edge_mask, self.scored.edge_order
        return t[m][o].contiguous() if o is not None else t[m].contiguous()

    def scored_endpoints(self):
        """GLOBAL ``(src, dst)`` of this rank's scored edges, in their local order."""
        lg, lo = self.scored, self.bounds[self.rank]
        ext = torch.cat((torch.arange(lo, lo + lg.n_own, device=lg.edge_index.device), lg.halo_ids.long()))
        return ext[lg.edge_index[0]], ext[lg.edge_index[1]]

    def build_edge_split(self, seed, fractions):
        """``--edge_split``: ``self.split``, the ``edge_split.EdgeSplit`` of this rank's scored edges from their global
        endpoints (no communication) with the counts and the train class balance over the group (one all-reduce).
        -> the split."""
        from .edge_split import EdgeSplit
        self.split = EdgeSplit.build(*self.scored_endpoints(), self.y, seed, fractions, self.group)
        return self.split

    # -- host round trip of the rank's local batch (bench.py's end-to-end leg) ----------------------
    _LOCALS = ("conv", "nb", "scored")

    def to_host_pinned(self):
        from types import SimpleNamespace
        h = SimpleNamespace(t={}, nbytes=0)
        def put(name, t):
            if t is not None:
                if name.endswith(".edge_index"):               # own + halo ids fit 32 bits: half the PCIe bytes
                    t = t.to(torch.int32)
                h.t[name] = t.detach().cpu().pin_memory()
                h.nbytes += t.numel() * t.element_size()
        for name in self._LOCALS:
            lg = getattr(self, name)
            if lg is not None:
                put(name + ".edge_index", lg.edge_index)
                put(name + ".edge_weight", lg.edge_weight)
        put("x", self.x); put("y", self.y); put("skip", self.skip)
        return h

    def rebuilt_from(self, host, device):
        """A new batch with the same partition metadata: H2D on the copy stream, edge lists first, and
        the CSR builds start as each edge list lands (same scheme as ``Data.to_pipelined``)."""
        from .data import _copy_stream
        dev = torch.device(device)
        cs, main = _copy_stream(dev), torch.cuda.current_stream(dev)
        cs.wait_stream(main)
        order = [n + ".edge_index" for n in ("scored", "conv", "nb")] + \
                [k for k in host.t if not k.endswith(".edge_index")]
        d, ready = {}, {}
        for k in order:
            if k not in host.t:
                continue
            v = host.t[k]
            d[k] = torch.empty(v.shape, dtype=v.dtype, device=dev)
            with torch.cuda.stream(cs):
                d[k].copy_(v, non_blocking=True)
                ready[k] = torch.cuda.Event()
                ready[k].record(cs)
        pg = object.__new__(PartitionedGraph)
        pg.__dict__.update(self.__dict__)
        for name in ("scored", "conv", "nb"):
            lg = getattr(self, name)
            if lg is None:
                continue
            main.wait_event(ready[name + ".edge_index"])
            ei = d[name + ".edge_index"]
            if ei.dtype != torch.int64:                        # widened on the device (the PyG-surface dtype)
                ei = ei.long()
            new = lg.rebuilt(ei, d.get(name + ".edge_weight"))
            new.gs.src                                         # both CSR orientations, while the next list copies
            if name == "scored":
                new.gs.endpoints32
            setattr(pg, name, new)
        for ev in ready.values():
            main.wait_event(ev)
        pg.x, pg.y, pg.skip = d["x"], d.get("y"), d.get("skip")
        return pg

    def prefetch_from(self, host, device, consumer=None):
        """``rebuilt_from`` on a preparation stream, for one batch of look-ahead: returns ``(batch, event)``;
        the consumer stream waits for ``event`` before its step.  Every tensor / structure of the batch is
        recorded for the consumer stream (caching-allocator hand-over), as ``data.PrefetchLoader`` does for
        whole graphs.  Call it right AFTER queueing the step it should overlap (the step's kernels then start
        at once and the copy + CSR builds run beside them)."""
        from .data import _PREP_STREAMS
        dev = torch.device(device)
        main = consumer if consumer is not None else torch.cuda.current_stream(dev)
        key = dev.index if dev.index is not None else torch.cuda.current_device()
        prep = _PREP_STREAMS.setdefault(key, torch.cuda.Stream(device=dev))
        with torch.cuda.stream(prep):
            pg = self.rebuilt_from(host, dev)
            ev = torch.cuda.Event()
            ev.record(prep)
        for t in (pg.x, pg.y, pg.skip):
            if t is not None:
                t.record_stream(main)
        for name in self._LOCALS:
            lg = getattr(pg, name)
            if lg is not None:
                for t in (lg.edge_index, lg.edge_weight):
                    if t is not None:
                        t.record_stream(main)
                lg.gs.built_on(prep, main)
        return pg, ev

    @classmethod
    def from_global(cls, graph, num_nodes, rank, world, genome_size=None, group=None):
        """Every rank holds the same whole-graph ``Data`` (small graphs, tests)."""
        bounds = balanced_bounds(num_nodes, world, genome_size)
        E = graph.edge_index.size(1)
        x_own = graph.x[bounds[rank]:bounds[rank + 1]]
        if args.union_edge_weights:
            conv_ei, conv_w, nb_ei = graph.union_edge_index, graph.edge_attr, None
        else:
            conv_ei, conv_w = graph.edge_index, graph.edge_attr[:E]
            nb_ei = None if args.base_model else graph.neighbour_edge_index
        return cls(bounds, rank, world, x_own, conv_ei, conv_w, nb_ei, graph.edge_index,
                   graph.edge_attr[:E], graph.y, group)

    @classmethod
    def from_simulation(cls, n, G, frac_pos, frags, shuf, rank, world, device, seed=0, group=None,
                        device_generator=False, keep_hits=False):
        """Partition-local build for ``--simulate_dataset`` graphs: the rank generates the hits of its
        own genomes plus one boundary genome on each side (their candidate sets are complete, and
        every edge INTO an owned node starts there), normalises them on its own device and keeps
        what it needs.  No data-path communication besides the halo plans.

        ``keep_hits`` (host generator only) also keeps what the per-edge output table needs: ``hits``, the
        generated raw hit table ``(q, t, bits)`` as host arrays — every (query, target genome) segment of an owned
        query is complete in it — and ``scored_w``, the Q-scores of the rank's scored edges."""
        from . import preprocessing as pp
        from .simulate import simulate_hits, simulate_hits_device
        if args.include_trivial and world > 1:
            raise NotImplementedError("--include_trivial joins every genome pair: the +-1 genome slab is not enough")
        if keep_hits and device_generator:
            raise NotImplementedError("keep_hits keeps the host generator's hit table")
        # whole genomes per rank when G divides evenly, otherwise a plain contiguous id split (C4: 20 genomes on 8
        # GPUs, SURVEY §8e); either way the rank generates every genome its id range touches, +- 1
        bounds = balanced_bounds(n * G, world, genome_size=n)
        g_lo, g_hi = bounds[rank] // n, -(-bounds[rank + 1] // n)
        N = n * G
        if device_generator:
            # Philox streams on the device (csrc/simulate.cu), one QUERY genome at a time: the candidate sets of a
            # query are complete inside its genome's slab, so generating and normalising slab by slab gives the same
            # table as one pass over all of the rank's genomes, at 1 / (genomes per rank + 2) of its peak memory (hit
            # table + sort workspace + normalisation buffers: ~85 B per hit)
            parts, gen_of, grp_of, grp_host = [], None, None, None
            for g in range(max(g_lo - 1, 0), min(g_hi + 1, G)):
                s = simulate_hits_device(n, G, frac_pos, frags, shuf, seed=seed, genomes=(g, g + 1),
                                         score_means=tuple(args.simulated_score_means), device=device, group_of=grp_host)
                if gen_of is None:                                # [N] maps: built and sent to the device once
                    grp_host = s["group_of"]
                    gen_of = torch.from_numpy(s["genome_of"]).to(device)
                    grp_of = torch.from_numpy(grp_host).to(device)
                parts.append(pp.normalize_sim_scores(s["q"], s["t"], s["bits"], gen_of, grp_of, num_nodes=N, device=device))
                del s
            src, dst, w, y = (torch.cat([p[i] for p in parts]) for i in range(4))
            del parts
        else:
            s = simulate_hits(n, G, frac_pos, frags, shuf, seed=seed, genomes=(g_lo - 1, g_hi + 1),
                              adjacent_only=not args.include_trivial,
                              score_means=tuple(args.simulated_score_means))
            src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"],
                                                     num_nodes=N, device=device)
            hits = (s["q"], s["t"], s["bits"]) if keep_hits else None
            del s
        sim_ei = torch.stack((src.long(), dst.long()))
        lo, hi = bounds[rank], bounds[rank + 1]
        k = args.neighbours
        j = torch.arange(lo, hi, device=device).repeat_interleave(2 * k + 1)
        i = j + torch.arange(-k, k + 1, device=device).repeat(hi - lo)
        ok = (i >= 0) & (i < N)
        band = torch.stack((i[ok], j[ok]))                                        # i -> j, dst owned
        x_own = torch.ones(hi - lo, 1, device=device)
        if args.union_edge_weights:
            conv_ei = torch.cat((sim_ei, band), dim=1)
            conv_w = torch.cat((w, torch.ones(band.size(1), device=device)))
            nb_ei = None
        else:
            conv_ei, conv_w = sim_ei, w
            nb_ei = None if args.base_model else band
        pg = cls(bounds, rank, world, x_own, conv_ei, conv_w, nb_ei, sim_ei, w, y, group)
        if keep_hits:
            pg.hits, pg.scored_w = hits, pg.pick(w)
        return pg


# ------------------------------------------------------------------------------------------------
# model
# ------------------------------------------------------------------------------------------------
def _fwd_buf(plan, site, F, device):
    """(out_full for the producing GEMM, dx_out for the consumer's backward) of an exchange site."""
    if plan.p2p is None:
        return None, None
    return (ops._alias(_sym(plan, "fwd", site, F, device)[0], (plan.n_own + plan.n_halo, F)),
            _sym(plan, "bwd", site, F, device)[0])


def _linear_with_halo(x_own, W, plan, site):
    """h_ext = [x_own W^T ; halo rows]: over peer memory the GEMM's epilogue stores the rows the
    neighbours need straight into their buffers (fused GEMM -> halo all-gather, one barrier after it);
    otherwise the GEMM leaves room and the exchange follows."""
    out_full, _ = _fwd_buf(plan, site, W.size(0), x_own.device)
    maps = plan.push_maps() if (plan.p2p is not None and W.size(0) in (64, 128) and W.size(1) in (64, 128)) else None
    if maps is None:
        return HaloFill.apply(ops.linear(x_own, W, extra_rows=plan.n_halo, out_full=out_full), plan, site)
    _, hdl = _sym(plan, "fwd", site, W.size(0), x_own.device)   # (no barrier before the stores: double-buffered, see _sym)
    push = [(m, plan.p2p.peer(hdl, p, plan.n_ext_max, W.size(0)), lo, hi) for p, m, lo, hi in maps]
    h_full = ops.linear(x_own, W, out_full=out_full, push=push)
    return HaloFill.apply(h_full, plan, site, True)             # barrier: every peer's rows have landed


def _layer(x_own, conv, lg, weighted, act, site):
    """One GCNConv (+ELU) on a partition.  The halo exchange runs at min(in, out) width."""
    W, b = conv.lin.weight, conv.bias
    val_dst, val_src = lg.norm(weighted)
    plan = lg.plan
    if ops.aggregate_first(W):
        _, dx_out = _fwd_buf(plan, site, W.size(1), x_own.device)
        x_ext = HaloGather.apply(x_own, plan, site)
        ax = ops.AggregateFn.apply(x_ext, None, lg.gs.dst, val_dst, lg.gs.src, val_src, lg.n_own, ops.ACT_NONE, dx_out)
        return ops.linear(ax, W, b, act)
    _, dx_out = _fwd_buf(plan, site, W.size(0), x_own.device)
    h_ext = _linear_with_halo(x_own, W, plan, site)
    return ops.AggregateFn.apply(h_ext, b, lg.gs.dst, val_dst, lg.gs.src, val_src, lg.n_own, act, dx_out)


def _embed_conv(m, pg, act, consumer=None):
    """Embedding ``Linear(1, D)`` + ``conv_in`` on a partition as one rank-2 update (``ops.RankOneFn``): the
    vectors ``a = A_hat x``, ``c = A_hat 1`` of the OWNED rows need the scalar features of the halo sources —
    one exchange of [n_halo] floats, cached with the partition's gcn_norm — and the layer itself needs no
    per-step communication at all: its parameter gradients are partial sums over the owned rows, completed by
    the weight-gradient all-reduce like every other.

    With ``consumer`` (the ``LocalGraph`` of the NEXT convolution) the result has that graph's own + halo rows:
    the halo rows of this layer's output are a function of the owners' (a, c) — fetched once, cached — so they
    are recomputed here as ghost rows instead of being exchanged every step, forward or backward.  A ghost
    row's gradient holds only the edges into this rank's nodes; every parameter gradient is linear in it, so
    the partial sums of all ranks add up to the whole-graph gradient in the all-reduce."""
    lg = pg.conv
    val_dst, _ = lg.norm(True)
    key = ("rank1", pg.x.data_ptr(), pg.x._version)
    ac = lg._norm.get(key)
    if ac is None:
        x_own = pg.x.reshape(-1, 1).float().contiguous()
        x_ext = torch.cat((x_own, lg.plan.gather(x_own)), dim=0)
        ac = lg._norm[key] = ops.rank1_vectors(lg.gs.dst, val_dst, x_ext, lg.n_own) + (pg.x,)
    a, c = ac[0], ac[1]
    if consumer is not None:
        key2 = ("rank1ext",) + key[1:]
        ext = consumer._norm.get(key2)
        if ext is None:
            both = torch.stack((a, c), dim=1).contiguous()                 # [n_own, 2]: one exchange for both
            both = torch.cat((both, consumer.plan.gather(both)), dim=0)
            ext = consumer._norm[key2] = (both[:, 0].contiguous(), both[:, 1].contiguous(), pg.x)
        a, c = ext[0], ext[1]
    return ops.RankOneFn.apply(a, c, m.embedding.weight, m.embedding.bias, m.conv_in.lin.weight,
                               m.conv_in.bias, act)


class DistModel:
    """Runs an ``AlternateGCN``'s parameters on a ``PartitionedGraph`` (mlp decoder, node_dim 64)."""

    def __init__(self, model, group=None):
        self.model, self.group = model, group

    def embed(self, pg):
        """``AlternateGCN.embed`` on the partition: the same embedding and ``conv_schedule``.  Each layer exchanges its
        halo (``_layer``; the exchange site is named by the layer's position), except a fused embedding and the layer
        that consumes its ghost rows (``_embed_conv``)."""
        m, ELU = self.model, ops.ACT_ELU
        schedule, done = m.conv_schedule(), 0
        if m._categorical:
            # A.6: one embedding row per gene, indexed by GLOBAL position (rows of other ranks get
            # zero gradient here; the flat all-reduce sums the disjoint row blocks)
            lo = pg.bounds[pg.rank]
            h = m.embedding(torch.arange(lo, lo + pg.n_own, device=pg.x.device))
        elif m.fuses_embedding(pg.x):
            mod, on, weighted = schedule[1]
            consumer = getattr(pg, on) if on is not None else None
            h, done = _embed_conv(m, pg, ELU, consumer), 1
            if consumer is not None:
                val_dst, val_src = consumer.norm(weighted)
                h = ops.gcn_layer_csr(h, mod.lin.weight, mod.bias, consumer.gs.dst, val_dst, consumer.gs.src, val_src,
                                      consumer.n_own, ELU)
                done = 2
        else:
            h = (torch.addcmul(m.embedding.bias, pg.x, m.embedding.weight.t())
                 if pg.x.dim() == 2 and pg.x.size(1) == 1 else m.embedding(pg.x))
        for i, (mod, on, weighted) in enumerate(schedule[done:], done):
            h = m.activation_fct(mod(h)) if on is None else _layer(h, mod, getattr(pg, on), weighted, ELU, f"conv{i}")
        return h

    def _scorer_inputs(self, pg, h):
        """-> (endpoint rows pq_ext [n_ext, 2D], the scorer's weights (w1c, b1, w2, b2, w3, b3), dpq_out)."""
        mlp, D = self.model.mlp, ops.SCORER_D
        if args.decoder != "mlp" or h.size(1) != D:
            raise NotImplementedError("the partitioned path scores edges with the fused mlp decoder at --node_dim 64")
        wcat, w1c = ops.split_w1(mlp[0].weight, pg.skip is not None)
        plan = pg.scored.plan
        _, dpq_out = _fwd_buf(plan, "pq", 2 * D, h.device)
        pq_ext = _linear_with_halo(h, wcat, plan, "pq")
        return pq_ext, (w1c, mlp[0].bias, mlp[2].weight, mlp[2].bias, mlp[4].weight, mlp[4].bias), dpq_out

    @torch.no_grad()
    def forward(self, pg):
        """Inference: logits of the locally scored edges (``pg.scored_edge_ids`` in the global list)."""
        next_step()
        pq_ext, weights, _ = self._scorer_inputs(pg, self.embed(pg))
        return ops.edge_score_pq_fwd(pq_ext, *weights, pg.scored.gs, pg.skip)

    __call__ = forward

    def forward_loss(self, pg, pos_weight, unit_grad=True, y=None, num_labelled=None):
        """-> (this rank's share of the global mean loss, logits of the locally scored edges).  ``unit_grad``: the
        loss is back-propagated as is (``loss.backward()``, checked on the device) — pass False to scale it first.
        ``y``: this rank's selected labels in place of ``pg.y`` (``-1`` = held out, ``--edge_split``), the mean then
        taken over ``num_labelled``, the GLOBAL number of edges with a label."""
        next_step()                                            # exchange buffers of the other parity (see _sym)
        pq_ext, weights, dpq_out = self._scorer_inputs(pg, self.embed(pg))
        n = pg.num_edges_total if num_labelled is None else int(num_labelled)
        return ops.EdgeScoreBCEPQFn.apply(pq_ext, *weights, pg.scored.gs, pg.skip, pg.y if y is None else y,
                                          float(pos_weight), 1.0 / max(n, 1), dpq_out, unit_grad)

    @torch.no_grad()
    def predict(self, pg, threshold):
        """This rank's ``(logits, prob, pred)`` of the edges ``pg.scored_edge_ids``: sigmoid and threshold fused into
        the scorer kernel, as ``AlternateGCN.predict``.  Reads no labels."""
        next_step()
        pq_ext, weights, _ = self._scorer_inputs(pg, self.embed(pg))
        return ops.edge_score_predict(pq_ext, *weights, pg.scored.gs, pg.skip, threshold)

    @torch.no_grad()
    def evaluate(self, pg, threshold, pos_weight=None, labels=None):
        """Test statistics of the whole partitioned graph, identical on every rank (``train.evaluate`` of the global
        graph, ``src/predict.py:29-55``): global confusion matrix (one all-reduce of four counts), precision /
        recall / F1 with ``eps=0``, the global mean BCE loss when ``pos_weight`` is given, and the exact global
        ranking metrics of the probabilities (``metrics.ranking_metrics`` over the group).  Also returns this
        rank's ``logits`` / ``prob`` / ``pred`` (edges ``pg.scored_edge_ids``).  A graph without labels (``pg.y``
        None) gets those and ``predicted_positive``, the global number of edges predicted positive, alone.
        ``labels``: this rank's selected labels (``-1`` outside the selection, ``--edge_split``): the counts, the loss
        and the ranking metrics are then over the selected edges of every rank alone, and ``sel`` is this rank's
        mask of them; ``logits`` / ``prob`` / ``pred`` stay those of every edge."""
        from .metrics import ranking_metrics
        from .train import prf
        logits, prob, pred = self.predict(pg, threshold)
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        y = pg.y
        if y is None:
            k = pred.sum(dtype=torch.int64)
            if world > 1:
                dist.all_reduce(k, group=self.group)
            return dict(logits=logits, prob=prob, pred=pred, predicted_positive=int(k))
        out = dict(logits=logits, prob=prob, pred=pred)
        if labels is not None:
            out["sel"] = labels >= 0
            y, logits, prob, pred = labels[out["sel"]], logits[out["sel"]], prob[out["sel"]], pred[out["sel"]]
        p, yl = pred.long(), y.long()
        tp = (p * yl).sum()
        fp = (p * (1 - yl)).sum()
        fn = ((1 - p) * yl).sum()
        cnt = torch.stack((torch.full_like(tp, y.numel()) - tp - fp - fn, fp, fn, tp))
        loss_sum = None
        if pos_weight is not None:
            loss_sum = torch.nn.functional.binary_cross_entropy_with_logits(
                logits, y, pos_weight=torch.as_tensor(float(pos_weight), device=logits.device), reduction="sum")
        if world > 1:
            dist.all_reduce(cnt, group=self.group)
            if loss_sum is not None:
                loss_sum = loss_sum.double()
                dist.all_reduce(loss_sum, group=self.group)
        tn, fp, fn, tp = (int(v) for v in cnt.tolist())
        pr, rc, f1 = prf(tn, fp, fn, tp, eps=0.0)
        rec = dict(tn=tn, fp=fp, fn=fn, tp=tp, precision=pr, recall=rc, f1=f1, **out)
        if loss_sum is not None:
            n = pg.num_edges_total if labels is None else tn + fp + fn + tp           # the global selected count
            rec["loss"] = float(loss_sum) / max(n, 1)
        rk = ranking_metrics(prob, y, self.group)
        rec.update(auroc=rk["auroc"], average_precision=rk["average_precision"],
                   youden_threshold=rk["youden_threshold"], num_runs=rk["num_runs"])
        return rec

    def _categorical_table(self):
        return self.model.embedding.weight if getattr(self.model, "_categorical", False) else None

    def allreduce_grads(self):
        """Sum the weight gradients over ranks: one flat bucket (~54 k floats).  The bucket is laid out from the
        rank-independent list of trainable parameters (a parameter without a gradient on this rank contributes
        zeros), so every rank reduces the same number of elements whatever its local graph looked like."""
        # --categorical_node: the [N, D] embedding table is sharded by ownership in effect — a rank only ever
        # reads and updates the rows of its own nodes (halo rows arrive through the layer exchange, their
        # gradients return to the owner) — so its 1 GB gradient is not all-reduced every step; call
        # ``sync_embedding()`` before saving or evaluating the model outside the partition.
        skip = self._categorical_table()
        params = [p for p in self.model.parameters() if p.requires_grad and p is not skip]
        if not params or not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return
        flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
        dist.all_reduce(flat, group=self.group)
        off = 0
        for p in params:
            g = flat[off:off + p.numel()].view_as(p)
            if p.grad is None:
                p.grad = g.clone()
            else:
                p.grad.copy_(g)
            off += p.numel()

    @torch.no_grad()
    def sync_embedding(self, bounds):
        """--categorical_node: make every replica's embedding table complete again — rank r broadcasts the row
        block ``[bounds[r], bounds[r+1])`` it owns and trains.  Without it ``state_dict()`` of any one rank holds
        the INITIAL rows of every other rank's genes and a single-GPU run from that checkpoint is wrong."""
        table = self._categorical_table()
        if table is None or not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return
        world = dist.get_world_size(self.group)
        for r in range(world):
            blk = table.data[int(bounds[r]):int(bounds[r + 1])]
            dist.broadcast(blk, src=dist.get_global_rank(self.group, r) if self.group is not None else r,
                           group=self.group)

    def state_dict(self, bounds):
        """The model's ``state_dict()`` with the sharded embedding table gathered (``torch.save`` this one)."""
        self.sync_embedding(bounds)
        return self.model.state_dict()
