"""Graph containers: the subset of PyG ``Data`` / ``Batch`` / ``DataLoader`` behaviour the
reference relies on (SURVEY.md A.3; call sites ``pangnn.py:121,152-153``, ``src/dataset.py:302-310``).
PyG is not a dependency of this implementation.
"""
import random

import torch


_COPY_STREAMS = {}


def _copy_stream(dev):
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _COPY_STREAMS[key]


class Data:
    """``Data(x, edge_index, edge_attr, y)`` attribute bag; extra attributes by assignment."""

    def __init__(self, x=None, edge_index=None, edge_attr=None, y=None, **kw):
        self.x, self.edge_index, self.edge_attr, self.y = x, edge_index, edge_attr, y
        for k, v in kw.items():
            setattr(self, k, v)

    @property
    def num_nodes(self):
        return self.x.size(0)

    def keys(self):
        return [k for k, v in self.__dict__.items() if v is not None and not k.startswith("_")]

    def to(self, device, non_blocking=False):
        out = Data()
        for k, v in self.__dict__.items():
            setattr(out, k, v.to(device, non_blocking=non_blocking) if torch.is_tensor(v) else v)
        return out

    def to_pipelined(self, device, order=("edge_index", "union_edge_index", "neighbour_edge_index",
                                          "edge_attr", "y", "x")):
        """H2D on a dedicated copy stream, tensor by tensor in ``order`` (structure first), each
        followed by an event: ``wait(name)`` makes the CURRENT stream wait for just that tensor, so
        the CSR build of the first edge list overlaps the copy of the next one.  Source tensors
        should be pinned."""
        dev = torch.device(device)
        out = Data()
        copy_stream = _copy_stream(dev)
        main = torch.cuda.current_stream(dev)
        copy_stream.wait_stream(main)              # destination blocks may still be in use upstream
        names = [k for k in order if torch.is_tensor(self.__dict__.get(k))]
        names += [k for k, v in self.__dict__.items() if torch.is_tensor(v) and k not in names]
        events = {}
        for k in names:
            v = self.__dict__[k]
            dst = torch.empty(v.shape, dtype=v.dtype, device=dev)      # allocated on the main stream
            with torch.cuda.stream(copy_stream):
                dst.copy_(v, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            events[k] = ev
            setattr(out, k, dst)
        for k, v in self.__dict__.items():
            if not torch.is_tensor(v):
                setattr(out, k, v)
        out._ready = events
        return out

    def wait(self, *names):
        """Order the current stream after the pipelined copies of ``names`` (all when empty)."""
        ready = self.__dict__.get("_ready") or {}
        for k in (names or list(ready)):
            ev = ready.get(k)
            if ev is not None:
                torch.cuda.current_stream().wait_event(ev)
        return self

    def pin_memory(self):
        out = Data()
        for k, v in self.__dict__.items():
            setattr(out, k, v.pin_memory() if torch.is_tensor(v) and not v.is_cuda else v)
        return out

    def cpu(self):
        return self.to("cpu")

    def to_dict(self):
        return dict(self.__dict__)

    def from_dict(self, d):
        self.__dict__.update(d)
        return self

    def __repr__(self):
        parts = [f"{k}={list(v.shape)}" if torch.is_tensor(v) else f"{k}=..." for k, v in self.__dict__.items()
                 if v is not None]
        return f"Data({', '.join(parts)})"


def collate(graphs):
    """``Batch.from_data_list``: attributes whose NAME contains 'index' are concatenated on the last
    dim and offset by the cumulative node count; other tensors are concatenated on dim 0; lists
    become lists of lists; ``batch`` and ``ptr`` are added."""
    out = Data()
    keys = [k for k in graphs[0].__dict__ if graphs[0].__dict__[k] is not None]
    offsets, off = [], 0
    for g in graphs:
        offsets.append(off)
        off += g.x.size(0)
    for k in keys:
        vals = [getattr(g, k) for g in graphs]
        if torch.is_tensor(vals[0]):
            if "index" in k:
                out.__dict__[k] = torch.cat([v + o for v, o in zip(vals, offsets)], dim=-1)
            else:
                out.__dict__[k] = torch.cat(vals, dim=0)
        else:
            out.__dict__[k] = vals
    out.batch = torch.cat([torch.full((g.x.size(0),), i, dtype=torch.long) for i, g in enumerate(graphs)])
    out.ptr = torch.tensor(offsets + [off], dtype=torch.long)
    out.num_graphs = len(graphs)
    return out


class DataLoader:
    """Minimal ``torch_geometric.loader.DataLoader``: shuffles, batches, collates, optionally pins
    and moves each batch to ``device`` (the role ``accelerate`` plays in the reference)."""

    def __init__(self, dataset, batch_size=1, shuffle=False, pin_memory=False, device=None, seed=None):
        self.dataset, self.batch_size, self.shuffle = list(dataset), max(int(batch_size), 1), shuffle
        self.pin_memory, self.device = pin_memory, device
        self._rng = random.Random(seed)

    def __len__(self):
        return (len(self.dataset) + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        order = list(range(len(self.dataset)))
        if self.shuffle:
            self._rng.shuffle(order)
        for i in range(0, len(order), self.batch_size):
            b = collate([self.dataset[j] for j in order[i:i + self.batch_size]])
            if self.device is not None:
                if self.pin_memory and torch.cuda.is_available():
                    b = b.pin_memory()
                b = b.to(self.device, non_blocking=True)
            yield b


class DeviceLoader:
    """``DataLoader`` with the split resident on the device and the collation done there (a12 as a device op,
    ``pangnn_collate``): same batches in the same order as ``DataLoader(dataset, batch_size, shuffle, seed=seed)``,
    without the per-step host ``torch.cat`` s and H2D copies (~1 ms of Python per batch of 32 sub-graphs, half of
    the reference regime's step).  One H2D of the epoch's permutation per epoch."""

    def __init__(self, dataset, batch_size=1, shuffle=False, device="cuda", seed=None):
        import numpy as np
        from . import ops
        if hasattr(dataset, "arena"):                        # subgraphs.GraphList: already packed on the device
            self.packed, self._ids = dataset.arena.packed, np.asarray(dataset.ids, dtype=np.int32)
        else:
            self.packed = ops.PackedGraphs(dataset, device)
            self._ids = np.arange(self.packed.num_graphs, dtype=np.int32)
        self.batch_size, self.shuffle, self.device = max(int(batch_size), 1), shuffle, torch.device(device)
        self._rng = random.Random(seed)

    def __len__(self):
        return (self._ids.size + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        return self.batches()

    def batches(self, shard=None, pad=True):
        """``__iter__`` with the ``shard`` / ``pad`` options of ``iter_ids``."""
        for packed, ids, ids_dev in self.iter_ids(shard, pad):
            yield packed.collate(ids, ids_dev)

    def iter_ids(self, shard=None, pad=True):
        """The same batches as ``__iter__`` as ``(packed, ids, ids_dev)`` — for a consumer that collates into its own
        buffers (``pangnn_b200.graphs.GraphedBatchStep.step_ids``).

        ``shard=(rank, world)``: this rank's part of the epoch's batch list, which is the same on every rank of a
        group with the same seed: batches ``rank, rank + world, ...``.  With ``pad`` the list is first padded to a
        multiple of ``world`` by repeating whole batches from its start (Accelerate's ``even_batches``), so every
        rank takes the same number of steps."""
        import numpy as np
        order = list(range(self._ids.size))
        if self.shuffle:
            self._rng.shuffle(order)
        order = self._ids[np.asarray(order, dtype=np.int64)] if order else self._ids[:0]
        order_dev = torch.from_numpy(order).to(self.device)
        starts = list(range(0, len(order), self.batch_size))
        if shard is not None:
            rank, world = shard
            if pad and starts:
                starts += [starts[i % len(starts)] for i in range(-len(starts) % world)]
            starts = starts[rank::world]
        for i in starts:
            yield self.packed, order[i:i + self.batch_size], order_dev[i:i + self.batch_size]



_PREP_STREAMS = {}


class PrefetchLoader:
    """Whole-graph batches from pinned HOST memory with one batch of look-ahead: while step ``i`` runs on the
    caller's stream, batch ``i+1`` is copied (copy stream) and its structures are built (``model.prepare``:
    neighbour band, union assembly, CSR builds) on a preparation stream.  Every tensor and structure handed to
    the caller is recorded for the caller's stream (the caching allocator defers their reuse accordingly) and
    the caller's stream waits for the batch's event.  The structures of a batch are evicted when the next one
    is handed out.

        loader = PrefetchLoader(host_batches, model, device)
        for g in loader:
            loss = step(g)            # queue the step ...
            loader.prefetch_next()    # ... then the copy + build of the next batch, so that they run beside it
            loss.item()

    Without the explicit call the next batch is started when it is asked for (no overlap with a step that has
    already been waited for)."""

    def __init__(self, host_batches, model, device, scored_only=True):
        self.host_batches, self.model, self.device = host_batches, model, torch.device(device)
        self.scored_only = scored_only
        self._it, self._pending, self._prev, self._exhausted = None, None, None, True

    def __len__(self):
        return len(self.host_batches)

    def _start(self, hb):
        from . import ops
        main, prep = self._main, self._prep
        with torch.cuda.stream(prep):
            g = hb.to_pipelined(self.device, order=self.model.transfer_order(scored_only=self.scored_only))
            g = self.model.prepare(g)
            ev = torch.cuda.Event()
            ev.record(prep)
        for v in g.__dict__.values():
            if torch.is_tensor(v) and v.is_cuda:
                v.record_stream(main)
        for gs in ops.cached_structs(g):
            gs.built_on(prep, main)
        return g, ev

    def __iter__(self):
        dev = self.device
        self._main = torch.cuda.current_stream(dev)
        key = dev.index if dev.index is not None else torch.cuda.current_device()
        self._prep = _PREP_STREAMS.setdefault(key, torch.cuda.Stream(device=dev))
        self._it, self._pending, self._prev, self._exhausted = iter(self.host_batches), None, None, False
        self.prefetch_next()
        return self

    def prefetch_next(self):
        """Queue the copy and the structure build of the next batch now (call it right after queueing a step)."""
        if self._pending is None and not self._exhausted:
            hb = next(self._it, None)
            if hb is None:
                self._exhausted = True
            else:
                self._pending = self._start(hb)

    def __next__(self):
        from . import ops
        self.prefetch_next()
        if self._prev is not None:
            ops.drop_structs(self._prev)
            self._prev = None
        if self._pending is None:
            raise StopIteration
        g, ev = self._pending
        self._pending = None
        self._main.wait_event(ev)
        self._prev = g
        return g
