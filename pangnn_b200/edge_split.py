"""Held-out validation and test edges of whole-graph training (``--edge_split VAL TEST``).

A scored edge with global endpoints ``(s, d)`` is assigned by its unordered pair ``a = min(s, d)``, ``b = max(s, d)``:
``x`` = the first 32-bit word of Philox4x32-10 keyed by ``(--seed, purpose 5)`` at counter ``(0, a, b, 0)``
(``csrc/edge_split.cu``, ``pangnn_edge_split``); validation if ``x < T_val``, test if ``x < T_val + T_test``, else train,
with ``T = floor(fraction * 2^32)``.  So both directions of a pair share a split (simulated pairs carry one score in
both directions: no label leaks between them), and the split depends on ``(seed, a, b)`` alone: a rank of a genome
partition splits its own edges without communication, any world size gives the same split, and a saved ``model.pkl``
can be scored again on its own held-out edges.

Held-out edges stay in message passing; only their labels are hidden.  The one representation of the selected labels
is ``EdgeSplit.labels(y, which)``: ``y`` with ``-1.0`` outside ``which``.  The training scorer takes it as is (an edge
with ``y < 0`` has no loss term and no gradient, ``include/pangnn_b200.h``); evaluation keeps the edges with
``labels >= 0`` (``select``) before the confusion counts and ``metrics.ranking_metrics``.
"""
import math

import torch
import torch.distributed as dist

from . import _abi
from .ops import _p, _stream, LAUNCHES

TRAIN, VAL, TEST = 0, 1, 2          # PANGNN_SPLIT_TRAIN / _VAL / _TEST
PURPOSE = 5                         # the Philox purpose of the split; 1-4 are the device simulator's


def check_flags(ns):
    """Raise ``ValueError`` when ``--edge_split`` is combined with flags it cannot serve.  Depends on the flags alone,
    so every rank of a multi-GPU run refuses alike, before any device work."""
    fr = getattr(ns, "edge_split", None)
    if fr is None:
        return
    bad = []
    val, test = (float(v) for v in fr)
    if not (0.0 < val and 0.0 < test and val + test < 1.0):
        bad.append(f"the fractions must satisfy 0 < VAL, 0 < TEST and VAL + TEST < 1 (got {val} {test})")
    if ns.train and not ns.whole_graph_training:
        bad.append("training needs --whole_graph_training (the sub-graph regime already splits by ortholog group)")
    if getattr(ns, "data_parallel", False):
        bad.append("--data_parallel trains on sub-graph batches, which are split by ortholog group")
    if not (bool(ns.simulate_dataset) or bool(ns.ribap_groups)):
        bad.append("it needs labels: name the RIBAP groups table with -r")
    if bad:
        raise ValueError("--edge_split: " + "; ".join(bad))


def thresholds(val, test):
    """``(T_val, T_test) = (floor(VAL * 2^32), floor(TEST * 2^32))`` as Python ints (scaling by a power of two is exact
    in binary floating point, so the floors are exact)."""
    return math.floor(float(val) * (1 << 32)), math.floor(float(test) * (1 << 32))


def split_codes(src, dst, seed, val, test):
    """int8 [E] split codes of the edges ``(src[e], dst[e])`` (global ids) on the device (``pangnn_edge_split``)."""
    lib = _abi.load()
    src = src.to(torch.int32).contiguous()
    dst = dst.to(torch.int32).contiguous()
    t_val, t_test = thresholds(val, test)
    codes = torch.empty(src.numel(), dtype=torch.int8, device=src.device)
    _abi.check(lib.pangnn_edge_split(_p(src), _p(dst), src.numel(), int(seed) & 0xFFFFFFFFFFFFFFFF, t_val, t_test,
                                     _p(codes), _stream()), "edge_split")
    LAUNCHES["count"] += 1
    return codes


def select(labels, *tensors):
    """Keep the edges with a selected label (``labels >= 0``): -> ``(labels[sel], *(t[sel] for t in tensors))``."""
    sel = labels >= 0
    return (labels[sel],) + tuple(t[sel] for t in tensors)


class EdgeSplit:
    """The split codes ``int8 [E]`` of a rank's scored edges (the whole graph's on one GPU) and the host counts per
    split, global over ``group`` when a process group with more than one rank is initialised: ``counts`` (train,
    val, test), ``train_positives`` and ``class_balance`` (neg / pos over the train edges, the ``pos_weight`` of the
    loss).  One all-reduce at construction."""

    def __init__(self, codes, y, group=None):
        self.codes = codes
        c = codes.long()
        red = torch.stack([(c == k).sum() for k in (TRAIN, VAL, TEST)] +
                          [((c == TRAIN) & (y > 0.5)).sum()]).double()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(red, group=group)
        n_train, n_val, n_test, pos = (int(v) for v in red.tolist())
        self.counts, self.train_positives = (n_train, n_val, n_test), pos
        if pos == 0:
            raise ValueError(f"--edge_split: no positive edge among the {n_train} train edges; the class balance "
                             f"(pos_weight) of the loss is undefined")
        self.class_balance = (n_train - pos) / pos

    @classmethod
    def build(cls, src, dst, y, seed, fractions, group=None):
        """The split of the edges ``(src, dst)`` (global ids, device) with labels ``y`` for ``--seed`` and
        ``--edge_split VAL TEST``."""
        return cls(split_codes(src, dst, seed, *fractions), y, group)

    def count(self, which):
        return self.counts[which]

    def labels(self, y, which):
        """``y`` with ``-1.0`` outside split ``which``."""
        return torch.where(self.codes == which, y, torch.full_like(y, -1.0))

    def describe(self):
        return ("edge split (train / val / test scored edges): " +
                " / ".join(str(n) for n in self.counts) + f"; train class balance {self.class_balance}")
