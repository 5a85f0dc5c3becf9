"""Exact ranking metrics on the device: ROC AUC, average precision (AP) and the Youden threshold.

The reference reports them through torchmetrics every epoch (``pangnn.py:27-30,220-222,262-268``) and through sklearn
at test time (``src/plot.py:103-107,131``).  ``ranking_metrics(scores, labels, group=None)`` computes them with the
CUDA kernels of ``csrc/metrics.cu``, on one GPU or over the ranks of a process group.

Contract.  ``scores`` is fp32 [E]; ``labels`` is fp32, integer or bool with values in {0, 1}.  P and N are the
numbers of positive and negative labels.  Runs are the distinct scores in decreasing order; run k holds pos_k
positives and neg_k negatives; TP_k and FP_k are cumulative over runs 1..k, TP_0 = FP_0 = 0.

* AUROC = sum_k neg_k (TP_{k-1} + TP_k) / (2 P N): sklearn ``roc_auc_score``, torchmetrics ``BinaryAUROC``
  (trapezoid over distinct thresholds; a tie gives half credit).
* AP = (1/P) sum_k pos_k TP_k / (TP_k + FP_k): sklearn ``average_precision_score``, torchmetrics
  ``BinaryAveragePrecision``.
* Youden threshold: the score of the first run that maximises TP_k/P - FP_k/N (fp64, that expression); None when the
  maximum is <= 0.  Equal to ``train.youden_threshold``.
* -0.0 and +0.0 are one score; +-inf are ordinary scores.  A NaN score or a label outside {0, 1} raises
  ``PangnnError``.  E = 0, P = 0 or N = 0 gives AUROC None; P = 0 gives AP None.  E >= 2^32 on one device raises.
* The numerators are exact integers (128-bit; AP terms in fixed point with 127 - bitlen(P) fraction bits), divided
  once here with Python integers: the result does not depend on the input order or on the number of ranks.

With a process group of world size > 1 every rank passes its own scores and labels and every rank gets the same dict
(the exact global metrics).  The runs of all ranks are merged by key range: a 65 536-bin histogram of the run keys'
top 16 bits (one all-reduce) cuts the key space into contiguous ranges with balanced run counts, the runs travel
to their range's owner (one all-to-all, 24 B per local run), equal keys are merged there, each rank reduces its
range with the class counts ranked ahead of it as offsets, and the per-rank results are combined in fixed order.  A
bin holds at most 2^16 distinct keys, so a rank receives at most its share plus one bin from every rank
(total_runs / world + world * 65 536 runs).

``roc_curve`` and ``precision_recall_curve`` return sklearn's curves (``src/plot.py:103-107,131``) as device tensors,
bit for bit: the kept runs' (score, TP_k, FP_k) come from ``pangnn_metric_curve`` and every rate is one fp64
division of exact counts.  Over a process group they use the same key-range merge; a rank's last keep decision reads
the first run of the next rank that holds runs, and the pieces are gathered in rank order.
"""
import struct
from fractions import Fraction

import torch
import torch.distributed as dist

from . import ops
from ._abi import PangnnError

_INFO, _OUT = slice(0, 6), slice(8, 16)
# sizes of the last multi-rank exchange on this rank (tools/bench_metrics.py reports them)
LAST_EXCHANGE = {}


def key_to_score(key):
    """Inverse of the kernels' order key (``score_key`` in csrc/metrics.cu)."""
    asc = ~int(key) & 0xFFFFFFFF
    u = asc & 0x7FFFFFFF if asc & 0x80000000 else ~asc & 0xFFFFFFFF
    return struct.unpack("<f", struct.pack("<I", u))[0]


def _u128(lo, hi):
    return (int(lo) & 0xFFFFFFFFFFFFFFFF) | ((int(hi) & 0xFFFFFFFFFFFFFFFF) << 64)


def _check_flags(flags, name="ranking_metrics"):
    if flags & ops.METRIC_NAN:
        raise PangnnError(f"{name}: a score is NaN")
    if flags & ops.METRIC_BAD_LABEL:
        raise PangnnError(f"{name}: a label is not 0 or 1")


def _finish(auc_num, ap_num, best_j, best_key, num_runs, P, N):
    j = struct.unpack("<d", struct.pack("<q", int(best_j)))[0]
    return dict(
        auroc=float(Fraction(auc_num, 2 * P * N)) if P and N else None,
        average_precision=float(Fraction(ap_num, P << (127 - P.bit_length()))) if P else None,
        youden_threshold=key_to_score(best_key) if P and N and j > 0 else None,
        num_pos=P, num_neg=N, num_runs=num_runs)


def ranking_metrics(scores, labels, group=None):
    """-> dict(auroc, average_precision, youden_threshold, num_pos, num_neg, num_runs) (Python floats / ints or None)
    of fp32 ``scores`` against {0, 1} ``labels``; over all ranks of ``group`` when its world size is > 1."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        return _ranking_metrics_dist(scores, labels, group)
    scores, labels = scores.reshape(-1), labels.reshape(-1)
    buf = torch.zeros(16, dtype=torch.int64, device=scores.device)
    info = buf[_INFO]
    runs = ops.metric_runs(scores, labels, info=info)
    ops.metric_reduce(runs, info, out=buf[_OUT])               # info = (runs, P, N, TP_0 = 0, FP_0 = 0, flags)
    h = buf.tolist()                                           # the one host read-back
    _check_flags(h[5])
    o = h[8:16]
    return _finish(_u128(o[0], o[1]), _u128(o[2], o[3]), o[4], o[5] & 0xFFFFFFFFFFFFFFFF, h[0], h[1], h[2])


def _splitters(ghist, world):
    """Bin boundaries [b_0 = 0, ..., b_world = 65536]: rank d owns the keys whose top 16 bits lie in [b_d, b_d+1),
    cut where the cumulative run count of the global histogram first reaches d / world of the total."""
    cum = torch.cumsum(ghist, 0)
    total = int(cum[-1])
    cuts = [0]
    for d in range(1, world):
        cuts.append(max(cuts[-1], int(torch.searchsorted(cum, -(-d * total // world), right=False)) + 1))
    cuts.append(ops.METRIC_HIST_BINS)
    return [min(c, ops.METRIC_HIST_BINS) for c in cuts]


def _all_gather(t, group, world):
    flat = torch.empty(world * t.numel(), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(flat, t, group=group)
    return flat.view(world, t.numel())


def _merge_runs(scores, labels, group, name):
    """Local runs of every rank merged by key range: -> (merged runs of this rank's range (the first ``params[0]``
    rows; none when the tensor is empty), device int64 params (runs, P, N, TP_0, FP_0) with (TP_0, FP_0) the classes
    ranked ahead of the range, device int64 (P, N)).  Every rank raises alike on a NaN score or a bad label."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    scores, labels = scores.reshape(-1), labels.reshape(-1)
    dev = scores.device
    # 1. local runs + histogram of their keys
    info = torch.zeros(6, dtype=torch.int64, device=dev)
    hist = torch.zeros(ops.METRIC_HIST_BINS, dtype=torch.int64, device=dev)
    runs = ops.metric_runs(scores, labels, info=info, hist=hist)
    # 2. splitters from the global histogram; flags and local run counts of every rank
    ghist = hist.clone()
    dist.all_reduce(ghist, group=group)
    infos = _all_gather(info, group, world)
    infos_h, ghist_h, lhist_h = infos.cpu(), ghist.cpu(), hist.cpu()
    flags = 0
    for f in infos_h[:, 5].tolist():
        flags |= f
    _check_flags(flags, name)                                  # every rank raises alike
    cuts = _splitters(ghist_h, world)
    lcum = torch.cat((torch.zeros(1, dtype=torch.int64), torch.cumsum(lhist_h, 0)))
    send = [int(lcum[cuts[d + 1]] - lcum[cuts[d]]) for d in range(world)]
    # 3. exchange: sizes first, then the runs (contiguous key ranges of the sorted local runs)
    send_t = torch.tensor(send, dtype=torch.int64, device=dev)
    recv_t = torch.empty_like(send_t)
    dist.all_to_all_single(recv_t, send_t, group=group)
    recv = recv_t.tolist()
    got = torch.empty(sum(recv), 3, dtype=torch.int64, device=dev)
    dist.all_to_all_single(got, runs[:sum(send)], recv, send, group=group)
    LAST_EXCHANGE.update(local_runs=sum(send), received_runs=sum(recv), bytes_sent=sum(send) * got.element_size() * 3)
    minfo = torch.zeros(6, dtype=torch.int64, device=dev)
    merged = ops.metric_runs(runs=got, info=minfo)
    # 4. offsets: the classes ranked ahead of this rank's key range are those of the lower ranks
    counts = _all_gather(minfo, group, world)[:, 1:3]
    before = counts[:rank].sum(0)
    tot = counts.sum(0)
    params = torch.stack((minfo[0], tot[0], tot[1], before[0], before[1]))
    return merged, params, tot


def _ranking_metrics_dist(scores, labels, group):
    world = dist.get_world_size(group)
    merged, params, tot = _merge_runs(scores, labels, group, "ranking_metrics")
    # 5. reduce the range, gather the per-rank results, combine in rank order
    out = ops.metric_reduce(merged, params)
    outs = _all_gather(out, group, world).tolist()
    P, N = int(tot[0]), int(tot[1])
    auc = ap = runs_total = 0
    best = None
    for o in outs:
        auc += _u128(o[0], o[1])
        ap += _u128(o[2], o[3])
        runs_total += o[6]
        j = struct.unpack("<d", struct.pack("<q", o[4]))[0]
        key = o[5] & 0xFFFFFFFFFFFFFFFF
        if best is None or j > best[0] or (j == best[0] and key < best[1]):
            best = (j, key, o[4])
    return _finish(auc, ap, best[2], best[1], runs_total, P, N)


# ---- curves ------------------------------------------------------------------------------------------------------
def _curve_points(scores, labels, group, mode, name):
    """The kept runs of the whole curve, in decreasing score order: -> (thresholds fp32, TP int64, FP int64) on the
    device, P, N (ints); None without any score."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        return _curve_points_dist(scores, labels, group, mode, name)
    scores, labels = scores.reshape(-1), labels.reshape(-1)
    dev = scores.device
    buf = torch.zeros(9, dtype=torch.int64, device=dev)
    info, count = buf[0:6], buf[6:9]
    runs = ops.metric_runs(scores, labels, info=info)
    R = runs.size(0)
    bound = torch.tensor([0, 0, ops.CURVE_FIRST], dtype=torch.int64, device=dev)
    thr, tp, fp, _ = ops.metric_curve(runs, info, bound, mode, out=(
        torch.empty(R, dtype=torch.float32, device=dev), torch.empty(R, dtype=torch.int64, device=dev),
        torch.empty(R, dtype=torch.int64, device=dev), count))
    h = buf.tolist()                                           # the one host read-back
    _check_flags(h[5], name)
    if h[0] == 0:
        return None
    K = h[6]
    return thr[:K], tp[:K], fp[:K], h[1], h[2]


def _curve_points_dist(scores, labels, group, mode, name):
    """Every rank computes the points of its key range, stitched to its neighbours: the keep rule of its last run
    reads the first run of the next non-empty rank (``bound``), and only the first non-empty rank starts the curve.
    The pieces are concatenated in rank order (rank 0 holds the highest scores)."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    merged, params, tot = _merge_runs(scores, labels, group, name)
    dev = merged.device
    head = torch.zeros(3, dtype=torch.int64, device=dev)      # runs, (pos, neg) of the first run
    head[0] = params[0]
    if merged.size(0):
        head[1:3] = merged[0, 1:3]
    heads = _all_gather(head, group, world).tolist()
    nxt = next((h for h in heads[rank + 1:] if h[0]), None)
    flags = (0 if any(h[0] for h in heads[:rank]) else ops.CURVE_FIRST) | (ops.CURVE_FOLLOWED if nxt else 0)
    bound = torch.tensor([nxt[1], nxt[2], flags] if nxt else [0, 0, flags], dtype=torch.int64, device=dev)
    thr, tp, fp, count = ops.metric_curve(merged, params, bound, mode)
    h = torch.cat((_all_gather(count[:1], group, world).view(-1), tot)).tolist()
    sizes, (P, N) = h[:world], h[world:]
    if P + N == 0:
        return None
    kmax, k = max(sizes), sizes[rank]
    pack = torch.zeros(3, kmax, dtype=torch.int64, device=dev)   # row 0 holds the fp32 thresholds, two per word
    pack[0].view(torch.float32)[:k] = thr[:k]
    pack[1, :k] = tp[:k]
    pack[2, :k] = fp[:k]
    g = _all_gather(pack.view(-1), group, world).view(world, 3, kmax)
    return (torch.cat([g[r, 0].view(torch.float32)[:sizes[r]] for r in range(world)]),
            torch.cat([g[r, 1, :sizes[r]] for r in range(world)]),
            torch.cat([g[r, 2, :sizes[r]] for r in range(world)]), P, N)


def roc_curve(scores, labels, group=None, drop_intermediate=True):
    """sklearn ``roc_curve(labels, scores, drop_intermediate=...)`` on the device -> (fpr, tpr, thresholds) fp64 tensors
    of length K' + 1, or None without any score.  ``thresholds[0]`` is +inf and the point (0, 0) is prepended;
    fpr = FP / N (all NaN when N = 0), tpr = TP / P (all NaN when P = 0), each one fp64 division of exact counts, so
    the arrays equal sklearn's bit for bit.  With ``drop_intermediate`` a run is kept if it is the first or the last
    one or its (pos, neg) differ from the next run's.  Over all ranks of ``group`` when its world size is > 1: every
    rank gets the same arrays."""
    c = _curve_points(scores, labels, group, ops.CURVE_ROC if drop_intermediate else ops.CURVE_ALL, "roc_curve")
    if c is None:
        return None
    thr, tp, fp, P, N = c
    dev = tp.device
    zero = torch.zeros(1, dtype=torch.float64, device=dev)
    den = torch.tensor([N, P], dtype=torch.float64, device=dev)   # device divisors: a true division, element-wise
    fpr = torch.cat((zero, fp.double())) / den[0]
    tpr = torch.cat((zero, tp.double())) / den[1]
    return fpr, tpr, torch.cat((torch.full((1,), float("inf"), dtype=torch.float64, device=dev), thr.double()))


def precision_recall_curve(scores, labels, group=None, drop_intermediate=False):
    """sklearn ``precision_recall_curve(labels, scores, drop_intermediate=...)`` on the device -> (precision, recall,
    thresholds): fp64 [K' + 1], fp64 [K' + 1], fp32 [K'] in ascending threshold order, ending in (1, 0); or None without
    any score.  precision = TP / (TP + FP) (0 where TP + FP = 0), recall = TP / P (all 1.0 when P = 0), bit for bit
    sklearn's.  With ``drop_intermediate`` a run is kept if it is the first or the last one, or it or the next run
    holds a positive.  Over all ranks of ``group`` when its world size is > 1: every rank gets the same arrays."""
    c = _curve_points(scores, labels, group, ops.CURVE_PR if drop_intermediate else ops.CURVE_ALL,
                      "precision_recall_curve")
    if c is None:
        return None
    thr, tp, fp, P, _ = c
    dev = tp.device
    tpd, fpd = tp.double(), fp.double()
    ps = tpd + fpd
    precision = torch.where(ps != 0, tpd / ps, 0.0)
    recall = torch.ones_like(tpd) if P == 0 else tpd / torch.tensor(P, dtype=torch.float64, device=dev)
    one = torch.ones(1, dtype=torch.float64, device=dev)
    return torch.cat((precision.flip(0), one)), torch.cat((recall.flip(0), one - 1)), thr.flip(0)
