"""Re-hosted driver for the reference's ``pangnn.py`` loop contract (``pangnn.py:36-373``): same flags
(``pangnn_b200.setup``), same dataset object, same optimiser / scheduler / loss, same ``model.pkl``
(``torch.save(model.state_dict())``), with the hot path on the CUDA kernels.  Reporting extras of the
reference (TensorBoard, plots, ``stats.csv``, rich progress bars) are out of scope (DESIGN.md §7); the
numbers they would show are logged and returned.

    python pangnn.py --simulate_dataset 10000 2 0.5 10 3 --train -e 5 -o runs      # train, save, test
    python pangnn.py --simulate_dataset 10000 2 0.5 10 3 -m runs/model.pkl         # inference only
"""
import os
import time

import numpy as np
import torch

from . import postprocessing as post
from . import setup
from .metrics import precision_recall_curve, ranking_metrics, roc_curve
from .data import DeviceLoader
from .dataset import UnionGraphDataset
from .gnn import AlternateGCN
from .setup import log


def confusion(pred, labels):
    """(tn, fp, fn, tp) of int predictions vs {0,1} labels — what torchmetrics' BinaryConfusionMatrix
    accumulates in the reference (``pangnn.py:27,222,266``)."""
    pred, labels = pred.long(), labels.long()
    tp = int((pred * labels).sum())
    fp = int((pred * (1 - labels)).sum())
    fn = int(((1 - pred) * labels).sum())
    return labels.numel() - tp - fp - fn, fp, fn, tp


def prf(tn, fp, fn, tp, eps=1e-10):
    """precision / recall / F1 with the reference's epsilons (``pangnn.py:291-294,315-318``).  With ``eps=0``
    (the test-time formulas, ``src/predict.py:114-121``) an empty denominator yields 0 instead of raising:
    no predicted positive -> precision 0, no positive label -> recall 0, precision + recall == 0 -> F1 0."""
    dp, dr = tp + fp + eps, tp + fn + eps
    p, r = (tp / dp if dp else 0.0), (tp / dr if dr else 0.0)
    return p, r, (2 * p * r / (p + r + eps) if (p + r + eps) else 0.0)


def youden_threshold(prob, labels):
    """``--dynamic_binary_threshold`` (``pangnn.py:229-233``, which crashes in the reference because ``labels`` and
    ``output`` are deleted first; SURVEY A.6: computed before the dels): the ROC threshold that maximises
    ``tpr - fpr`` — sklearn's ``roc_curve`` semantics (distinct scores in decreasing order, first maximum) as
    one device sort + two running sums."""
    prob, labels = prob.reshape(-1), labels.reshape(-1)
    if prob.numel() == 0:
        return None
    order = torch.argsort(prob, descending=True, stable=True)
    p, y = prob[order], labels[order].double()
    last = torch.ones_like(p, dtype=torch.bool)
    last[:-1] = p[1:] != p[:-1]                                 # last entry of every run of equal scores
    tp, fp = torch.cumsum(y, 0)[last], torch.cumsum(1.0 - y, 0)[last]
    P, Nn = float(y.sum()), float(y.numel() - y.sum())
    if P == 0 or Nn == 0:
        return None
    j = tp / P - fp / Nn
    best = int(torch.argmax(j))
    return float(p[last][best]) if float(j[best]) > 0 else None


def evaluate(model, graphs, threshold, pos_weight=None, group=None):
    """Whole-batch inference as ``src/predict.py:29-55``: logits, sigmoid, threshold, confusion; plus the ROC AUC, AP
    and Youden threshold of the probabilities (``src/plot.py:103-107,131``; exact, ``metrics.ranking_metrics`` over
    ``group``: pass a group of one rank for a replica's own graphs while a default process group exists)."""
    model.eval()
    out = []
    for g in graphs:
        logits, prob, pred = model.predict(g, threshold)
        tn, fp, fn, tp = confusion(pred, g.y)
        p, r, f1 = prf(tn, fp, fn, tp, eps=0.0)
        rec = dict(tn=tn, fp=fp, fn=fn, tp=tp, precision=p, recall=r, f1=f1, logits=logits, prob=prob, pred=pred)
        rk = ranking_metrics(prob, g.y, group)
        rec.update(auroc=rk["auroc"], average_precision=rk["average_precision"],
                   youden_threshold=rk["youden_threshold"])
        if pos_weight is not None:
            rec["loss"] = float(torch.nn.functional.binary_cross_entropy_with_logits(
                logits, g.y, pos_weight=torch.as_tensor(float(pos_weight), device=logits.device)))
        out.append(rec)
    return out


def _fmt(v):
    return "n/a" if v is None else f"{v:.4f}"


def log_ranking(stats):
    for s in stats:
        log.info(f"test: auroc {_fmt(s['auroc'])} average precision {_fmt(s['average_precision'])} "
                 f"youden threshold {_fmt(s['youden_threshold'])}")


def _whole_graph(dataset, graph):
    return getattr(graph, "node_id", None) is None or graph.node_id.numel() == dataset.num_genes


def _logit_baseline(dataset, graph, stat):
    """Max-logit-candidate baseline labels of the scored edges (``src/predict.py:84-88``), kept in the stat."""
    from . import preprocessing as pp
    if "logit_baseline" not in stat:
        genome_d = torch.as_tensor(dataset.genome_of, device=graph.edge_index.device)
        ei = graph.edge_index
        stat["logit_baseline"] = pp.baseline_labels(ei[0].int(), ei[1].int(), stat["logits"], genome_d)
    return stat["logit_baseline"]


def add_baselines(dataset, graph, stat):
    """Precision / recall / F1 of the max-candidate baselines next to the model's (``src/predict.py:77-89``):
    ``stat["baselines"] = {name: (p, r, f1)}`` for the whole test graph (a sub-graph batch has no baseline)."""
    if not _whole_graph(dataset, graph):
        return None
    cand = {"base_labels": dataset.base_labels, "base_labels_raw": dataset.base_labels_raw,
            "logit_baseline": _logit_baseline(dataset, graph, stat)}
    out = {}
    for name, lab in cand.items():
        if lab is None or len(lab) == 0:
            continue
        pred = torch.as_tensor(lab, device=graph.y.device)
        out[name] = prf(*confusion(pred, graph.y), eps=0.0)
    stat["baselines"] = out
    log.info("baselines (precision / recall / f1): " +
             "; ".join(f"{k} {p:.4f} / {r:.4f} / {f:.4f}" for k, (p, r, f) in out.items()))
    return out


def _epoch_ranking(probs, labels):
    if not probs:
        return dict(auroc=None, average_precision=None)
    return ranking_metrics(torch.cat(probs), torch.cat(labels))


def write_groups(dataset, graph, stat, out_dir):
    """Ortholog groups of the whole test graph = connected components of the edges predicted positive
    (``src/postprocessing.py:5-36``, device components) -> ``<out_dir>/holiest_of_all_tables.csv``."""
    labels, groups = post.ortholog_groups(graph.edge_index, stat["pred"], graph.x.size(0))
    stat["group_labels"], stat["groups"] = labels, groups
    node_id = getattr(graph, "node_id", None)
    if node_id is not None:                                   # a sub-graph: local ids -> positions in the gene list
        glob = node_id.cpu().tolist()
        groups = [[glob[g] for g in grp] for grp in groups]
    path = post.write_groups_file(groups, dataset.gene_str_ids_lst, os.path.join(out_dir, "holiest_of_all_tables.csv"))
    log.info(f"Wrote {len(groups)} ortholog groups to '{path}'")
    return path


def write_curves(graph, stat, out_dir, group=None):
    """``roc_curve.csv`` (threshold,fpr,tpr) and ``precision_recall_curve.csv`` (threshold,precision,recall; the final
    (1, 0) point has no threshold) of the test probabilities, thinned as sklearn's ``drop_intermediate=True``: the
    data of the reference's ROC and PR figures (``src/plot.py:103-107,131``).  Floats are written round-trip exact."""
    roc = roc_curve(stat["prob"], graph.y, group)
    if roc is None:
        return None
    return write_curve_files(roc, precision_recall_curve(stat["prob"], graph.y, group, drop_intermediate=True), out_dir)


def write_curve_files(roc, pr, out_dir):
    """The two files of ``write_curves`` from the arrays of ``metrics.roc_curve`` / ``metrics.precision_recall_curve``
    (``drop_intermediate=True``)."""
    os.makedirs(out_dir, exist_ok=True)
    paths = os.path.join(out_dir, "roc_curve.csv"), os.path.join(out_dir, "precision_recall_curve.csv")
    fpr, tpr, th = roc
    np.savetxt(paths[0], torch.stack((th, fpr, tpr), 1).cpu().numpy(), fmt="%.17g", delimiter=",",
               header="threshold,fpr,tpr", comments="")
    precision, recall, th = pr
    with open(paths[1], "w") as f:
        f.write("threshold,precision,recall\n")
        np.savetxt(f, torch.stack((th.double(), precision[:-1], recall[:-1]), 1).cpu().numpy(), fmt="%.17g",
                   delimiter=",")
        f.write(f",{float(precision[-1]):.17g},{float(recall[-1]):.17g}\n")
    log.info(f"Wrote '{paths[0]}' ({fpr.numel()} points) and '{paths[1]}' ({precision.numel()} points)")
    return paths


def write_edge_table(dataset, graph, stat, out_dir):
    """``q_score_vs_logit.csv`` for the whole test graph (``src/predict.py:84-88``: the max-logit-candidate
    baseline — a segmented arg-max over the logits — and the table itself, ``src/plot.py:473-504``)."""
    if not _whole_graph(dataset, graph):
        return None                       # a sub-graph batch: the reference has no gene mapping for those either
    ei = graph.edge_index
    logit_base = _logit_baseline(dataset, graph, stat)
    path = post.write_q_score_vs_logit(ei, graph.edge_attr, stat["logits"], graph.y, dataset.gene_str_ids_lst,
                                       dataset.base_labels or None, dataset.base_labels_raw or None, logit_base,
                                       os.path.join(out_dir, "q_score_vs_logit.csv"))
    log.info(f"Wrote '{path}' ({ei.size(1)} scored edges)")
    return path


def run(args, device=None):
    """The reference's main flow.  Returns a dict with the model, per-epoch history and test statistics.

    With a default process group initialised (``main`` under ``torchrun``) every rank runs the genome-partitioned
    driver, ``pangnn_b200.dist_train.run_partitioned``; in a group of one rank the reference's sub-graph training
    (``--train`` without ``--whole_graph_training``) has nothing to partition and runs the loop below.  With
    ``--train --data_parallel`` in a group, every rank runs ``dist_train.run_data_parallel`` instead."""
    from . import dist_train
    if dist_train.data_parallel(args):
        return dist_train.run_data_parallel(args, device)
    if dist_train.partitioned(args):
        return dist_train.run_partitioned(args, device)
    device = torch.device(device if device is not None else "cuda")
    dataset, model = build_dataset_and_model(args, device)
    optimizer = torch.optim.Adam(model.parameters(), lr=0.001)                        # pangnn.py:88
    scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", patience=10, factor=0.6)
    pos_weight = float(dataset.class_balance) if dataset.class_balance else 1.0       # pangnn.py:98
    threshold = args.binary_threshold
    history = []
    test = [g.to(device) for g in dataset.test]

    if not args.train or os.path.exists(args.model_args):                             # pangnn.py:125-144
        if os.path.exists(args.model_args):
            log.info(f"Found model file '{args.model_args}' with trained parameters, restoring model state for inference..")
            model.load_state_dict(torch.load(args.model_args, map_location=device))
        stats = evaluate(model, test, threshold, pos_weight)
        for s in stats:
            log.info(f"test: f1 {s['f1']:.4f} precision {s['precision']:.4f} recall {s['recall']:.4f} loss {s.get('loss', float('nan')):.4f}")
        log_ranking(stats)
        if stats:
            add_baselines(dataset, test[0], stats[0])
            write_groups(dataset, test[0], stats[0], args.output)
            write_curves(test[0], stats[0], args.output)                              # src/plot.py:103-107,131
            write_edge_table(dataset, test[0], stats[0], args.output)                 # src/predict.py:84-88
        return dict(model=model, dataset=dataset, history=history, test=stats)

    # the splits live packed on the device; batches are collated there (a12: pangnn_collate)
    def loader(graphs, seed):
        return DeviceLoader(graphs, batch_size=args.batch_size, shuffle=True, device=device, seed=seed) if graphs else []
    train_loader, val_loader = loader(dataset.train, args.seed), loader(dataset.val, args.seed + 1)
    if args.whole_graph_training:
        # one batch = the whole graph (what the genome-partitioned multi-GPU path and bench.py train on; the
        # reference's per-group sub-graph regime cannot scale past ~1e5 genes, SURVEY F7/F8)
        whole = test[0] if (args.simulate_dataset and test) else dataset.generate_graphs().to(device)
        train_loader, val_loader = [whole], [whole]
        pos_weight = float(dataset.class_balance)                                     # src/dataset.py:346
    stepper = None
    if getattr(args, "cuda_graphs", False) and isinstance(train_loader, DeviceLoader):
        # the loop body below as ONE CUDA graph per batch-size bucket; the learning rate lives in device memory so
        # that ReduceLROnPlateau's in-place updates reach the captured graphs
        from .graphs import GraphedBatchStep
        optimizer = torch.optim.Adam(model.parameters(), lr=torch.tensor(0.001, device=device), capturable=True)
        scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", patience=10, factor=0.6)
        stepper = GraphedBatchStep(model, optimizer, pos_weight)
    for epoch in range(args.epochs):                                                  # pangnn.py:167-238
        model.train()
        train_loss, cm = 0.0, [0, 0, 0, 0]
        ep_prob, ep_y = [], []                                 # the epoch's (prob, label) pairs, on the device
        batches = train_loader.iter_ids() if stepper is not None else train_loader
        for batch in batches:
            if stepper is not None:
                loss, logits = stepper.step_ids(*batch)
                labels = stepper.last_y
            else:
                optimizer.zero_grad()
                loss, logits = model.forward_loss(batch, pos_weight)                  # criterion(model(batch), labels), fused
                loss.backward()
                optimizer.step()
                labels = batch.y
            train_loss += loss.item()
            prob = torch.sigmoid(logits)
            ep_prob.append(prob.detach())
            ep_y.append(labels.clone() if stepper is not None else labels)   # the stepper's labels are static buffers
            pred = (prob >= threshold).int()
            cm = [a + b for a, b in zip(cm, confusion(pred, labels))]
            if args.dynamic_binary_threshold:                                         # pangnn.py:229-233
                th = youden_threshold(prob, labels)
                threshold = th if th is not None else threshold
        val_loss, cmv = 0.0, [0, 0, 0, 0]
        val_prob, val_y = [], []
        model.eval()
        with torch.no_grad():                                                         # pangnn.py:241-275
            for batch in val_loader:
                logits, prob, pred = model.predict(batch, threshold)
                val_prob.append(prob)
                val_y.append(batch.y)
                val_loss += float(torch.nn.functional.binary_cross_entropy_with_logits(
                    logits, batch.y, pos_weight=torch.as_tensor(pos_weight, device=logits.device)))
                cmv = [a + b for a, b in zip(cmv, confusion(pred, batch.y))]
        p, r, f1 = prf(*cm)
        pv, rv, f1v = prf(*cmv)
        mean_val = val_loss / max(len(val_loader), 1)
        scheduler.step(mean_val)                                                      # pangnn.py:296
        # epoch-level ranking metrics (torchmetrics' compute() over the whole epoch, pangnn.py:279-326)
        rk_tr, rk_val = _epoch_ranking(ep_prob, ep_y), _epoch_ranking(val_prob, val_y)
        history.append(dict(epoch=epoch, train_loss=train_loss / max(len(train_loader), 1), val_loss=mean_val,
                            f1_train=f1, f1_val=f1v, precision_val=pv, recall_val=rv,
                            auroc_train=rk_tr["auroc"], ap_train=rk_tr["average_precision"],
                            auroc_val=rk_val["auroc"], ap_val=rk_val["average_precision"]))
        log.info(f"epoch {epoch}: train loss {history[-1]['train_loss']:.4f} f1 {f1:.4f} | val loss {mean_val:.4f} f1 {f1v:.4f}")
        log.info(f"epoch {epoch}: train auroc {_fmt(rk_tr['auroc'])} ap {_fmt(rk_tr['average_precision'])} | "
                 f"val auroc {_fmt(rk_val['auroc'])} ap {_fmt(rk_val['average_precision'])}")

    stats, path = save_test_and_write(args, model, dataset, test, threshold, pos_weight)
    return dict(model=model, dataset=dataset, history=history, test=stats, model_path=path)


def build_dataset_and_model(args, device):
    """The dataset (simulated or read) and the freshly initialised model of ``run``, from ``args.seed``."""
    torch.manual_seed(args.seed)
    t0 = time.time()
    if args.simulate_dataset:
        log.info("Simulating dataset.")
        dataset = UnionGraphDataset(calculate_baseline=True, split=(0.7, 0.15, 0.01),
                                    categorical_nodes=args.categorical_node, device=device)
    else:
        dataset = UnionGraphDataset(args.annotation, args.similarity, args.ribap_groups, split=(0.7, 0.15, 0.01),
                                    categorical_nodes=args.categorical_node, calculate_baseline=True, device=device)
    log.info(f"Dataset: {dataset.num_genes} genes, class balance {dataset.class_balance}, built in {time.time() - t0:.1f} s")
    model = AlternateGCN(device, dataset, dataset.categorical_nodes, dims=[args.node_dim, args.hidden_dim]).to(device)
    return dataset, model


def save_test_and_write(args, model, dataset, test, threshold, pos_weight, write=True, group=None):
    """The end of a training run: save ``model.pkl``, test, and write the test outputs.  ``write=False`` (every rank
    of a data-parallel run but the first) tests without saving or writing; ``group`` as in ``evaluate``.
    -> (test stats, model path)."""
    path = os.path.join(args.output, os.path.basename(args.model_args))
    if write:
        os.makedirs(args.output, exist_ok=True)
        torch.save(model.state_dict(), path)                                          # pangnn.py:339-341
        log.info(f"Saved model parameters to '{path}'")
    stats = evaluate(model, test, threshold, pos_weight, group)                       # pangnn.py:344-346
    for s in stats:
        log.info(f"test: f1 {s['f1']:.4f} precision {s['precision']:.4f} recall {s['recall']:.4f}")
    log_ranking(stats)
    if stats:
        add_baselines(dataset, test[0], stats[0])
        if write:
            write_groups(dataset, test[0], stats[0], args.output)
            write_curves(test[0], stats[0], args.output, group)                       # src/plot.py:103-107,131
            if args.simulate_dataset:                                                 # src/predict.py:84: not args.train or simulate
                write_edge_table(dataset, test[0], stats[0], args.output)
    return stats, path


def main(argv=None):
    """``pangnn.py``.  Under ``torchrun --nproc-per-node N`` (``WORLD_SIZE`` > 1) each process joins an NCCL group
    from the environment on the GPU ``LOCAL_RANK`` and runs the genome-partitioned driver (the data-parallel one with
    ``--train --data_parallel``); the group is destroyed on exit, also on an error."""
    args = setup.parse(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return run(args)
    import torch.distributed as dist
    from .dist_train import check_partition_flags
    check_partition_flags(args, world)                        # every rank refuses alike, before any device work
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    dist.init_process_group("nccl", init_method="env://", device_id=device)
    try:
        return run(args, device)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
