"""``pangnn.py`` on several GPUs: the reference's main flow (``train.run``) with the graph partitioned by genome
(``dist.PartitionedGraph``, ``dist.DistModel``), one process per GPU under ``torchrun``.

    torchrun --nproc-per-node 8 pangnn.py --simulate_dataset 100000 80 0.0004 10 3 --train --whole_graph_training -e 5

Every rank builds its partition (simulated data: its own genomes +- 1, never the whole graph; input files: the
whole dataset, then its slice), trains the same ``AlternateGCN`` parameters on the whole graph and takes every
decision (scheduler, dynamic threshold) from global values, so all ranks stay identical.  Rank 0 logs and writes
``model.pkl``, the curves and the groups file with the names and formats of the one-GPU CLI; the per-edge table is
appended rank after rank in global ``(src, dst)`` order, so no rank ever holds all of it.
"""
import contextlib
import logging
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from . import dist as pdist
from . import edge_split as es
from . import ops
from . import postprocessing as post
from . import preprocessing as pp
from .dataset import UnionGraphDataset
from .gnn import AlternateGCN
from .metrics import precision_recall_curve, ranking_metrics, roc_curve
from .setup import check_label_flags, log
from .train import _fmt, log_test, prf, write_curve_files


def check_partition_flags(args, world):
    """Raise ``ValueError`` when the flags ask for something the partitioned driver at ``world`` ranks cannot do.
    Depends on the flags and ``world`` alone, so every rank refuses alike, before any device work."""
    check_label_flags(args)
    es.check_flags(args)
    bad = []
    if getattr(args, "data_parallel", False):
        if args.whole_graph_training:
            bad.append("--data_parallel replicates the model over sub-graph batches and --whole_graph_training "
                       "partitions the graph: choose one")
        if not args.train:
            bad.append("--data_parallel needs --train (inference runs on the genome partition)")
        if bad:
            raise ValueError(f"pangnn.py on {world} GPU(s): " + "; ".join(bad))
        if _trains_replicated(args):
            return                          # the replicas run the one-GPU model code: every flag of the one-GPU loop
    if world > 1 and args.train and not args.whole_graph_training:
        bad.append("--train needs --whole_graph_training (partition the graph by genome and train on the whole graph) "
                   "or --data_parallel (replicate the model and shard the reference's -b sub-graph batches)")
    if world > 1 and args.include_trivial and args.simulate_dataset:
        bad.append("--include_trivial with --simulate_dataset joins every genome pair, but a rank generates only "
                   "its own genomes and one on each side")
    if args.decoder != "mlp" or args.node_dim != ops.SCORER_D:
        bad.append(f"the partitioned path scores edges with the fused mlp decoder at --node_dim {ops.SCORER_D} "
                   f"(got --decoder {args.decoder} --node_dim {args.node_dim})")
    if world > 1 and getattr(args, "cuda_graphs", False):
        bad.append("--cuda_graphs replays the one-GPU sub-graph step")
    if bad:
        raise ValueError(f"pangnn.py on {world} GPU(s): " + "; ".join(bad))


def partitioned(args):
    """Whether ``train.run`` takes the partitioned driver: a default process group is initialised, except for the
    sub-graph training regime in a group of one rank (nothing to partition; it stays on the one-GPU loop)."""
    if not (dist.is_available() and dist.is_initialized()):
        return False
    return dist.get_world_size() > 1 or not args.train or args.whole_graph_training


def _trains_replicated(args):
    """``--train --data_parallel`` trains replicas unless ``-m`` names an existing model file, which the reference
    restores for inference instead (``pangnn.py:125-144``): that inference runs on the genome partition, under its
    flag checks."""
    return (bool(getattr(args, "data_parallel", False)) and args.train and not args.whole_graph_training
            and not os.path.exists(args.model_args))


def data_parallel(args):
    """Whether ``train.run`` takes the data-parallel driver: a default process group is initialised and the flags
    ask for replicated training (``_trains_replicated``)."""
    return _trains_replicated(args) and dist.is_available() and dist.is_initialized()


@contextlib.contextmanager
def _info_on_rank0(rank):
    level = log.level
    if rank:
        log.setLevel(logging.WARNING)
    try:
        yield
    finally:
        log.setLevel(level)


def _counts(pred, y):
    """Device (tn, fp, fn, tp) int64 [4] of {0,1} predictions vs labels (``train.confusion`` without the host read)."""
    p, yl = pred.long(), y.long()
    tp = (p * yl).sum()
    fp = (p * (1 - yl)).sum()
    fn = ((1 - p) * yl).sum()
    return torch.stack((torch.full_like(tp, y.numel()) - tp - fp - fn, fp, fn, tp))


def _partition(args, device, rank, world):
    """-> (pg, dataset or None, number of genes, per-edge tables of the rank's scored edges): global ids, global
    endpoints, Q-scores, the two input-side baselines (None: computed from the rank's hits) and the genome map."""
    if args.simulate_dataset:
        log.info("Simulating dataset.")
        n, G, frac, frags, shuf = args.simulate_dataset
        n, G = int(n), int(G)
        pg = pdist.PartitionedGraph.from_simulation(n, G, float(frac), frags, shuf, rank, world, device,
                                                    seed=args.seed, keep_hits=True)
        N, dataset = n * G, None
        # ranks own contiguous source ranges, so a rank's scored edges are one block of the whole graph's
        # (src, dst)-sorted list, at the offset of the lower ranks' edges
        sizes = torch.zeros(world, dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(sizes, torch.tensor([pg.y.numel()], dtype=torch.int64, device=device))
        pos = torch.cumsum(pg.scored.edge_mask, 0) - 1
        gid = pos[pg.scored_edge_ids] + int(sizes[:rank].sum())
        t = dict(w=pg.scored_w, q_base=None, raw_base=None, names=None,
                 genome_of=np.repeat(np.arange(G, dtype=np.int32), n))
    else:
        dataset = UnionGraphDataset(args.annotation, args.similarity, args.ribap_groups, split=(0.7, 0.15, 0.01),
                                    categorical_nodes=args.categorical_node, calculate_baseline=True, device=device)
        graph = dataset.generate_graphs().to(device)
        N = dataset.num_genes
        pg = pdist.PartitionedGraph.from_global(graph, N, rank, world)
        gid = pg.scored_edge_ids
        lab = lambda v: pg.pick(torch.as_tensor(v, dtype=torch.int64, device=device))
        t = dict(w=pg.pick(graph.edge_attr[:graph.edge_index.size(1)]), q_base=lab(dataset.base_labels),
                 raw_base=lab(dataset.base_labels_raw), names=dataset.gene_str_ids_lst, genome_of=dataset.genome_of)
    src, dst = pg.scored_endpoints()
    t.update(gid=gid, src=src, dst=dst)
    return pg, dataset, N, t


def run_partitioned(args, device=None):
    """``train.run`` on the ranks of the default process group.  Returns the same dict (plus ``graph``, the rank's
    ``PartitionedGraph``, and ``timings``); ``test[0]`` holds this rank's ``logits`` / ``prob`` / ``pred`` and their
    global edge ids ``edge_ids`` (positions in the whole graph's ``(src, dst)``-sorted edge list)."""
    rank, world = dist.get_rank(), dist.get_world_size()
    check_partition_flags(args, world)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    with _info_on_rank0(rank):
        return _run(args, device, rank, world)


def _run(args, device, rank, world):
    t0 = time.time()
    pg, dataset, N, tables = _partition(args, device, rank, world)
    pos_weight = pg.class_balance                                                    # src/dataset.py:346, global
    log.info(f"Dataset: {N} genes, class balance {pos_weight}, built in {time.time() - t0:.1f} s")
    fit, val_labels, test_labels = {}, None, None
    if args.edge_split is not None:
        # --edge_split: the split of the rank's own scored edges; counts and the train class balance are global
        split = pg.build_edge_split(args.seed, args.edge_split)
        log.info(split.describe())
        pos_weight = split.class_balance
        fit = dict(y=split.labels(pg.y, es.TRAIN), num_labelled=split.count(es.TRAIN))
        val_labels, test_labels = split.labels(pg.y, es.VAL), split.labels(pg.y, es.TEST)
    torch.manual_seed(args.seed)                                                     # the one-GPU CLI's parameters
    model = AlternateGCN(device, N if args.categorical_node else dataset, args.categorical_node,
                         dims=[args.node_dim, args.hidden_dim]).to(device)
    if world > 1:
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    dm = pdist.DistModel(model)
    optimizer = torch.optim.Adam(model.parameters(), lr=0.001)                        # pangnn.py:88
    scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", patience=10, factor=0.6)
    threshold = args.binary_threshold
    history, timings = [], dict(train_s=[], val_s=[])

    if not args.train or os.path.exists(args.model_args):                             # pangnn.py:125-144
        if os.path.exists(args.model_args):
            log.info(f"Found model file '{args.model_args}' with trained parameters, restoring model state for inference..")
            model.load_state_dict(torch.load(args.model_args, map_location=device))
        stat = _test(dm, pg, threshold, pos_weight, tables, test_labels)
        log_test([stat], loss=True)
        timings["outputs_s"] = _outputs(args, pg, stat, tables, N, rank, world, edge_table=True)
        return dict(model=model, dataset=dataset, history=history, test=[stat], graph=pg, timings=timings)

    for epoch in range(args.epochs):                                                  # pangnn.py:167-238
        t_ep = time.perf_counter()
        optimizer.zero_grad()
        loss, logits = dm.forward_loss(pg, pos_weight, **fit)
        loss.backward()
        dm.allreduce_grads()
        optimizer.step()
        prob = torch.sigmoid(logits.detach())
        y = pg.y
        if fit:                                               # the train edges alone
            y, prob = es.select(fit["y"], prob)
        # the loss is this rank's share of the global mean: the sum over ranks is the one-GPU value
        red = torch.cat((loss.detach().double().view(1), _counts(prob >= threshold, y).double()))
        if world > 1:
            dist.all_reduce(red)
        red = red.tolist()
        train_loss, cm = red[0], [int(v) for v in red[1:]]
        rk_tr = ranking_metrics(prob, y)                      # over the default group: global, the same on every rank
        if args.dynamic_binary_threshold:                     # pangnn.py:229-233; == train.youden_threshold
            threshold = rk_tr["youden_threshold"] if rk_tr["youden_threshold"] is not None else threshold
        t_val = time.perf_counter()
        # validation: the same whole graph (its validation edges with --edge_split), global
        val = dm.evaluate(pg, threshold, pos_weight, val_labels)
        t_end = time.perf_counter()
        timings["train_s"].append(t_val - t_ep)
        timings["val_s"].append(t_end - t_val)
        p, r, f1 = prf(*cm)
        pv, rv, f1v = prf(val["tn"], val["fp"], val["fn"], val["tp"])
        mean_val = val["loss"]
        scheduler.step(mean_val)                                                      # pangnn.py:296
        history.append(dict(epoch=epoch, train_loss=train_loss, val_loss=mean_val,
                            f1_train=f1, f1_val=f1v, precision_val=pv, recall_val=rv,
                            auroc_train=rk_tr["auroc"], ap_train=rk_tr["average_precision"],
                            auroc_val=val["auroc"], ap_val=val["average_precision"]))
        if val_labels is not None:                            # --edge_split: the validation edges' (tn, fp, fn, tp)
            history[-1]["val_confusion"] = (val["tn"], val["fp"], val["fn"], val["tp"])
        log.info(f"epoch {epoch}: train loss {train_loss:.4f} f1 {f1:.4f} | val loss {mean_val:.4f} f1 {f1v:.4f}")
        log.info(f"epoch {epoch}: train auroc {_fmt(rk_tr['auroc'])} ap {_fmt(rk_tr['average_precision'])} | "
                 f"val auroc {_fmt(val['auroc'])} ap {_fmt(val['average_precision'])}")
        log.debug(f"epoch {epoch}: train step {t_val - t_ep:.3f} s, validation {t_end - t_val:.3f} s")

    path = os.path.join(args.output, os.path.basename(args.model_args))
    sd = dm.state_dict(pg.bounds)                             # collective: gathers the --categorical_node table
    if rank == 0:
        os.makedirs(args.output, exist_ok=True)
        torch.save(sd, path)                                                          # pangnn.py:339-341
    log.info(f"Saved model parameters to '{path}'")
    stat = _test(dm, pg, threshold, pos_weight, tables, test_labels)                  # pangnn.py:344-346
    log_test([stat])
    timings["outputs_s"] = _outputs(args, pg, stat, tables, N, rank, world, edge_table=bool(args.simulate_dataset))
    return dict(model=model, dataset=dataset, history=history, test=[stat], model_path=path, graph=pg, timings=timings)


def _test(dm, pg, threshold, pos_weight, tables, labels=None):
    stat = dm.evaluate(pg, threshold, pos_weight, labels)
    stat["edge_ids"] = tables["gid"]
    return stat


def _outputs(args, pg, stat, t, N, rank, world, edge_table):
    """The one-GPU CLI's test outputs (``train.add_baselines``, ``write_groups``, ``write_curves``,
    ``write_edge_table``) for the whole partitioned graph.  Without labels (``pg.y`` None) the baselines are not scored,
    no curves are written and the table's ``homolog`` column is -1.  With ``stat["sel"]`` (``--edge_split``) the
    baselines and curves are those of the test edges; the groups and the table cover every edge.  -> seconds spent."""
    t0 = time.perf_counter()
    dev = stat["logits"].device
    genome_d = torch.as_tensor(t["genome_of"], device=dev)
    order = torch.argsort(t["gid"])                           # the rank's rows in global (src, dst) order
    src, dst = t["src"][order], t["dst"][order]
    y = pg.y[order] if pg.y is not None else None
    logits = stat["logits"][order]
    q_base = (t["q_base"][order] if t["q_base"] is not None else pp.baseline_labels(src, dst, t["w"][order], genome_d))
    raw_base = (t["raw_base"][order] if t["raw_base"] is not None else
                UnionGraphDataset.raw_baseline_labels(pg.hits, src, dst, genome_d, N))
    logit_base = pp.baseline_labels(src, dst, logits, genome_d)    # segments of owned queries are all on this rank
    stat["logit_baseline"] = torch.empty_like(logit_base).index_copy_(0, order, logit_base)

    # baselines line: precision / recall / F1 from the all-reduced confusion counts (src/predict.py:77-89)
    if y is not None:
        cand = {"base_labels": q_base, "base_labels_raw": raw_base, "logit_baseline": logit_base}
        keep = stat["sel"][order] if "sel" in stat else None
        cnt = torch.stack([_counts(v, y) if keep is None else _counts(v[keep], y[keep]) for v in cand.values()])
        if world > 1:
            dist.all_reduce(cnt)
        out = {k: prf(*c, eps=0.0) for k, c in zip(cand, cnt.tolist())} if pg.num_edges_total else {}
        stat["baselines"] = out
        log.info("baselines (precision / recall / f1): " +
                 "; ".join(f"{k} {p:.4f} / {r:.4f} / {f:.4f}" for k, (p, r, f) in out.items()))

    # ortholog groups: the predicted-positive edges in global ids, gathered on rank 0 (counts, then one padded
    # gather), and the one-GPU connected components there
    sel = stat["pred"].bool()
    pos = torch.stack((t["src"][sel], t["dst"][sel]))
    sizes = torch.zeros(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(sizes, torch.tensor([pos.size(1)], dtype=torch.int64, device=dev))
    sizes = sizes.tolist()
    kmax = max(sizes)
    pad = torch.zeros(2, kmax, dtype=torch.int64, device=dev)
    pad[:, :pos.size(1)] = pos
    got = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    if kmax:
        dist.gather(pad, got, dst=0)
    if rank == 0:
        ei = torch.cat([g[:, :k] for g, k in zip(got, sizes)], dim=1)
        if ei.size(1):
            labels, groups = post.ortholog_groups(ei, torch.ones(ei.size(1), dtype=torch.int32, device=dev), N)
        else:
            labels, groups = torch.arange(N, dtype=torch.int32, device=dev), []
        stat["group_labels"], stat["groups"] = labels, groups
        path = post.write_groups_file(groups, t["names"], os.path.join(args.output, "holiest_of_all_tables.csv"))
        log.info(f"Wrote {len(groups)} ortholog groups to '{path}'")

    # ROC and precision-recall curves over the group, written by rank 0 (src/plot.py:103-107,131)
    prob, yc = stat["prob"], pg.y
    if yc is not None and "sel" in stat:
        prob, yc = prob[stat["sel"]], yc[stat["sel"]]
    roc = roc_curve(prob, yc) if yc is not None else None
    if roc is not None:
        pr = precision_recall_curve(prob, yc, drop_intermediate=True)
        if rank == 0:
            write_curve_files(roc, pr, args.output)

    # q_score_vs_logit.csv: header by rank 0, then every rank appends its rows in turn (src/predict.py:84-88)
    if edge_table:
        path = os.path.join(args.output, "q_score_vs_logit.csv")
        for r in range(world):
            if r == rank:
                post.write_q_score_vs_logit(torch.stack((src, dst)), t["w"][order], logits, y, t["names"], q_base,
                                            raw_base, logit_base, path, header=rank == 0, append=rank > 0)
            if world > 1:
                dist.barrier()
        log.info(f"Wrote '{path}' ({pg.num_edges_total} scored edges)")
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    log.debug(f"outputs written in {dt:.3f} s")
    return dt


# ------------------------------------------------------------------------------------------------
# data-parallel sub-graph training
# ------------------------------------------------------------------------------------------------
def run_data_parallel(args, device=None):
    """``train.run`` with ``--train --data_parallel`` on the ranks of the default process group: DDP under
    ``accelerate launch`` as the reference has it (``pangnn.py:25,122,155,207``).

    Every rank builds the same dataset and model from ``args.seed`` (the parameters are broadcast from rank 0), takes
    batches ``rank, rank + W, ...`` of the epoch's ``-b`` sub-graph batch list (padded to a multiple of ``W`` from its
    start, Accelerate's ``even_batches``; validation unpadded) and averages the gradients over the ranks between
    backward and the optimizer step (``dist.GradReducer``), eagerly or inside the ``--cuda_graphs`` step.  ``-b`` is
    the batch per rank; the loss is each rank's own batch mean.  The epoch's statistics are global: one all-reduce of
    the loss sums, step and batch counts and confusion counts, and the ranking metrics over the group; the scheduler
    steps on the global validation loss, so the ranks stay identical.  ``--dynamic_binary_threshold`` takes the
    Youden threshold of each step's ``W`` batches together (the one-GPU loop takes it per batch).  Every rank tests
    the model; rank 0 logs and writes ``model.pkl`` and the test outputs as ``train.run`` does."""
    rank, world = dist.get_rank(), dist.get_world_size()
    check_partition_flags(args, world)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    with _info_on_rank0(rank):
        return _run_data_parallel(args, device, rank, world)


def _run_data_parallel(args, device, rank, world):
    from .data import DeviceLoader
    from .graphs import GraphedBatchStep
    from .train import build_dataset_and_model, save_test_and_write
    dataset, model = build_dataset_and_model(args, device)
    for p in model.parameters():
        dist.broadcast(p.data, 0)
    reducer = pdist.GradReducer(list(model.parameters()))
    pos_weight = float(dataset.class_balance) if dataset.class_balance else 1.0       # pangnn.py:98
    threshold = args.binary_threshold
    history = []
    test = [g.to(device) for g in dataset.test]
    loader = lambda graphs, seed: (DeviceLoader(graphs, batch_size=args.batch_size, shuffle=True, device=device,
                                                seed=seed) if graphs else None)
    train_loader, val_loader = loader(dataset.train, args.seed), loader(dataset.val, args.seed + 1)
    stepper = None
    if args.cuda_graphs:
        optimizer = torch.optim.Adam(model.parameters(), lr=torch.tensor(0.001, device=device), capturable=True)
        stepper = GraphedBatchStep(model, optimizer, pos_weight, reduce_grads=reducer)
    else:
        optimizer = torch.optim.Adam(model.parameters(), lr=0.001)                    # pangnn.py:88
    scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", patience=10, factor=0.6)
    shard = (rank, world)
    dist.barrier()                                     # dataset build skew never counts against the reduction's wait

    for epoch in range(args.epochs):                                                  # pangnn.py:167-238
        t_ep = time.perf_counter()
        model.train()
        # [train loss sum, steps, train tn fp fn tp, val tn fp fn tp, val loss sum, val batches]
        red = torch.zeros(12, dtype=torch.float64, device=device)
        ep_prob, ep_y = [], []
        n_batches = len(train_loader) if train_loader is not None else 0
        for i, (packed, ids, ids_dev) in enumerate(train_loader.iter_ids(shard) if train_loader is not None else ()):
            if stepper is not None:
                loss, logits = stepper.step_ids(packed, ids, ids_dev)
                labels = stepper.last_y.clone()                  # the stepper's labels are static buffers
            else:
                batch = packed.collate(ids, ids_dev)
                optimizer.zero_grad()
                loss, logits = model.forward_loss(batch, pos_weight)
                loss.backward()
                reducer()
                optimizer.step()
                labels = batch.y
            prob = torch.sigmoid(logits.detach())
            if i * world + rank < n_batches:     # not a repeat of the even-batches padding (Accelerate's
                red[0] += loss.detach().double()  # gather_for_metrics drops those too): the epoch's statistics
                red[1] += 1
                ep_prob.append(prob)
                ep_y.append(labels)
                red[2:6] += _counts(prob >= threshold, labels).double()
            if args.dynamic_binary_threshold:                                         # pangnn.py:229-233
                # the step's W batches together (a padding repeat included: every rank joins every step's call)
                th = ranking_metrics(prob, labels)["youden_threshold"]
                threshold = th if th is not None else threshold
        t_val = time.perf_counter()
        model.eval()
        val_prob, val_y = [], []
        with torch.no_grad():                                                         # pangnn.py:241-275
            for batch in (val_loader.batches(shard, pad=False) if val_loader is not None else ()):
                logits, prob, pred = model.predict(batch, threshold)
                val_prob.append(prob)
                val_y.append(batch.y)
                red[10] += torch.nn.functional.binary_cross_entropy_with_logits(
                    logits, batch.y, pos_weight=torch.as_tensor(pos_weight, device=logits.device)).double()
                red[11] += 1
                red[6:10] += _counts(pred, batch.y).double()
        dist.all_reduce(red)
        reducer.check()
        red = red.tolist()
        cm, cmv = [int(v) for v in red[2:6]], [int(v) for v in red[6:10]]
        p, r, f1 = prf(*cm)
        pv, rv, f1v = prf(*cmv)
        mean_val = red[10] / max(int(red[11]), 1)
        scheduler.step(mean_val)                                                      # pangnn.py:296
        cat = lambda v: torch.cat(v) if v else torch.zeros(0, device=device)
        rk_tr = ranking_metrics(cat(ep_prob), cat(ep_y))                              # over the default group
        rk_val = ranking_metrics(cat(val_prob), cat(val_y))
        history.append(dict(epoch=epoch, train_loss=red[0] / max(int(red[1]), 1), val_loss=mean_val,
                            f1_train=f1, f1_val=f1v, precision_val=pv, recall_val=rv,
                            auroc_train=rk_tr["auroc"], ap_train=rk_tr["average_precision"],
                            auroc_val=rk_val["auroc"], ap_val=rk_val["average_precision"]))
        log.info(f"epoch {epoch}: train loss {history[-1]['train_loss']:.4f} f1 {f1:.4f} | val loss {mean_val:.4f} f1 {f1v:.4f}")
        log.info(f"epoch {epoch}: train auroc {_fmt(rk_tr['auroc'])} ap {_fmt(rk_tr['average_precision'])} | "
                 f"val auroc {_fmt(rk_val['auroc'])} ap {_fmt(rk_val['average_precision'])}")
        log.debug(f"epoch {epoch}: train steps {time.perf_counter() - t_ep:.3f} s ({int(red[1])} over {world} ranks)")

    # every replica tests its own identical copy of the test graphs: their metrics must not merge over the group (and
    # rank 0's curve files must not wait for the others), so they go through a group of this rank alone
    solo = [dist.new_group([r]) for r in range(world)][rank]
    stats, path = save_test_and_write(args, model, dataset, test, threshold, pos_weight, write=rank == 0, group=solo)
    dist.barrier()                                     # rank 0's files are complete when every rank returns
    return dict(model=model, dataset=dataset, history=history, test=stats, model_path=path)
