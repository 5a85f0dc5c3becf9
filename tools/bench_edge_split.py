"""Cost of ``--edge_split`` on the C3 whole-graph training step, on one GPU.

    python tools/bench_edge_split.py --out profiles/edge_split.json

The C3 step (``forward_loss``, backward, Adam) with all labels and with held-out labels (``--edge_split 0.15 0.15``:
``y = -1`` on validation and test edges, the mean over train edges) alternate in one process: ``--rounds`` rounds of
``--steps`` steps each, CUDA events around every round, after ``--warmup`` steps of each.  The scorer reads the same
bytes either way, so no difference beyond noise is expected.  Also timed: the split build (``EdgeSplit.build``: the
split kernel, the counts and their host read) and one epoch's validation compaction (``labels >= 0`` selection of
the logits, probabilities and predictions).  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()}


def c3_graph(dev, n, G):
    from pangnn_b200 import ops, setup
    from pangnn_b200 import preprocessing as pp
    from pangnn_b200.data import Data
    from pangnn_b200.simulate import simulate_hits
    setup.reset()
    setup.args.union_edge_weights, setup.args.neighbours, setup.args.skip_connections = True, 3, True
    s = simulate_hits(n, G, 0.5, 50, 10, seed=0)
    N = s["num_genes"]
    src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"], num_nodes=N,
                                             t_norm=0.8, include_trivial=False, device=dev)
    ei = torch.stack((src.long(), dst.long()))
    union = ops.union_index(ei, N, 3)
    g = Data(torch.ones(N, 1, device=dev), ei, ops.union_weights(w, union.size(1)), y)
    g.union_edge_index = union
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=100000)
    ap.add_argument("--genomes", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_edge_split needs a CUDA device")
    from pangnn_b200.edge_split import TRAIN, VAL, EdgeSplit, select
    from pangnn_b200.gnn import AlternateGCN
    dev = torch.device("cuda:0")
    info = gpu_info()
    g = c3_graph(dev, a.genes, a.genomes)
    E = g.edge_index.size(1)
    torch.manual_seed(0)
    model = AlternateGCN(dev, None, False).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    pw_all = float(((g.y == 0).sum() / g.y.sum()).item())

    def build():
        return EdgeSplit.build(*g.edge_index, g.y, 0, (0.15, 0.15))

    sp = build()
    arms = {"all_labels": dict(y=None, num_labelled=None, pw=pw_all),
            "edge_split": dict(y=sp.labels(g.y, TRAIN), num_labelled=sp.count(TRAIN), pw=sp.class_balance)}

    def step(arm):
        opt.zero_grad()
        loss, _ = model.forward_loss(g, arm["pw"], y=arm["y"], num_labelled=arm["num_labelled"])
        loss.backward()
        opt.step()

    for arm in arms.values():
        for _ in range(a.warmup):
            step(arm)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for name, arm in arms.items():                    # alternate the two in every round
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(a.steps):
                step(arm)
            t1.record()
            t1.synchronize()
            times[name].append(t0.elapsed_time(t1) / a.steps)

    # the split build (kernel + counts + host read) and one epoch's validation compaction
    def timed(fn, reps=20):
        fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append((time.perf_counter() - t0) * 1e3)
        return out

    yv = sp.labels(g.y, VAL)
    with torch.no_grad():
        logits, prob, pred = model.predict(g, 0.5)
    res = dict(gpu=info, workload=f"C3 whole graph: --simulate_dataset {a.genes} {a.genomes} 0.5 50 10 "
                                   f"--union_edge_weights --neighbours 3 --skip_connections",
               scored_edges=E, split_counts=sp.counts, steps_per_round=a.steps, rounds=a.rounds,
               step_ms={k: v for k, v in times.items()},
               step_ms_median={k: float(np.median(v)) for k, v in times.items()},
               split_build_ms=timed(build), val_compaction_ms=timed(lambda: select(yv, logits, prob, pred)))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
