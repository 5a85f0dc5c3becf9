"""Ranking metrics (``pangnn_b200.metrics.ranking_metrics``) on the B200: whole call, sort share, post-sort share,
algorithmic bytes, peak extra memory, sklearn on the host for comparison, and the multi-GPU merge.  With ``--curves``:
``roc_curve`` / ``precision_recall_curve`` instead: whole calls, the share of the curve kernels
(``pangnn_metric_curve`` timed alone on the same runs), curve lengths with and without thinning, and sklearn's
``roc_curve`` / ``precision_recall_curve`` on the host for the same input.

    python tools/bench_metrics.py --out profiles/metrics_1gpu.json
    python tools/bench_metrics.py --gpus 2 --out profiles/metrics_2gpu.json
    python tools/bench_metrics.py --curves --out profiles/curves_1gpu.json

Inputs are model-shaped: sigmoid of a bimodal logit (positives N(4, 3), negatives N(-4, 3)) at the positive fraction
of C3 (18 %) and of C5 (1 %), with 2 % of the scores saturated at 1.0f (ties).  E >= 1e7 exceeds the L2 (8 + 4 B per
score in, 12 B per element per sort pass); the 1e6 size is L2-resident after the first pass.  The sort share is the
same four-pass ``pangnn_sort_pairs_u64`` timed alone on the same number of (key, label) pairs; the rest of the call
(key pass, compaction, reduction, one host read-back) is the difference.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FRACTIONS = {"C3": 0.18, "C5": 0.01}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()}


def scores(E, frac, device, seed=0):
    g = torch.Generator(device=device).manual_seed(seed)
    y = torch.rand(E, generator=g, device=device) < frac
    logit = torch.randn(E, generator=g, device=device) * 3.0 + torch.where(y, 4.0, -4.0)
    prob = torch.sigmoid(logit)
    prob[torch.rand(E, generator=g, device=device) < 0.02] = 1.0
    return prob.float(), y.float()


def timed(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def algorithmic_bytes(E, R):
    """Bytes the pipeline has to move: key pass (read 4 + 4, write 8 + 4), four sort passes (histogram read 8,
    scatter read 12 + write 12), compaction (two reads of 12 B per element, 24 B per run written), reduction (two
    reads of 24 B per run)."""
    key = E * 20
    sort = 4 * E * 32
    post = E * 24 + R * 24 + R * 48
    return key, sort, post


def one_gpu(sizes, reps):
    from pangnn_b200 import ops
    from pangnn_b200.metrics import ranking_metrics
    dev = torch.device("cuda:0")
    rows = []
    for name, frac in FRACTIONS.items():
        for E in sizes:
            s, y = scores(E, frac, dev)
            r = ranking_metrics(s, y)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            ranking_metrics(s, y)
            peak = torch.cuda.max_memory_allocated() - base
            reps_e = max(3, reps // max(1, E // 10_000_000))
            t_call = timed(lambda: ranking_metrics(s, y), reps_e)
            keys = torch.randint(0, 1 << 32, (E,), device=dev, dtype=torch.int64)
            vals = y.int()
            t_sort = timed(lambda: ops.sort_pairs_u64(keys, vals, key_bits=32), reps_e)
            kb, sb, pb = algorithmic_bytes(E, r["num_runs"])
            rows.append(dict(
                workload=name, pos_fraction=frac, E=E, runs=r["num_runs"], auroc=r["auroc"],
                average_precision=r["average_precision"], call_ms=t_call, sort_ms=t_sort,
                rest_ms=t_call - t_sort, sort_share=t_sort / t_call, rest_share=(t_call - t_sort) / t_call,
                algorithmic_bytes=dict(key_pass=kb, sort=sb, post_sort=pb),
                call_GBps=(kb + sb + pb) / (t_call * 1e6), sort_GBps=sb / (t_sort * 1e6),
                peak_extra_bytes_per_edge=peak / E))
            print(json.dumps(rows[-1]), flush=True)
            del s, y, keys, vals
            torch.cuda.empty_cache()
    return rows


def sklearn_rows(sizes):
    from sklearn.metrics import average_precision_score, roc_auc_score
    from pangnn_b200.metrics import ranking_metrics
    rows = []
    for E in sizes:
        s, y = scores(E, FRACTIONS["C3"], torch.device("cuda:0"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sh, yh = s.cpu().numpy(), y.cpu().numpy()
        auc, ap = roc_auc_score(yh, sh), average_precision_score(yh, sh)
        t = time.perf_counter() - t0
        r = ranking_metrics(s, y)
        rows.append(dict(E=E, sklearn_incl_d2h_ms=t * 1e3, auroc_abs_diff=abs(auc - r["auroc"]),
                         ap_abs_diff=abs(ap - r["average_precision"])))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def curve_rows(sizes, reps):
    """Whole calls of the four curve variants, ``metric_runs`` and ``metric_curve`` alone (per mode) on the same
    input, curve lengths, and the curve pass's algorithmic bytes: two reads of 24 B per run (tile statistics, emit)
    and 20 B per kept point (fp32 threshold, int64 TP and FP)."""
    from pangnn_b200 import ops
    from pangnn_b200.metrics import precision_recall_curve, roc_curve
    dev = torch.device("cuda:0")
    calls = {"roc_thinned": lambda s, y: roc_curve(s, y),
             "roc_all": lambda s, y: roc_curve(s, y, drop_intermediate=False),
             "pr_all": lambda s, y: precision_recall_curve(s, y),
             "pr_thinned": lambda s, y: precision_recall_curve(s, y, drop_intermediate=True)}
    modes = {"all": ops.CURVE_ALL, "roc": ops.CURVE_ROC, "pr": ops.CURVE_PR}
    rows = []
    for name, frac in FRACTIONS.items():
        for E in sizes:
            s, y = scores(E, frac, dev)
            reps_e = max(3, reps // max(1, E // 10_000_000))
            row = dict(workload=name, pos_fraction=frac, E=E)
            for k, fn in calls.items():
                row[f"{k}_len"] = fn(s, y)[0].numel()
                row[f"{k}_ms"] = timed(lambda: fn(s, y), reps_e)
            info = torch.zeros(6, dtype=torch.int64, device=dev)
            row["metric_runs_ms"] = timed(lambda: ops.metric_runs(s, y, info=info), reps_e)
            runs = ops.metric_runs(s, y, info=info)
            R = int(info[0])
            bound = torch.tensor([0, 0, ops.CURVE_FIRST], dtype=torch.int64, device=dev)
            out = (torch.empty(runs.size(0), dtype=torch.float32, device=dev),
                   torch.empty(runs.size(0), dtype=torch.int64, device=dev),
                   torch.empty(runs.size(0), dtype=torch.int64, device=dev), torch.empty(3, dtype=torch.int64, device=dev))
            row["runs"] = R
            for k, mode in modes.items():
                t = timed(lambda: ops.metric_curve(runs, info, bound, mode, out=out), reps_e)
                kept = int(out[3][0])
                row[f"curve_kernel_{k}_ms"] = t
                row[f"curve_kernel_{k}_kept"] = kept
                row[f"curve_kernel_{k}_GBps"] = (48 * R + 20 * kept) / (t * 1e6)
            row["curve_kernel_share_of_roc_thinned"] = row["curve_kernel_roc_ms"] / row["roc_thinned_ms"]
            row["curve_kernel_share_of_pr_all"] = row["curve_kernel_all_ms"] / row["pr_all_ms"]
            row["curve_kernel_roc_vs_metric_runs"] = row["curve_kernel_roc_ms"] / row["metric_runs_ms"]
            rows.append(row)
            print(json.dumps(row), flush=True)
            del s, y, runs, out
            torch.cuda.empty_cache()
    return rows


def sklearn_curve_rows(sizes):
    """sklearn on the host (including the device-to-host copy of the scores) and bit-equality with the device."""
    import numpy as np
    from sklearn.metrics import precision_recall_curve as sk_pr, roc_curve as sk_roc
    from pangnn_b200.metrics import precision_recall_curve, roc_curve
    rows = []
    for E in sizes:
        s, y = scores(E, FRACTIONS["C3"], torch.device("cuda:0"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sh, yh = s.cpu().numpy(), y.cpu().numpy()
        roc = sk_roc(yh, sh)
        t_roc = time.perf_counter() - t0
        t0 = time.perf_counter()
        sh, yh = s.cpu().numpy(), y.cpu().numpy()
        pr = sk_pr(yh, sh)
        t_pr = time.perf_counter() - t0
        same = all(a.dtype == b.cpu().numpy().dtype and np.array_equal(a, b.cpu().numpy())
                   for a, b in zip(roc + pr, roc_curve(s, y) + precision_recall_curve(s, y)))
        rows.append(dict(E=E, sklearn_roc_curve_incl_d2h_ms=t_roc * 1e3, sklearn_pr_curve_incl_d2h_ms=t_pr * 1e3,
                         bit_equal_to_device=same))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def _dist_worker(rank, world, init_file, sizes, reps, out_path):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    try:
        from pangnn_b200 import metrics
        rows = []
        for E in sizes:
            s, y = scores(E // world, FRACTIONS["C3"], dev, seed=rank + 1)
            r = metrics.ranking_metrics(s, y)

            def call():
                metrics.ranking_metrics(s, y)
                dist.barrier()
            t = timed(call, reps)
            ex = dict(metrics.LAST_EXCHANGE)
            got = [None] * world
            dist.all_gather_object(got, ex)
            if rank == 0:
                rows.append(dict(world=world, E_total=E, E_local=E // world, call_ms=t, runs=r["num_runs"],
                                 bytes_sent_per_rank=[g["bytes_sent"] for g in got],
                                 local_runs_per_rank=[g["local_runs"] for g in got],
                                 received_runs_per_rank=[g["received_runs"] for g in got]))
                print(json.dumps(rows[-1]), flush=True)
        if rank == 0:
            with open(out_path, "w") as f:
                json.dump(rows, f)
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--curves", action="store_true", help="time roc_curve / precision_recall_curve (one GPU)")
    a = ap.parse_args()
    from pangnn_b200 import build
    if not build.is_current():
        raise SystemExit("the CUDA library is not built or is stale: run `python -m pangnn_b200.build`")
    res = dict(gpu=gpu_info())
    if a.curves:
        res["curves"] = curve_rows([1_000_000, 10_000_000, 100_000_000], a.reps)
        res["sklearn_curves_host"] = sklearn_curve_rows([1_000_000, 10_000_000])
    elif a.gpus == 1:
        res["one_gpu"] = one_gpu([1_000_000, 10_000_000, 100_000_000], a.reps)
        res["sklearn_host"] = sklearn_rows([1_000_000, 10_000_000])
    else:
        import tempfile
        import torch.multiprocessing as mp
        if torch.cuda.device_count() < a.gpus:
            raise SystemExit(f"--gpus {a.gpus}: only {torch.cuda.device_count()} devices")
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "rows.json")
            mp.spawn(_dist_worker, args=(a.gpus, os.path.join(tmp, "rdv"), [10_000_000, 100_000_000], a.reps, path),
                     nprocs=a.gpus, join=True)
            with open(path) as f:
                res["multi_gpu"] = json.load(f)
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
