"""Data-parallel sub-graph training (``pangnn.py --train --data_parallel``) on the GPUs of one box: the training step
of ``dist_train.run_data_parallel`` in ``W`` spawned NCCL ranks, and the gradient average alone.

    python tools/bench_data_parallel.py --out profiles/r07_data_parallel.json

For every world size W in {1, 2, 4, 8} that the box has, every workload, eager and ``--cuda_graphs``, and both
transports of ``dist.GradReducer`` (NVLink peer memory and NCCL all-reduce; one run at W = 1, where the reducer does
nothing): ms per step, from CUDA events around whole epochs (one warm-up epoch, then ``--epochs`` timed), and scored
train edges per second summed over the ranks.  ``-b`` is the batch per rank, as under Accelerate.

The reducer alone: ``GradReducer()`` on a fixed list of the model's default gradient sizes (54 k floats, 216 KB) over
``--calls`` calls between CUDA events, both transports; at W = 1 the kernel pair is timed with one emulated rank, both
as Python calls and replayed from a CUDA graph (device time alone).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

WORKLOADS = {
    "config2": ["--simulate_dataset", "10000", "2", "0.5", "10", "3", "-b", "32"],        # BASELINE config 2
    "larger": ["--simulate_dataset", "20000", "4", "0.5", "10", "3", "-b", "128"],
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()}


def _train_epochs(argv, graphs, epochs, dev, rank, world):
    """The step loop of ``run_data_parallel`` (no validation): -> (ms per step, scored edges per rank per epoch)."""
    import torch.distributed as dist
    from pangnn_b200 import dist as pdist, ops, setup
    from pangnn_b200.data import DeviceLoader
    from pangnn_b200.graphs import GraphedBatchStep
    from pangnn_b200.train import build_dataset_and_model
    setup.reset()
    ops.clear_cache()
    args = setup.parse(argv)
    dataset, model = build_dataset_and_model(args, dev)
    for p in model.parameters():
        dist.broadcast(p.data, 0)
    reducer = pdist.GradReducer(list(model.parameters()))
    pw = float(dataset.class_balance)
    loader = DeviceLoader(dataset.train, batch_size=args.batch_size, shuffle=True, device=dev, seed=args.seed)
    if graphs:
        opt = torch.optim.Adam(model.parameters(), lr=torch.tensor(0.001, device=dev), capturable=True)
        stepper = GraphedBatchStep(model, opt, pw, reduce_grads=reducer)
    else:
        opt = torch.optim.Adam(model.parameters(), lr=0.001)

    def epoch():
        steps, edges = 0, torch.zeros((), dtype=torch.int64, device=dev)
        for packed, ids, ids_dev in loader.iter_ids((rank, world)):
            if graphs:
                _, logits = stepper.step_ids(packed, ids, ids_dev)
            else:
                batch = packed.collate(ids, ids_dev)
                opt.zero_grad()
                loss, logits = model.forward_loss(batch, pw)
                loss.backward()
                reducer()
                opt.step()
            edges += logits.numel()
            steps += 1
        return steps, edges
    dist.barrier()
    epoch()                                                 # warm-up: captures, lazy inits
    torch.cuda.synchronize()
    dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    steps, edges = 0, 0
    for _ in range(epochs):
        s, e = epoch()
        steps, edges = steps + s, edges + int(e)
    t1.record()
    torch.cuda.synchronize()
    reducer.check()
    ms = t0.elapsed_time(t1)
    setup.reset()
    return ms / steps, edges / (ms / 1e3)


def _reducer_alone(dev, rank, world, calls):
    import torch.distributed as dist
    from pangnn_b200 import dist as pdist, ops
    from pangnn_b200.gnn import AlternateGCN
    torch.manual_seed(0)
    model = AlternateGCN(dev, None, False).to(dev)
    params = [p for p in model.parameters()]
    for p in params:
        p.grad = torch.randn_like(p)
    out = {"floats": sum(p.numel() for p in params)}
    for p2p in ("1", "0"):
        os.environ["PANGNN_P2P"] = p2p
        red = pdist.GradReducer(params)
        if world == 1:                                      # the kernel pair with one emulated rank
            half = ops.grad_bucket_floats(red.numels)
            bucket = torch.zeros(2, half, device=dev)
            sig = torch.zeros(8, dtype=torch.int32, device=dev)
            ctrl = torch.zeros(4, dtype=torch.int32, device=dev)
            grads, numels = [p.grad for p in params], red.numels
            red = lambda: (ops.grad_push(grads, numels, bucket, half, [sig.data_ptr()], 0, ctrl),
                           ops.grad_reduce(grads, numels, [bucket.data_ptr()], half, sig, 0, ctrl))
            transport = "kernels, one emulated rank"
        else:
            transport = "p2p" if red.p2p is not None else "nccl"
        for _ in range(20):
            red()
        torch.cuda.synchronize()
        dist.barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(calls):
            red()
        t1.record()
        torch.cuda.synchronize()
        out[transport] = {"us_per_call": t0.elapsed_time(t1) * 1e3 / calls, "calls": calls}
        if world == 1:
            # the same pair captured 100 times in one CUDA graph and replayed: device time without the host calls
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(100):
                    red()
            g.replay()
            torch.cuda.synchronize()
            reps = max(calls // 100, 1)
            t0.record()
            for _ in range(reps):
                g.replay()
            t1.record()
            torch.cuda.synchronize()
            out[transport]["us_per_call_graph_replay"] = t0.elapsed_time(t1) * 1e3 / (100 * reps)
            break
    os.environ["PANGNN_P2P"] = "1"
    return out


def _worker(rank, world, init_file, opts, out_dir):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    res = {"reducer": None, "steps": []}
    try:
        res["reducer"] = _reducer_alone(dev, rank, world, opts["calls"])
        for name, argv in WORKLOADS.items():
            for graphs in (False, True):
                for p2p in (("1", "0") if world > 1 else ("1",)):
                    os.environ["PANGNN_P2P"] = p2p
                    extra = ["--train", "--data_parallel", "--seed", "0"] + (["--cuda_graphs"] if graphs else [])
                    ms, eps = _train_epochs(argv + extra, graphs, opts["epochs"], dev, rank, world)
                    res["steps"].append(dict(workload=name, argv=argv + extra, cuda_graphs=graphs,
                                             transport=("p2p" if p2p == "1" else "nccl") if world > 1 else "none",
                                             ms_per_step=ms, edges_per_s=eps))
        if rank == 0:
            with open(os.path.join(out_dir, "w.json"), "w") as f:
                json.dump(res, f)
        # every rank's edges/s: summed over the ranks below
        with open(os.path.join(out_dir, f"eps_r{rank}.json"), "w") as f:
            json.dump([s["edges_per_s"] for s in res["steps"]], f)
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, nargs="*", default=[1, 2, 4, 8])
    ap.add_argument("--epochs", type=int, default=2)
    ap.add_argument("--calls", type=int, default=2000)
    ap.add_argument("--out", default=None)
    o = ap.parse_args()
    import torch.multiprocessing as mp
    from pangnn_b200 import build
    build.build()
    report = {"gpu": gpu_info(), "gpus_visible": torch.cuda.device_count(), "worlds": {}}
    for world in o.worlds:
        if world > torch.cuda.device_count():
            report["worlds"][str(world)] = "not measured: not enough GPUs"
            continue
        with tempfile.TemporaryDirectory() as tmp:
            mp.spawn(_worker, args=(world, os.path.join(tmp, "rdv"), {"epochs": o.epochs, "calls": o.calls}, tmp),
                     nprocs=world, join=True)
            res = json.load(open(os.path.join(tmp, "w.json")))
            eps = [json.load(open(os.path.join(tmp, f"eps_r{r}.json"))) for r in range(world)]
        for i, s in enumerate(res["steps"]):
            s["edges_per_s_rank0"] = s.pop("edges_per_s")
            s["edges_per_s_all_ranks"] = sum(e[i] for e in eps)
        report["worlds"][str(world)] = res
        print(json.dumps({world: res}, indent=1), flush=True)
    if o.out:
        os.makedirs(os.path.dirname(o.out) or ".", exist_ok=True)
        with open(o.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
