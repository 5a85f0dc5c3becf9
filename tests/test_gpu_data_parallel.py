"""``pangnn.py --train --data_parallel`` (pangnn_b200/dist_train.run_data_parallel) in spawned NCCL ranks.

* world 1 (an NCCL group of one rank) is bit-identical to ``train.run`` without a group, eager and ``--cuda_graphs``;
* world 2 (needs 2 GPUs; skipped otherwise): the ranks stay bitwise identical after every epoch, equal a one-process
  emulation of the global step (backward of batches 2k and 2k+1, gradients times 0.5, Adam) and agree across the
  peer-memory and NCCL transports; ``model.pkl`` of a world-2 run reproduces rank 0's test logits on one GPU.
"""
import datetime
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SIM = ["--simulate_dataset", "300", "4", "0.5", "10", "3", "--seed", "1"]
DP = ["--train", "--data_parallel", "-e", "3"]
UNION = ["--union_edge_weights", "--neighbours", "3", "--skip_connections"]
HIST = ("train_loss", "val_loss", "f1_train", "f1_val", "auroc_train", "ap_train", "auroc_val", "ap_val")


def _dirs(tmp, name):
    return ["-o", os.path.join(tmp, name), "-m", os.path.join(tmp, name, "model.pkl")]


def _run(argv, device, snapshots=None):
    from pangnn_b200 import dist as pdist, ops, setup, train
    setup.reset()
    ops.clear_cache()
    check = pdist.GradReducer.check

    def snap(self):                                           # once per epoch, after the epoch's all-reduce
        snapshots.append([p.detach().cpu().numpy().copy() for p in self.params])
        return check(self)
    if snapshots is not None:
        pdist.GradReducer.check = snap
    try:
        return train.run(setup.parse(argv), device=device)
    finally:
        pdist.GradReducer.check = check
        setup.reset()
        ops.clear_cache()


def _summary(res, snaps=()):
    t = res["test"][0]
    out = dict(logits=t["logits"].float().cpu().numpy(), pred=t["pred"].cpu().numpy().astype(np.int64))
    for k in HIST:
        out[k] = np.array([np.nan if h[k] is None else h[k] for h in res["history"]], dtype=np.float64)
    for e, ps in enumerate(snaps):
        for i, p in enumerate(ps):
            out[f"e{e}_p{i}"] = p
    return out


def _worker(rank, world, init_file, runs, out_dir, p2p, backend="nccl"):
    """``backend="gloo"`` puts every rank on GPU 0 (gloo moves CUDA tensors through the host): the driver at world > 1
    on a one-GPU box, with the all-reduce form of the gradient average."""
    import torch.distributed as dist
    os.environ["PANGNN_P2P"] = p2p
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    kw = dict(device_id=dev) if backend == "nccl" else {}
    # a rank that fails leaves its peer in a collective: a bounded timeout turns that into an error, not a hang
    dist.init_process_group(backend, init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=180), **kw)
    try:
        for i, argv in enumerate(runs):
            snaps = []
            res = _run(argv, dev, snaps)
            np.savez(os.path.join(out_dir, f"run{i}_r{rank}.npz"), **_summary(res, snaps))
    finally:
        dist.destroy_process_group()


def _same(a, b, keys=None):
    for k in (keys or a.keys()):
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "cuda_graphs"])
def test_world1_group_is_bit_identical_to_one_gpu_loop(graphs):
    extra = ["--cuda_graphs"] if graphs else []
    with tempfile.TemporaryDirectory() as tmp:
        ref = _summary(_run(SIM + DP + extra + _dirs(tmp, "ref"), "cuda:0"))
        _worker(0, 1, os.path.join(tmp, "rdv"), [SIM + DP + extra + _dirs(tmp, "dp")], tmp, "1")
        out = dict(np.load(os.path.join(tmp, "run0_r0.npz")))
        _same(ref, out, ["logits", "pred"] + list(HIST))
        a = torch.load(os.path.join(tmp, "ref", "model.pkl"), map_location="cpu")
        b = torch.load(os.path.join(tmp, "dp", "model.pkl"), map_location="cpu")
        assert list(a) == list(b)
        for k in a:
            assert torch.equal(a[k], b[k]), k
        for f in ("roc_curve.csv", "precision_recall_curve.csv", "q_score_vs_logit.csv", "holiest_of_all_tables.csv"):
            assert open(os.path.join(tmp, "ref", f), "rb").read() == open(os.path.join(tmp, "dp", f), "rb").read(), f


def _emulate(argv, epochs):
    """One process, one GPU: the world-2 global step as gradient accumulation.  -> per-epoch parameter lists."""
    from pangnn_b200 import ops, setup
    from pangnn_b200.data import DeviceLoader
    from pangnn_b200.train import build_dataset_and_model
    setup.reset()
    ops.clear_cache()
    try:
        args = setup.parse(argv)
        dev = torch.device("cuda:0")
        dataset, model = build_dataset_and_model(args, dev)
        pw = float(dataset.class_balance) if dataset.class_balance else 1.0
        opt = torch.optim.Adam(model.parameters(), lr=0.001)
        # one loader per emulated rank, seeded alike: each shuffles once per epoch, as every real rank does
        loaders = [DeviceLoader(dataset.train, batch_size=args.batch_size, shuffle=True, device=dev, seed=args.seed)
                   for _ in range(2)]
        out = []
        for _ in range(epochs):
            model.train()
            steps = [list(ld.iter_ids((r, 2))) for r, ld in enumerate(loaders)]
            for b0, b1 in zip(*steps):
                opt.zero_grad()
                for packed, ids, ids_dev in (b0, b1):
                    loss, _ = model.forward_loss(packed.collate(ids, ids_dev), pw)
                    loss.backward()
                for p in model.parameters():
                    if p.grad is not None:
                        p.grad.mul_(0.5)
                opt.step()
            out.append([p.detach().cpu().numpy().copy() for p in model.parameters()])
        return out
    finally:
        setup.reset()
        ops.clear_cache()


def _spawn(tmp, runs, p2p, tag, backend="nccl"):
    import torch.multiprocessing as mp
    d = os.path.join(tmp, tag)
    os.makedirs(d)
    mp.spawn(_worker, args=(2, os.path.join(d, "rdv"), runs, d, p2p, backend), nprocs=2, join=True)
    return [[dict(np.load(os.path.join(d, f"run{i}_r{r}.npz"))) for r in range(2)] for i in range(len(runs))]


def _params(o, epoch):
    return [o[k] for k in sorted((k for k in o if k.startswith(f"e{epoch}_p")), key=lambda k: int(k.split("_p")[1]))]


def _check_against_emulation(outs, flagsets):
    """Per-epoch parameters of every rank and run bitwise equal to the emulation; the ranks' statistics agree."""
    for i, ex in enumerate(flagsets):
        emu = _emulate(SIM + DP + ex, 3)
        runs = [o[i] for o in outs]
        a0 = runs[0][0]
        for e in range(3):
            for o in (r for pair in runs for r in pair):
                for x, y in zip(_params(o, e), emu[e]):
                    assert np.array_equal(x, y), (i, e)
        for o in (r for pair in runs for r in pair):
            for k in ("f1_train", "f1_val", "auroc_train", "ap_train", "auroc_val", "ap_val"):
                assert np.array_equal(o[k], a0[k], equal_nan=True), k
            for k in ("train_loss", "val_loss"):
                assert np.all(np.abs(o[k] - a0[k]) <= 1e-6 * np.abs(a0[k])), k
            assert np.array_equal(o["logits"], a0["logits"])


def test_world2_on_one_gpu_over_gloo_matches_gradient_accumulation():
    """The data-parallel driver at world 2 with both ranks on one GPU (gloo: the all-reduce gradient average)."""
    with tempfile.TemporaryDirectory() as tmp:
        flagsets = [[], UNION]
        out = _spawn(tmp, [SIM + DP + ex + _dirs(tmp, f"g{i}") for i, ex in enumerate(flagsets)], "0", "gloo", "gloo")
        _check_against_emulation([out], flagsets)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_world2_matches_gradient_accumulation_on_both_transports():
    with tempfile.TemporaryDirectory() as tmp:
        flagsets = [[], UNION]
        runs = lambda tag: [SIM + DP + ex + _dirs(tmp, f"{tag}{i}") for i, ex in enumerate(flagsets)]
        res = [_spawn(tmp, runs(t), "1" if t == "p2p" else "0", t) for t in ("p2p", "nccl")]
        _check_against_emulation(res, flagsets)                            # ranks and transports, bitwise


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_world2_cuda_graphs_threshold_and_categorical():
    from pangnn_b200 import setup
    with tempfile.TemporaryDirectory() as tmp:
        extras = [["--cuda_graphs"], ["--dynamic_binary_threshold"], ["--categorical_node"]]
        outs = _spawn(tmp, [SIM + DP + ex + _dirs(tmp, f"w2_{i}") for i, ex in enumerate(extras)], "1", "w2")
        for o0, o1 in outs:                                           # the ranks stay identical
            _same(o0, o1)
        # --cuda_graphs with the NCCL all-reduce captured in the graphs instead of the peer-memory kernels
        nccl = _spawn(tmp, [SIM + DP + ["--cuda_graphs"] + _dirs(tmp, "w2_nccl")], "0", "w2_nccl")[0]
        _same(*nccl)
        # --cuda_graphs against the eager emulation, with the graphs-vs-eager tolerance of test_gpu_train.py
        emu = _emulate(SIM + DP, 3)
        for o in (outs[0][0], nccl[0]):
            for e in range(3):
                for x, y in zip(_params(o, e), emu[e]):
                    assert float(np.abs(x - y).max()) <= 2e-5 * max(float(np.abs(y).max()), 1e-3)
        # model.pkl of a world-2 run in a one-GPU inference run: rank 0's test logits
        for i, ex in enumerate(extras):
            model = os.path.join(tmp, f"w2_{i}", "model.pkl")
            shape = [a for a in ex if a == "--categorical_node"]              # the flags the parameters depend on
            inf = _summary(_run(SIM + shape + ["-o", os.path.join(tmp, f"inf{i}"), "-m", model], "cuda:0"))
            assert np.array_equal(inf["logits"], outs[i][0]["logits"]), ex
        setup.reset()
