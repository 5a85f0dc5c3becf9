"""Host side of data-parallel sub-graph training (``pangnn.py --train --data_parallel`` under torchrun): the flag
checks, the batch sharding of ``DeviceLoader.iter_ids`` and the all-reduce form of ``dist.GradReducer`` over gloo."""
import os
import tempfile

import numpy as np
import pytest
import torch

BASE = ["--simulate_dataset", "300", "4", "0.5", "10", "3"]
DP = ["--train", "--data_parallel"]


@pytest.fixture
def flags():
    from pangnn_b200 import setup
    setup.reset()
    yield lambda argv: setup._post(setup.parser.parse_args(argv))
    setup.reset()


@pytest.mark.parametrize("extra", [["--cuda_graphs"], ["--decoder", "cosine"], ["--node_dim", "32"],
                                   ["--include_trivial"], []])
def test_data_parallel_accepts_one_gpu_flags(flags, extra):
    from pangnn_b200.dist_train import check_partition_flags
    check_partition_flags(flags(BASE + DP + extra), 2)


@pytest.mark.parametrize("argv,needle", [
    (BASE + DP + ["--whole_graph_training"], "choose one"),
    (BASE + ["--data_parallel"], "needs --train"),
    (BASE + ["--train"], "--data_parallel"),
    (BASE + ["--train"], "--whole_graph_training"),
])
def test_data_parallel_refusals(flags, argv, needle):
    from pangnn_b200.dist_train import check_partition_flags
    with pytest.raises(ValueError, match=needle.replace("-", r"\-")):
        check_partition_flags(flags(argv), 2)


@pytest.mark.parametrize("extra,needle", [(["--decoder", "cosine"], "mlp decoder"), (["--node_dim", "32"], "--node_dim 64"),
                                          (["--cuda_graphs"], "--cuda_graphs")])
def test_data_parallel_with_an_existing_model_file_is_checked_as_partitioned_inference(flags, tmp_path, extra, needle):
    """``-m`` naming an existing file restores it for inference, which runs on the genome partition: its refusals
    apply up front, as without --data_parallel."""
    from pangnn_b200.dist_train import check_partition_flags, data_parallel
    model = tmp_path / "model.pkl"
    model.write_bytes(b"")
    args = flags(BASE + DP + extra + ["-m", str(model)])
    assert not data_parallel(args)
    with pytest.raises(ValueError, match=needle.replace("-", r"\-")):
        check_partition_flags(args, 2)


def test_data_parallel_driver_needs_a_group(flags):
    """``python pangnn.py ... --data_parallel`` without torchrun stays on the one-GPU loop."""
    from pangnn_b200.dist_train import data_parallel
    assert not torch.distributed.is_initialized()
    assert not data_parallel(flags(BASE + DP))


# ------------------------------------------------------------------------------------------------
# sharding
# ------------------------------------------------------------------------------------------------
def _loader(num_graphs, batch_size, seed):
    """A ``DeviceLoader`` over ``num_graphs`` graph ids whose packed split is a stand-in (no device needed)."""
    import random
    from pangnn_b200.data import DeviceLoader
    ld = object.__new__(DeviceLoader)
    ld.packed, ld._ids = "packed", np.arange(num_graphs, dtype=np.int32) + 1000
    ld.batch_size, ld.shuffle, ld.device = batch_size, True, torch.device("cpu")
    ld._rng = random.Random(seed)
    return ld


def _ids(it):
    return [tuple(ids.tolist()) for _, ids, ids_dev in it]


def test_shard_of_one_rank_is_the_unsharded_epoch():
    for n, b in ((210, 32), (7, 3), (1, 32), (64, 32)):
        for pad in (True, False):
            a, s = _loader(n, b, 5), _loader(n, b, 5)
            for _ in range(3):                                         # successive epochs
                assert _ids(a.iter_ids()) == _ids(s.iter_ids((0, 1), pad))


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("n,b", [(210, 32), (192, 32), (24, 3), (5, 2), (3, 32)])
def test_shards_cover_the_epoch_padded_from_its_start(world, n, b):
    ref = _loader(n, b, 7)
    ranks = [_loader(n, b, 7) for _ in range(world)]
    for _ in range(2):
        full = _ids(ref.iter_ids())
        parts = [_ids(ld.iter_ids((r, world))) for r, ld in enumerate(ranks)]
        assert len({len(p) for p in parts}) == 1                    # the same number of steps on every rank
        nb = len(full)
        padded = full + [full[i % nb] for i in range(-nb % world)]
        assert len(parts[0]) * world == len(padded)
        for r in range(world):
            assert parts[r] == padded[r::world]
        for i in range(len(parts[0])):                              # global step i: batches i*W .. i*W + W-1
            assert [parts[r][i] for r in range(world)] == padded[i * world:(i + 1) * world]
        # validation: the same split without padding
        val = [_ids(ld.iter_ids((r, world), pad=False)) for r, ld in enumerate([_loader(n, b, 9) for _ in range(world)])]
        assert sorted(sum(val, [])) == sorted(_ids(_loader(n, b, 9).iter_ids()))


# ------------------------------------------------------------------------------------------------
# GradReducer, all-reduce form (gloo)
# ------------------------------------------------------------------------------------------------
SIZES = [1, 3, 64, 8192, 8256, 17]


def _grads(rank, step):
    g = torch.Generator().manual_seed(100 * step + rank)
    return [torch.randn(n, generator=g) if i != 2 else None for i, n in enumerate(SIZES)]


def _reduce_worker(rank, world, init_file, out_dir):
    import torch.distributed as dist
    from pangnn_b200.dist import GradReducer
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        params = [torch.nn.Parameter(torch.zeros(n)) for n in SIZES]
        red = GradReducer(params)
        assert red.p2p is None
        out = {}
        for step in range(3):
            for p, g in zip(params, _grads(rank, step)):
                p.grad = None if g is None else g.clone()
            red()
            red.check()
            for i, p in enumerate(params):
                out[f"s{step}_{i}"] = np.zeros(0) if p.grad is None else p.grad.numpy()
                out[f"none{step}_{i}"] = np.array(p.grad is None)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **out)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_all_reduce_reducer_over_gloo(world):
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_reduce_worker, args=(world, os.path.join(tmp, "rdv"), tmp), nprocs=world, join=True)
        outs = [dict(np.load(os.path.join(tmp, f"r{r}.npz"))) for r in range(world)]
    for step in range(3):
        for i in range(len(SIZES)):
            for o in outs:
                assert bool(o[f"none{step}_{i}"]) == (i == 2)                   # a None gradient stays None
                assert np.array_equal(o[f"s{step}_{i}"], outs[0][f"s{step}_{i}"])   # bitwise the same on every rank
            if i == 2:
                continue
            mean = np.mean([_grads(r, step)[i].numpy().astype(np.float64) for r in range(world)], axis=0)
            np.testing.assert_allclose(outs[0][f"s{step}_{i}"], mean, rtol=1e-6, atol=1e-7)


def test_main_refusal_names_both_choices(monkeypatch):
    from pangnn_b200 import setup, train
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("LOCAL_RANK", "1")
    try:
        with pytest.raises(ValueError, match=r"\-\-whole_graph_training.*\-\-data_parallel"):
            train.main(BASE + ["--train"])
    finally:
        setup.reset()
    assert not torch.distributed.is_initialized()
