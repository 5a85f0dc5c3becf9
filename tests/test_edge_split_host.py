"""``--edge_split`` on the host (pangnn_b200/edge_split.py): a numpy restatement of the split rule (Philox4x32-10 keyed
by (seed, purpose 5) at counter (0, min, max, 0)), its symmetry, fractions and order independence, the flag refusals,
and the global counts and class balance over gloo at world 2 and 3, with the numpy rule standing in for the kernel."""
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

M = 0xFFFFFFFF


def philox_first_word(seed, purpose, a, b):
    """First output word of Philox4x32-10 keyed by (seed, purpose) at counter (0, a, b, 0), vectorised over a, b
    (``csrc/philox.cuh``)."""
    a = np.asarray(a, dtype=np.uint64) & M
    b = np.asarray(b, dtype=np.uint64) & M
    c0, c1, c2, c3 = np.zeros_like(a), a, b, np.zeros_like(a)
    k0 = np.uint64(seed & M)
    k1 = np.uint64(((seed >> 32) & M) ^ ((purpose * 0x9E3779B9) & M))
    m0, m1, mask = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(M)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                       # < 2^64: exact in uint64
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & mask, (k1 + np.uint64(0xBB67AE85)) & mask
    return c0


def split_rule(src, dst, seed, val, test):
    """int8 codes (0 train, 1 validation, 2 test) of the edges (src, dst)."""
    from pangnn_b200.edge_split import PURPOSE, thresholds
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    t_val, t_test = thresholds(val, test)
    x = philox_first_word(seed, PURPOSE, np.minimum(src, dst), np.maximum(src, dst)).astype(np.int64)
    return np.where(x < t_val, 1, np.where(x < t_val + t_test, 2, 0)).astype(np.int8)


def test_philox_known_answer():
    """The Random123 known-answer vector of Philox4x32-10 (key 0, counter 0): first word 0x6627e8d5.  Purpose 0 and
    seed 0 give key (0, 0) in the project's keying."""
    assert int(philox_first_word(0, 0, [0], [0])[0]) == 0x6627E8D5


def test_thresholds_are_integer_floors():
    from pangnn_b200.edge_split import thresholds
    assert thresholds(0.5, 0.25) == (1 << 31, 1 << 30)
    assert thresholds(0.15, 0.15) == (644245094, 644245094)
    t_val, t_test = thresholds(0.3, 0.6999999)
    assert t_val + t_test < 1 << 32


def test_symmetric_and_order_independent():
    rng = np.random.default_rng(0)
    s, d = rng.integers(0, 2 ** 31 - 1, 10000), rng.integers(0, 2 ** 31 - 1, 10000)
    a = split_rule(s, d, 7, 0.2, 0.1)
    assert np.array_equal(a, split_rule(d, s, 7, 0.2, 0.1))
    perm = rng.permutation(s.size)
    assert np.array_equal(a[perm], split_rule(s[perm], d[perm], 7, 0.2, 0.1))
    assert not np.array_equal(a, split_rule(s, d, 8, 0.2, 0.1))     # the seed keys the split


def test_fractions_within_5_sigma():
    n = 1_000_000
    rng = np.random.default_rng(1)
    s = rng.integers(0, 50_000_000, n)
    d = s + 1 + rng.integers(0, 1000, n)
    for val, test in ((0.15, 0.15), (0.01, 0.3)):
        codes = split_rule(s, d, 3, val, test)
        for code, f in ((1, val), (2, test), (0, 1 - val - test)):
            k = int((codes == code).sum())
            assert abs(k - n * f) <= 5 * np.sqrt(n * f * (1 - f)), (val, test, code, k)


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
SIM = ["--simulate_dataset", "300", "4", "0.5", "10", "3"]
REFUSED = {
    "subgraph_training": SIM + ["--train", "--edge_split", "0.1", "0.1"],
    "data_parallel": SIM + ["--train", "--data_parallel", "--edge_split", "0.1", "0.1"],
    "no_labels": ["-a", "x.gff", "-s", "h.tsv", "-r", "", "--edge_split", "0.1", "0.1"],
    "zero_val": SIM + ["--train", "--whole_graph_training", "--edge_split", "0", "0.1"],
    "zero_test": SIM + ["--train", "--whole_graph_training", "--edge_split", "0.1", "0"],
    "negative": SIM + ["--train", "--whole_graph_training", "--edge_split", "-0.1", "0.2"],
    "sum_one": SIM + ["--train", "--whole_graph_training", "--edge_split", "0.5", "0.5"],
}
ACCEPTED = {
    "whole_graph": SIM + ["--train", "--whole_graph_training", "--edge_split", "0.15", "0.15"],
    "inference": SIM + ["--edge_split", "0.15", "0.15"],
    "files_inference": ["-a", "x.gff", "-s", "h.tsv", "-r", "groups.csv", "--edge_split", "0.1", "0.2"],
    "off": SIM + ["--train"],
}


def _ns(argv):
    from pangnn_b200 import setup
    return setup._post(setup.parser.parse_args(argv))


@pytest.mark.parametrize("name", sorted(REFUSED))
@pytest.mark.parametrize("world", [1, 2])
def test_refused_by_flags(name, world):
    from pangnn_b200 import dist_train, edge_split
    ns = _ns(REFUSED[name])
    with pytest.raises(ValueError, match="--edge_split"):
        edge_split.check_flags(ns)
    with pytest.raises(ValueError, match="--edge_split"):
        dist_train.check_partition_flags(ns, world)


@pytest.mark.parametrize("name", sorted(REFUSED))
def test_refused_by_train_run_before_device_work(name):
    from pangnn_b200 import train
    with pytest.raises(ValueError, match="--edge_split"):
        train.run(_ns(REFUSED[name]), device="cpu")


@pytest.mark.parametrize("name", sorted(ACCEPTED))
def test_accepted(name):
    from pangnn_b200 import dist_train, edge_split
    ns = _ns(ACCEPTED[name])
    edge_split.check_flags(ns)
    dist_train.check_partition_flags(ns, 1)


def test_flag_default_is_off():
    assert _ns([]).edge_split is None


# ------------------------------------------------------------------------------------------------
# EdgeSplit on the host, world 1 and over gloo
# ------------------------------------------------------------------------------------------------
def _graph(seed=5, n=3000, e=20000):
    rng = np.random.default_rng(seed)
    s = rng.integers(0, n, e)
    d = (s + 1 + rng.integers(0, n - 1, e)) % n
    y = (rng.random(e) < 0.3).astype(np.float32)
    return s, d, y


def test_edge_split_counts_labels_and_select():
    from pangnn_b200.edge_split import TEST, TRAIN, VAL, EdgeSplit, select
    s, d, y = _graph()
    codes = split_rule(s, d, 11, 0.15, 0.15)
    sp = EdgeSplit(torch.from_numpy(codes), torch.from_numpy(y))
    assert sp.counts == tuple(int((codes == k).sum()) for k in (TRAIN, VAL, TEST))
    pos = int(((codes == TRAIN) & (y == 1)).sum())
    assert sp.train_positives == pos and sp.class_balance == (sp.counts[TRAIN] - pos) / pos
    yt = torch.from_numpy(y)
    for k in (TRAIN, VAL, TEST):
        lab = sp.labels(yt, k)
        assert torch.equal(lab[torch.from_numpy(codes == k)], yt[torch.from_numpy(codes == k)])
        assert bool((lab[torch.from_numpy(codes != k)] == -1).all())
        kept, p = select(lab, torch.arange(y.size))
        assert torch.equal(p, torch.from_numpy(np.nonzero(codes == k)[0]))
        assert torch.equal(kept, yt[p])


def test_edge_split_without_positive_train_edge_raises():
    from pangnn_b200.edge_split import EdgeSplit
    s, d, _ = _graph()
    codes = split_rule(s, d, 11, 0.15, 0.15)
    y = np.where(codes == 0, 0.0, 1.0).astype(np.float32)
    with pytest.raises(ValueError, match="no positive edge"):
        EdgeSplit(torch.from_numpy(codes), torch.from_numpy(y))


def _worker(rank, world, init_file, parts, out_dir):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        from pangnn_b200 import edge_split
        s, d, y = parts[rank]
        # the numpy rule stands in for the kernel: every rank splits its own edges
        edge_split.split_codes = lambda src, dst, seed, val, test: torch.from_numpy(
            split_rule(src.numpy(), dst.numpy(), seed, val, test))
        sp = edge_split.EdgeSplit.build(torch.from_numpy(s), torch.from_numpy(d), torch.from_numpy(y), 11, (0.15, 0.15))
        torch.save(dict(counts=sp.counts, pos=sp.train_positives, balance=sp.class_balance),
                   os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_global_counts_equal_world1(world):
    from pangnn_b200.edge_split import EdgeSplit
    s, d, y = _graph()
    ref = EdgeSplit(torch.from_numpy(split_rule(s, d, 11, 0.15, 0.15)), torch.from_numpy(y))
    # ranks own contiguous source ranges, as on the genome partition
    n = int(max(s.max(), d.max())) + 1
    cuts = np.linspace(0, n, world + 1).astype(np.int64)
    parts = [tuple(a[(s >= lo) & (s < hi)] for a in (s, d, y)) for lo, hi in zip(cuts[:-1], cuts[1:])]
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, os.path.join(tmp, "rdv"), parts, tmp), nprocs=world, join=True)
        for r in range(world):
            got = torch.load(os.path.join(tmp, f"r{r}.pt"))
            assert got["counts"] == ref.counts and got["pos"] == ref.train_positives
            assert got["balance"] == ref.class_balance
