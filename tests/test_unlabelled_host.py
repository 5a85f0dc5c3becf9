"""Host side of inference without labels (``-r ''``): the flag checks that refuse training without a RIBAP table on
every rank alike, the per-edge table without its ``homolog`` column, and a partition of a graph without ``y``."""
import numpy as np
import pytest
import torch

FILES = ["-a", "a.gff", "b.gff", "-s", "hits.tsv"]
SIM = ["--simulate_dataset", "300", "4", "0.5", "10", "3"]


@pytest.fixture
def flags():
    from pangnn_b200 import setup
    setup.reset()
    yield lambda argv: setup._post(setup.parser.parse_args(argv))
    setup.reset()


@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("extra", [["--train"], ["--train", "--whole_graph_training"], ["--train", "--data_parallel"]],
                         ids=["subgraphs", "whole_graph", "data_parallel"])
def test_training_without_labels_is_refused(flags, world, extra):
    from pangnn_b200.dist_train import check_partition_flags
    with pytest.raises(ValueError, match="--train needs labels.*-r"):
        check_partition_flags(flags(FILES + ["-r", ""] + extra), world)


@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("argv", [FILES + ["-r", "", "-m", "model.pkl"],                  # inference without labels
                                  SIM + ["-r", "", "--train", "--whole_graph_training"]],  # simulated data has labels
                         ids=["files_inference", "simulated_train"])
def test_unlabelled_inference_and_simulated_training_are_accepted(flags, world, argv):
    from pangnn_b200 import setup
    from pangnn_b200.dist_train import check_partition_flags
    ns = flags(argv)
    setup.check_label_flags(ns)
    check_partition_flags(ns, world)


def test_has_labels(flags):
    from pangnn_b200 import setup
    assert setup.has_labels(flags(FILES + ["-r", "ribap.csv"]))
    assert setup.has_labels(flags(FILES))                                    # the default table
    assert not setup.has_labels(flags(FILES + ["-r", ""]))
    assert setup.has_labels(flags(SIM + ["-r", ""]))


def test_cli_refuses_training_without_labels_before_any_device_work(monkeypatch):
    """One process (``train.run``) and every rank under torchrun (``train.main`` with ``WORLD_SIZE=2``) stop on the
    flags before they build a dataset, touch a GPU or join a process group (this box has neither)."""
    from pangnn_b200 import setup, train
    try:
        with pytest.raises(ValueError, match="--train needs labels"):
            train.run(setup.parse(FILES + ["-r", "", "--train"]))
        setup.reset()
        monkeypatch.setenv("WORLD_SIZE", "2")
        monkeypatch.setenv("LOCAL_RANK", "1")
        with pytest.raises(ValueError, match="--train needs labels"):
            train.main(FILES + ["-r", "", "--train", "--whole_graph_training"])
    finally:
        setup.reset()
    assert not torch.distributed.is_initialized()


@pytest.mark.parametrize("names", [False, True])
def test_q_score_table_without_labels(tmp_path, names):
    """``labels=None``: ``homolog`` is -1 on every row, every other byte is the labelled call's."""
    from pangnn_b200.postprocessing import Q_SCORE_VS_LOGIT_COLUMNS, write_q_score_vs_logit
    rng = np.random.default_rng(1)
    E, N = 311, 70
    ei = np.stack((np.sort(rng.integers(0, N, E)), rng.integers(0, N, E)))
    w = rng.random(E, dtype=np.float32)
    logits = (rng.standard_normal(E) * 3).astype(np.float32)
    y = rng.integers(0, 2, E).astype(np.float32)
    base = [rng.integers(0, 2, E) for _ in range(3)]
    gene = [f"G{i}_{i:06d}" for i in range(N)] if names else None
    a, b = str(tmp_path / "labelled.csv"), str(tmp_path / "unlabelled.csv")
    write_q_score_vs_logit(ei, w, logits, y, gene, *base, path=a)
    write_q_score_vs_logit(ei, w, logits, None, gene, *base, path=b)
    la, lb = open(a).read().splitlines(), open(b).read().splitlines()
    assert la[0] == lb[0] == ",".join(Q_SCORE_VS_LOGIT_COLUMNS) and len(la) == len(lb) == E + 1
    h = Q_SCORE_VS_LOGIT_COLUMNS.index("homolog")
    for ra, rb in zip(la[1:], lb[1:]):
        fa, fb = ra.split(","), rb.split(",")
        assert fb[h] == "-1" and fa[h] in ("0", "1")
        assert fa[:h] + fa[h + 1:] == fb[:h] + fb[h + 1:]


def test_partition_of_a_graph_without_labels():
    """``PartitionedGraph(y=None)`` (one rank, on the host: pure index arithmetic) keeps no labels and no class
    balance, and counts the same scored edges as with labels."""
    from pangnn_b200 import setup
    from pangnn_b200.dist import PartitionedGraph
    setup.reset()
    g = torch.Generator().manual_seed(0)
    N, E = 40, 200
    key = torch.unique(torch.randint(0, N * N, (E,), generator=g))
    ei = torch.stack((key // N, key % N))
    w = torch.rand(ei.size(1), generator=g)
    y = (torch.rand(ei.size(1), generator=g) < 0.3).float()
    band = torch.stack((torch.arange(N), torch.arange(N)))
    parts = [PartitionedGraph([0, N], 0, 1, torch.ones(N, 1), ei, w, band, ei, w, lab) for lab in (y, None)]
    assert parts[0].num_edges_total == parts[1].num_edges_total == ei.size(1)
    assert parts[0].class_balance == pytest.approx(float((y == 0).sum() / y.sum()))
    assert parts[1].y is None and parts[1].class_balance is None
    assert torch.equal(parts[0].scored_edge_ids, parts[1].scored_edge_ids)
