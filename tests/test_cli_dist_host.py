"""Host side of ``pangnn.py`` on several GPUs (pangnn_b200/dist_train.py): the flag combinations the partitioned
driver refuses, and the per-edge table written in rank-ordered pieces."""
import numpy as np
import pytest
import torch

BASE = ["--simulate_dataset", "300", "4", "0.5", "10", "3"]
TRAIN = ["--train", "--whole_graph_training"]


@pytest.fixture
def flags():
    from pangnn_b200 import setup
    setup.reset()
    yield lambda argv: setup._post(setup.parser.parse_args(argv))
    setup.reset()


@pytest.mark.parametrize("argv,world,needle", [
    (BASE + ["--train"], 2, "--whole_graph_training"),
    (BASE + TRAIN + ["--include_trivial"], 2, "--include_trivial"),
    (BASE + TRAIN + ["--decoder", "cosine"], 2, "mlp decoder"),
    (BASE + TRAIN + ["--node_dim", "32"], 2, "--node_dim 64"),
    (BASE + ["--decoder", "dot"], 1, "mlp decoder"),
    (BASE + TRAIN + ["--cuda_graphs"], 4, "--cuda_graphs"),
])
def test_partitioned_driver_refuses(flags, argv, world, needle):
    from pangnn_b200.dist_train import check_partition_flags
    with pytest.raises(ValueError, match=needle.replace("-", r"\-")):
        check_partition_flags(flags(argv), world)


@pytest.mark.parametrize("argv,world", [
    (BASE + TRAIN, 8),
    (BASE + TRAIN + ["--union_edge_weights", "--neighbours", "3", "--skip_connections"], 2),
    (BASE + TRAIN + ["--base_model", "--categorical_node", "--dynamic_binary_threshold"], 2),
    (BASE, 2),                                                   # inference
    (BASE + ["--train"], 1),                                     # one rank: the one-GPU sub-graph loop
    (BASE + TRAIN + ["--include_trivial", "--cuda_graphs"], 1),
    (["-a", "a.gff", "b.gff", "-s", "hits.tsv", "--include_trivial"] + TRAIN, 2),
])
def test_partitioned_driver_accepts(flags, argv, world):
    from pangnn_b200.dist_train import check_partition_flags
    check_partition_flags(flags(argv), world)


def test_main_refuses_under_torchrun_before_any_device_work(monkeypatch):
    """Every rank of ``torchrun --nproc-per-node 2 pangnn.py --train ...`` stops on the flags, before it touches a GPU
    or joins a process group (this box has neither)."""
    from pangnn_b200 import setup, train
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("LOCAL_RANK", "1")
    try:
        with pytest.raises(ValueError, match="whole_graph_training"):
            train.main(BASE + ["--train"])
    finally:
        setup.reset()
    assert not torch.distributed.is_initialized()


@pytest.mark.parametrize("names", [False, True])
def test_q_score_table_in_rank_ordered_pieces_equals_one_call(tmp_path, names):
    """Rank 0 writes the header and its rows, rank 1 appends its rows: the file is the one-call file, byte for byte."""
    from pangnn_b200.postprocessing import write_q_score_vs_logit
    rng = np.random.default_rng(0)
    E, N = 257, 60
    src = np.sort(rng.integers(0, N, E))
    ei = np.stack((src, rng.integers(0, N, E)))
    w = rng.random(E, dtype=np.float32)
    logits = (rng.standard_normal(E) * 3).astype(np.float32)
    y = rng.integers(0, 2, E).astype(np.float32)
    base = [rng.integers(0, 2, E) for _ in range(3)]
    gene = [f"g{i}_x" for i in range(N)] if names else None
    cols = lambda s: (ei[:, s], w[s], logits[s], y[s], gene, base[0][s], base[1][s], base[2][s])
    whole = str(tmp_path / "whole.csv")
    write_q_score_vs_logit(*cols(slice(None)), path=whole)
    parts = str(tmp_path / "parts.csv")
    cut = 100
    write_q_score_vs_logit(*cols(slice(0, cut)), path=parts, header=True)
    write_q_score_vs_logit(*cols(slice(cut, E)), path=parts, header=False, append=True)
    write_q_score_vs_logit(*cols(slice(E, E)), path=parts, header=False, append=True)   # a rank without edges
    assert open(parts, "rb").read() == open(whole, "rb").read()
