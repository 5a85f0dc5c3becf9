"""Flag surface of the reference CLI (``src/setup.py:15-50``) — same names, defaults and types.

The reference parses ``sys.argv`` at import time and every module reads the resulting global
``args`` (also inside ``AlternateGCN.forward``, ``src/gnn.py:128,132,143,171-172``).  Here the
parser is built at import but only *applied* by ``parse(argv)`` (the CLI calls it); library users
and tests mutate ``args`` in place.
"""
import argparse
import logging
import os


def build_parser():
    p = argparse.ArgumentParser(prog="pangnn.py", formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                description="panGNN on B200: drop-in CLI for the reference's flags.")
    p.add_argument("-d", "--debug", action="store_true")
    p.add_argument("-p", "--plot_graph", action="store_true")
    p.add_argument("-t", "--traceback", action="store_true")
    p.add_argument("-c", "--cache", action="store_true")
    p.add_argument("-l", "--log_level", default="INFO", type=str)
    p.add_argument("-m", "--model_args", default="model.pkl", type=str)
    p.add_argument("-n", "--neighbours", default=1, type=int)
    p.add_argument("-a", "--annotation", type=str, nargs="*",
                   default=[os.path.join("data", "Cga_08-1274-3_RENAMED.gff"),
                            os.path.join("data", "Cga_12-4358_RENAMED.gff")])
    p.add_argument("-s", "--similarity", default=os.path.join("data", "mmseq2_result.csv"), type=str)
    p.add_argument("--binary_threshold", default=0.5, type=float)
    p.add_argument("--dynamic_binary_threshold", action="store_true")
    p.add_argument("--simulate_dataset", nargs=5, type=str, default=None)
    p.add_argument("--simulated_score_means", nargs=2, type=int, default=[200, 500])
    p.add_argument("--union_edge_weights", action="store_true")
    p.add_argument("--include_trivial", action="store_true")
    p.add_argument("--skip_connections", action="store_true")
    p.add_argument("--categorical_node", action="store_true")
    p.add_argument("--no_q_score_transform", action="store_false")
    p.add_argument("--normalization_temp", default=0.8, type=float)
    p.add_argument("--tb_comment", default="")
    p.add_argument("--from_pickle", default="")
    p.add_argument("--to_pickle", default="")
    p.add_argument("--fix_dataset", default=[], type=str, nargs="*")
    p.add_argument("--node_dim", default=64, type=int)
    p.add_argument("--hidden_dim", default=128, type=int)
    p.add_argument("--decoder", default="mlp", type=str)
    p.add_argument("--base_model", action="store_true")
    p.add_argument("-o", "--output", default="runs", type=str)
    p.add_argument("--train", action="store_true")
    p.add_argument("-b", "--batch_size", default=32, type=int)
    p.add_argument("-e", "--epochs", default=10, type=int)
    p.add_argument("-r", "--ribap_groups", default=os.path.join("data", "holy_python_ribap_95.csv"), type=str)
    p.add_argument("-@", "--cpus", default=2, type=int)
    p.add_argument("--mixed_precision", default="no", type=str)
    # additions of this implementation (not in the reference)
    p.add_argument("--cuda_graphs", action="store_true",
                   help="(new) training: replay every batch's step as one CUDA graph per size bucket "
                        "(pangnn_b200.graphs.GraphedBatchStep; batches over 4096 edges per list stay eager)")
    p.add_argument("--whole_graph_training", action="store_true",
                   help="train on the whole graph as one batch instead of per-group sub-graphs")
    p.add_argument("--data_parallel", action="store_true",
                   help="(new) with --train under torchrun: replicate the model, shard the sub-graph batches, average "
                        "gradients each step (pangnn_b200.dist_train.run_data_parallel)")
    p.add_argument("--edge_split", nargs=2, type=float, default=None, metavar=("VAL", "TEST"),
                   help="(new) with --whole_graph_training: hold out these fractions of the scored edges (by unordered "
                        "gene pair, from --seed) as validation and test edges; they stay in message passing, only "
                        "their labels are hidden from training (pangnn_b200.edge_split)")
    p.add_argument("--seed", default=0, type=int)
    return p


parser = build_parser()
args = parser.parse_args([])           # defaults; mutated in place by parse()
log = logging.getLogger("pangnn")


def _post(ns):
    if ns.simulate_dataset is not None and isinstance(ns.simulate_dataset[0], str):
        s = ns.simulate_dataset                      # src/setup.py:54-56
        ns.simulate_dataset = [int(s[0]), int(s[1]), float(s[2]), float(s[3]), float(s[4])]
    return ns


# Flags of the reference CLI that are accepted for command-line compatibility but select nothing on this path
# (reporting, pickling, plotting, Accelerate's autocast — DESIGN.md §7); setting one is reported, not ignored silently.
_INERT = {"plot_graph": False, "cache": False, "tb_comment": "", "from_pickle": "", "to_pickle": "",
          "fix_dataset": [], "mixed_precision": "no"}


def inert_flags(ns):
    return [k for k, default in _INERT.items() if getattr(ns, k, default) != default]


def has_labels(ns):
    """Whether the run's edges have labels: simulated data always has them; with input files ``-r ''`` names no RIBAP
    table, for inference on genomes whose ortholog groups are not known yet."""
    return bool(ns.simulate_dataset) or bool(ns.ribap_groups)


def check_label_flags(ns):
    """Raise ``ValueError`` when the flags ask for training without labels.  Depends on the flags alone, so every rank
    of a multi-GPU run refuses alike, before any device work."""
    if ns.train and not has_labels(ns):
        raise ValueError("--train needs labels: name the RIBAP groups table with -r (-r '' runs inference only)")


def parse(argv=None):
    """Parse ``argv`` INTO the module-global ``args`` (so every importer sees the same object)."""
    ns = _post(parser.parse_args(argv))
    args.__dict__.update(ns.__dict__)
    logging.basicConfig(level="DEBUG" if args.debug else args.log_level, format="%(message)s")
    for k in inert_flags(args):
        log.warning(f"--{k} is accepted for compatibility with the reference CLI but has no effect here "
                    f"(fp32 compute, no pickling / plotting / TensorBoard: DESIGN.md section 7)")
    return args


def reset():
    args.__dict__.update(parser.parse_args([]).__dict__)
    return args
