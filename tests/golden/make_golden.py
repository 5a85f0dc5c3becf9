#!/usr/bin/env python3
"""Mint golden vectors by running the UNMODIFIED reference (``/root/reference/src``) under the
import shim in ``oracle/ref_shim.py``.  Build-container only (needs ``/root/reference``).

    python tests/golden/make_golden.py            # all cases, one subprocess each
    python tests/golden/make_golden.py --case c1  # a single case, in this process

Each case freezes the INPUTS the reference saw (hit table in node ids, genome / group maps) and
the OUTPUTS it produced (normalised weights, edge index, labels, neighbour graph, baselines,
model logits / loss / gradients for a seeded state dict) into ``tests/golden/<case>.npz``.
Edge lists are stored canonicalised by ``(src, dst)`` because the reference's own order is
CPython set order (SURVEY.md F10).  Seeds: PYTHONHASHSEED=0, random/numpy/torch seed 0.
"""
import argparse
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

DUMMY = ["-a", "data/dummy_dataset/dummy1.gff", "data/dummy_dataset/dummy2.gff",
         "-s", "data/dummy_dataset/dummy_mmseqs2.csv",
         "-r", "data/dummy_dataset/dummy_ribap.csv", "--include_trivial"]

CASES = {
    # name: (reference argv, model-flag variants to run on the whole graph)
    "minimal": ([], ["base", "default"]),
    "dummy": (DUMMY, ["default", "base", "union_skip"]),
    "c1": ([], ["default", "base", "union_skip", "cosine", "union_n4"]),
    # the committed excerpts of the bundled files (tests/golden/make_parser_fixtures.py): pins the real-data path
    # from the raw GFF3 / MMseqs2 / RIBAP bytes (device parsers) to the graph
    "c1_excerpt": (["-a", os.path.join(HERE, "parsers", "Cga_08-1274-3_RENAMED.gff"),
                    os.path.join(HERE, "parsers", "Cga_12-4358_RENAMED.gff"),
                    "-s", os.path.join(HERE, "parsers", "hits.tsv"), "-r", os.path.join(HERE, "parsers", "ribap.csv")],
                   ["default"]),
    "c1_sub": (["--train", "-@", "2"], []),
    "c2": (["--simulate_dataset", "10000", "2", "0.5", "10", "3"], ["default", "union_skip"]),
    "sim5": (["--simulate_dataset", "300", "5", "0.5", "10", "3"], ["default", "union_skip", "union_n4"]),
    "sim5_trivial": (["--simulate_dataset", "200", "4", "0.3", "10", "3", "--include_trivial"], ["default"]),
    "sim5_sub": (["--simulate_dataset", "60", "3", "0.5", "6", "2", "--train", "-@", "2", "-n", "2"], []),
    "trivial_c1": (["--include_trivial"], []),
    "trivial_sim": (["--simulate_dataset", "150", "4", "0.4", "10", "3", "--include_trivial"], []),
}

VARIANTS = {
    "default": dict(),
    "base": dict(base_model=True),
    "union_skip": dict(union_edge_weights=True, neighbours=3, skip_connections=True),
    "union_n4": dict(union_edge_weights=True, neighbours=4),
    "cosine": dict(decoder="cosine"),
}


def seed_all():
    import random
    import numpy as np
    import torch
    random.seed(0); np.random.seed(0); torch.manual_seed(0)


def hits_of(sim_dict, gene_pos):
    from oracle.preprocess import dict_to_hits
    return dict_to_hits(sim_dict, gene_pos)


def canon(ei, *vals):
    import numpy as np
    src, dst = np.asarray(ei[0], dtype=np.int64), np.asarray(ei[1], dtype=np.int64)
    order = np.lexsort((dst, src))
    return (np.stack((src[order], dst[order])),) + tuple(np.asarray(v)[order] for v in vals)


def run_model(ref, graph, variant, num_nodes, out, prefix):
    """Reference AlternateGCN (src/gnn.py) over the restated GCNConv; seeded state dict."""
    import numpy as np
    import torch
    args = ref.args
    saved = {k: getattr(args, k) for k in ("union_edge_weights", "base_model", "skip_connections",
                                           "decoder", "neighbours")}
    for k, v in VARIANTS[variant].items():
        setattr(args, k, v)
    try:
        from oracle.params import make_state_dict
        model = ref.gnn.AlternateGCN(device="cpu", dataset=None, categorical_nodes=False,
                                     dims=[args.node_dim, args.hidden_dim])
        # strict load: proves the key names / shapes of oracle/params.py match src/gnn.py
        model.load_state_dict(make_state_dict(args.node_dim, args.hidden_dim,
                                              args.skip_connections, seed=1234), strict=True)
        y = graph.y
        pw = float((y == 0).sum() / y.sum())
        logits = model(graph)
        loss = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(pw))(logits, y)
        loss.backward()
        out[f"{prefix}/pos_weight"] = np.float64(pw)
        out[f"{prefix}/logits"] = logits.detach().numpy()
        out[f"{prefix}/loss"] = np.float64(loss.item())
        out[f"{prefix}/state_dict_keys"] = np.asarray(",".join(model.state_dict().keys()))
        for k, p in model.named_parameters():
            if p.grad is not None:
                out[f"{prefix}/grad/{k}"] = p.grad.numpy().copy()
    finally:
        for k, v in saved.items():
            setattr(args, k, v)


def whole_graph_case(ref, name, variants, out):
    """Run UnionGraphDataset in inference mode (whole graph, src/dataset.py:163-166,325-395)."""
    import numpy as np
    import torch
    args = ref.args
    UGD = ref.dataset.UnionGraphDataset
    if args.simulate_dataset:
        ds = UGD(calculate_baseline=True, split=(0.7, 0.15, 0.01), categorical_nodes=False)
    else:
        ds = UGD(args.annotation, args.similarity, args.ribap_groups, split=(0.7, 0.15, 0.01),
                 categorical_nodes=False, calculate_baseline=True)
    genes = ds.gene_str_ids_lst
    gene_pos = ds.gene_id_position_dict
    N = len(genes)
    prefixes = sorted({g.split("_")[0] for g in genes}, key=lambda p: next(i for i, g in enumerate(genes) if g.startswith(p)))
    genome_of = np.asarray([prefixes.index(g.split("_")[0]) for g in genes], dtype=np.int64)
    group_of = np.full(N, -1, dtype=np.int64)
    gid = {}
    for g, others in ds.ribap_groups_dict.items():
        if g not in gene_pos:
            continue
        key = frozenset([g] + list(others))
        group_of[gene_pos[g]] = gid.setdefault(key, len(gid))
    out["num_genes"] = np.int64(ds.num_genes)
    out["genome_of"] = genome_of
    out["group_of"] = group_of
    out["neighbours"] = np.int64(args.neighbours)
    # INPUT: raw hit table after the trivial-case filter (what normalize_sim_scores consumed)
    q, t, b = hits_of(ds.sim_score_dict_raw, gene_pos)
    out["raw/q"], out["raw/t"], out["raw/bits"] = q, t, b
    # OUTPUT of normalisation, canonical
    nq, nt, nw = hits_of(ds.sim_score_dict, gene_pos)
    ei, w64 = canon((nq, nt), nw)
    out["norm/edge_index"], out["norm/w64"] = ei, w64
    # OUTPUT whole graph
    g = ds.test[0]
    gei, gw, gy, bl, blr = canon(g.edge_index.numpy(), g.edge_attr.numpy(), g.y.numpy(),
                                 np.asarray(ds.base_labels), np.asarray(ds.base_labels_raw))
    out["graph/edge_index"], out["graph/edge_attr"], out["graph/y"] = gei, gw, gy
    out["graph/base_labels"], out["graph/base_labels_raw"] = bl, blr
    out["graph/neighbour_edge_index"] = g.neighbour_edge_index.numpy()
    out["graph/class_balance"] = np.float64(float(ds.class_balance))
    out["graph/x"] = g.x.numpy()

    # model variants on the canonical graph (so per-edge outputs line up with the fixture)
    def build(variant):
        v = VARIANTS[variant]
        saved = (args.union_edge_weights, args.neighbours)
        args.union_edge_weights = v.get("union_edge_weights", False)
        args.neighbours = v.get("neighbours", saved[1])
        try:
            gg = ds.generate_graphs()
        finally:
            args.union_edge_weights, args.neighbours = saved
        return gg

    for variant in variants:
        gg = build(variant)
        order = np.lexsort((gg.edge_index[1].numpy(), gg.edge_index[0].numpy()))
        E = gg.edge_index.shape[1]
        o = torch.from_numpy(order)
        gg.edge_index = gg.edge_index[:, o]
        gg.y = gg.y[o]
        if hasattr(gg, "union_edge_index"):
            # whole graph union = [sim ; nb] (src/dataset.py:374-376): permute the sim prefix only
            full = torch.cat((o, torch.arange(E, gg.union_edge_index.shape[1])))
            gg.union_edge_index = gg.union_edge_index[:, full]
            gg.edge_attr = gg.edge_attr[full].float()
            out[f"model/{variant}/union_edge_index"] = gg.union_edge_index.numpy()
            out[f"model/{variant}/edge_attr"] = gg.edge_attr.numpy()
        else:
            gg.edge_attr = gg.edge_attr[o]
            out[f"model/{variant}/neighbour_edge_index"] = gg.neighbour_edge_index.numpy()
        run_model(ref, gg, variant, N, out, f"model/{variant}")


def minimal_case(ref, variants, out):
    import numpy as np
    g = ref.helper.generate_minimal_dataset()            # src/helper.py:149-172
    out["graph/x"] = g.x.numpy()
    out["graph/edge_index"] = g.edge_index.numpy()
    out["graph/edge_attr"] = g.edge_attr.numpy()
    out["graph/y"] = g.y.numpy()
    out["graph/union_edge_index"] = g.union_edge_index.numpy()
    E = g.edge_index.shape[1]
    # the literal fixture has no neighbour graph: use the non-sim tail of its union index
    g.neighbour_edge_index = g.union_edge_index[:, E:]
    out["graph/neighbour_edge_index"] = g.neighbour_edge_index.numpy()
    for variant in variants:
        run_model(ref, g, variant, 12, out, f"model/{variant}")


def sub_graph_case(ref, out):
    """Training-mode sub-graphs (src/dataset.py:222-322), stored in GLOBAL node ids."""
    import numpy as np
    args = ref.args
    UGD = ref.dataset.UnionGraphDataset
    if args.simulate_dataset:
        ds = UGD(calculate_baseline=True, split=(0.7, 0.15, 0.01), categorical_nodes=False)
    else:
        ds = UGD(args.annotation, args.similarity, args.ribap_groups, split=(0.7, 0.15, 0.01),
                 categorical_nodes=False, calculate_baseline=True)
    gene_pos = ds.gene_id_position_dict
    genes = ds.gene_str_ids_lst
    N = len(genes)
    prefixes = []
    for gname in genes:
        p = gname.split("_")[0]
        if p not in prefixes:
            prefixes.append(p)
    out["genome_of"] = np.asarray([prefixes.index(g.split("_")[0]) for g in genes], dtype=np.int64)
    group_of = np.full(N, -1, dtype=np.int64)
    gid = {}
    for g, others in ds.ribap_groups_dict.items():
        if g in gene_pos:
            group_of[gene_pos[g]] = gid.setdefault(frozenset([g] + list(others)), len(gid))
    out["group_of"] = group_of
    out["num_genes"] = np.int64(N)
    out["neighbours"] = np.int64(args.neighbours)
    nq, nt, nw = hits_of(ds.sim_score_dict, gene_pos)
    ei, w64 = canon((nq, nt), nw)
    out["norm/edge_index"], out["norm/w64"] = ei, w64
    # the split shuffles and deletes gene_lst from train/val graphs (src/dataset.py:199-205);
    # re-generate the sub-graphs deterministically from the same group list instead
    import pandas as pd  # noqa: F401
    if args.simulate_dataset:
        groups = [list(g) for g in zip(*[[x for x in genes if x.startswith(p)] for p in prefixes])]
        # simulated groups are "gene p of every genome" BEFORE the synteny shuffle
        by_num = {}
        for gname in genes:
            by_num.setdefault(gname.split("_")[1], []).append(gname)
        groups = [sorted(v) for _, v in sorted(by_num.items())]
    else:
        _, groups, _ = ref.preprocessing.load_ribap_groups(
            args.ribap_groups,
            [os.path.basename(f).rsplit(".", 1)[0].replace("_RENAMED", "") for f in args.annotation])
    data_lst, _, base, base_raw = ds.generate_sub_graphs(groups)
    kept = [g for g in groups if len(g) > 1]
    out["num_sub_graphs"] = np.int64(len(data_lst))
    node_ptr, sim_ptr, nb_ptr = [0], [0], [0]
    nodes, sim_src, sim_dst, sim_w, sim_y, nb_src, nb_dst = [], [], [], [], [], [], []
    seeds, seed_ptr = [], [0]
    gi = 0
    for grp in kept:
        if gi >= len(data_lst):
            break
        d = data_lst[gi]
        if not set(grp).issubset(d.gene_lst):
            continue
        gi += 1
        loc2glob = np.asarray([gene_pos[s] for s in d.gene_lst], dtype=np.int64)
        nodes.append(loc2glob); node_ptr.append(node_ptr[-1] + loc2glob.size)
        seeds.append(np.asarray([gene_pos[s] for s in grp], dtype=np.int64))
        seed_ptr.append(seed_ptr[-1] + len(grp))
        s, t = loc2glob[d.edge_index[0].numpy()], loc2glob[d.edge_index[1].numpy()]
        ce, cw, cy = canon((s, t), d.edge_attr.numpy(), d.y.numpy())
        sim_src.append(ce[0]); sim_dst.append(ce[1]); sim_w.append(cw); sim_y.append(cy)
        sim_ptr.append(sim_ptr[-1] + s.size)
        ns, nt_ = loc2glob[d.neighbour_edge_index[0].numpy()], loc2glob[d.neighbour_edge_index[1].numpy()]
        (cn,) = canon((ns, nt_))
        nb_src.append(cn[0]); nb_dst.append(cn[1]); nb_ptr.append(nb_ptr[-1] + ns.size)
    assert gi == len(data_lst), (gi, len(data_lst))
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    out["sub/node_ptr"] = np.asarray(node_ptr); out["sub/nodes"] = cat(nodes, np.int64)
    out["sub/seed_ptr"] = np.asarray(seed_ptr); out["sub/seeds"] = cat(seeds, np.int64)
    out["sub/sim_ptr"] = np.asarray(sim_ptr)
    out["sub/sim_src"], out["sub/sim_dst"] = cat(sim_src, np.int64), cat(sim_dst, np.int64)
    out["sub/sim_w"], out["sub/sim_y"] = cat(sim_w, np.float32), cat(sim_y, np.float32)
    out["sub/nb_ptr"] = np.asarray(nb_ptr)
    out["sub/nb_src"], out["sub/nb_dst"] = cat(nb_src, np.int64), cat(nb_dst, np.int64)


def trivial_case(ref, out):
    """a1 in isolation: the unfiltered dict and what ``remove_trivial_cases`` makes of it
    (src/preprocessing.py:370-385), for real data (incl. self hits, min-centred scores) and for
    simulated data."""
    import numpy as np
    args = ref.args
    if args.simulate_dataset:
        n, G, f = args.simulate_dataset[:3]
        _, by_genome = ref.simulate.simulate_gene_ids(int(n), int(G))
        raw, _, _ = ref.simulate.simulate_similarity_scores_and_ribap_dict(by_genome, f)
        genes = [x for xs in by_genome for x in xs]
    else:
        genes = []
        for f in args.annotation:
            genes += list(ref.preprocessing.load_gff(f).index)
        raw = ref.preprocessing.load_similarity_score(args.similarity, {g: i for i, g in enumerate(genes)})
    gene_pos = {g: i for i, g in enumerate(genes)}
    prefixes = []
    for g in genes:
        if g.split("_")[0] not in prefixes:
            prefixes.append(g.split("_")[0])
    out["genome_of"] = np.asarray([prefixes.index(g.split("_")[0]) for g in genes], dtype=np.int64)
    out["unfiltered/q"], out["unfiltered/t"], out["unfiltered/bits"] = hits_of(raw, gene_pos)
    filt = ref.preprocessing.remove_trivial_cases(raw)
    fq, ft, fb = hits_of(filt, gene_pos)
    ei, b = canon((fq, ft), fb)
    out["filtered/edge_index"], out["filtered/bits"] = ei, b


def save_npz(path, arrays):
    """``np.savez_compressed`` with LZMA instead of deflate: ``np.load`` reads it unchanged (through ``zipfile``) and the
    largest case (c2) stays under 1 MB (deflate: 1.36 MB)."""
    import io
    import zipfile
    import numpy as np
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(v), allow_pickle=False)
            zf.writestr(f"{k}.npy", buf.getvalue())


def run_case(name):
    import numpy as np
    from oracle import ref_shim
    argv, variants = CASES[name]
    work = tempfile.mkdtemp(prefix=f"pangnn_golden_{name}_")
    ref = ref_shim.load_reference(argv, work)
    seed_all()
    out = {}
    if name == "minimal":
        minimal_case(ref, variants, out)
    elif name.endswith("_sub"):
        sub_graph_case(ref, out)
    elif name.startswith("trivial_"):
        trivial_case(ref, out)
    else:
        whole_graph_case(ref, name, variants, out)
    out["argv"] = np.asarray(" ".join(argv))
    path = os.path.join(HERE, f"{name}.npz")
    save_npz(path, out)
    print(f"[golden] {name}: {len(out)} arrays -> {path} ({os.path.getsize(path)/1024:.0f} KiB)")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default=None)
    a = ap.parse_args()
    if a.case:
        run_case(a.case)
    else:
        env = dict(os.environ, PYTHONHASHSEED="0")
        for c in CASES:
            subprocess.run([sys.executable, os.path.abspath(__file__), "--case", c], check=True, env=env)


# tests/golden/params_seed1234.npz — the seeded AlternateGCN state dicts (oracle/params.py, seed 1234, with and
# without --skip_connections) every model golden above was minted with, frozen so that bench.py's multi-GPU
# parity gate (tools/parity_gate.py) can load them without importing oracle/:
#   python - <<'PY'
#   import numpy as np; from oracle.params import make_state_dict
#   np.savez_compressed("tests/golden/params_seed1234.npz", **{f"skip{int(s)}/{k}": v.numpy()
#       for s in (False, True) for k, v in make_state_dict(64, 128, s, seed=1234).items()})
#   PY
