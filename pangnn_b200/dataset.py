"""``UnionGraphDataset`` — drop-in for ``src/dataset.py:16-555`` on the device preprocessing path.

Same constructor, same public attributes (``train`` / ``val`` / ``test`` lists of graphs,
``class_balance``, ``num_genes``, ``gene_str_ids_lst``, ``gene_id_position_dict``, ``base_labels``,
``base_labels_raw``), same graph attribute bag (``x, edge_index, edge_attr, y`` +
``neighbour_edge_index`` | ``union_edge_index``).  Where the reference keeps dict-of-dicts keyed by
gene-id strings (``sim_score_dict`` / ``sim_score_dict_raw``) this keeps arrays in node ids:
``sim_edges`` = ``(src, dst, w, y)`` sorted by (src, dst) and ``raw_hits`` = ``(q, t, bits)``.

Edge order inside every graph is the canonical (src, dst) order (the reference's is CPython set
order, SURVEY.md F10).
"""
import math
import random

import numpy as np
import torch

from . import ops
from . import preprocessing as pp
from . import simulate as sim
from . import subgraphs
from .data import Data
from .setup import args, log


class UnionGraphDataset:
    def __init__(self, gff_files=[], similarity_score_file="", ribap_groups_file=None,
                 split=(0.7, 0.15, 0.15), categorical_nodes=False, calculate_baseline=False,
                 device=None):
        self.device = torch.device(device if device is not None else "cuda")
        self.gene_str_ids_lst, self.gene_id_position_dict = [], {}
        self.data_lst, self.base_labels, self.base_labels_raw = [], [], []
        self.categorical_nodes, self.num_genes, self.split = categorical_nodes, 0, split
        self.val, self.train, self.test = [], [], []
        self.class_balance = None
        self.gff_is_subset = False
        self.calculate_baseline = calculate_baseline
        self.groups = []

        if not gff_files or args.simulate_dataset:
            if not args.simulate_dataset:
                log.info("No annotation files provided.")
                return
            n, G, frac, frags, shuf = args.simulate_dataset                      # src/dataset.py:64
            s = sim.simulate_hits(int(n), int(G), float(frac), frags, shuf,
                                  score_means=tuple(args.simulated_score_means), seed=args.seed)
            self.num_genes = s["num_genes"]
            self.genome_of, self.group_of = s["genome_of"], s["group_of"]
            self.raw_hits = (s["q"], s["t"], s["bits"])
            self.gene_str_ids_lst = None                                         # ids are positions
            order = np.argsort(self.group_of, kind="stable")
            self.groups = np.split(order, np.cumsum(np.bincount(self.group_of))[:-1])
            has_labels = True
        else:
            # input files parsed on the device (SURVEY §8f rank 2): GFF3 -> gene order + id hashes, hit table and RIBAP
            # table -> node ids through the sorted hash table; the host keeps the id strings for the output tables
            genome_names, genome_of, hashes = [], [], []
            on_device = torch.device(self.device).type == "cuda"
            for gi, f in enumerate(gff_files):                                   # src/dataset.py:77-96
                if on_device:
                    ids, h = pp.load_gff_device(f, device=self.device)
                    hashes.append(h)
                else:
                    ids = pp.load_gff(f)
                self.gene_str_ids_lst += ids
                genome_of += [gi] * len(ids)
                genome_names.append(pp.genome_name_of(f))
            self.num_genes = len(self.gene_str_ids_lst)
            self.gene_id_position_dict = {g: i for i, g in enumerate(self.gene_str_ids_lst)}
            # the reference derives the genome from the id prefix, not from the file (src/preprocessing.py:375)
            prefixes = {}
            self.genome_of = np.asarray([prefixes.setdefault(g.split("_")[0], len(prefixes))
                                         for g in self.gene_str_ids_lst], dtype=np.int32)
            has_labels = bool(ribap_groups_file)
            self.group_of = None
            if on_device:
                table = ops.gene_id_table_from_hashes(torch.cat(hashes), self.device)
                self.raw_hits = pp.load_similarity_score_device(similarity_score_file, None, table=table, device=self.device)
                if has_labels:
                    self.group_of, self.groups, self.gff_is_subset = pp.load_ribap_groups_device(
                        ribap_groups_file, genome_names, table, self.num_genes, device=self.device)
            else:                                   # host parsers: construction without a GPU (tests of the host logic)
                self.raw_hits = pp.load_similarity_score(similarity_score_file, self.gene_id_position_dict)
                if has_labels:
                    self.group_of, self.groups, self.gff_is_subset = pp.load_ribap_groups(
                        ribap_groups_file, genome_names, self.gene_id_position_dict)

        # ---- device: sort / dedupe / trivial filter / softmax + Q-score / labels  (a1-a7)
        src, dst, w, y = pp.normalize_sim_scores(*self.raw_hits, self.genome_of, self.group_of,
                                                 num_nodes=self.num_genes, device=self.device)
        # without a RIBAP table the normalisation writes zeros for y: they are not labels and go no further
        self.sim_edges = (src, dst, w, y if has_labels else None)
        self.has_labels = has_labels

        if args.train:
            self.data_lst, self.class_balance = self.generate_sub_graphs(self.groups)
            self.split_data(split, args.batch_size)
            if args.simulate_dataset:
                self.test = [self.generate_graphs()]
        else:
            self.test = [self.generate_graphs()]

    # ------------------------------------------------------------------------------------------
    def generate_graphs(self):
        """Whole graph (``src/dataset.py:325-395``): sim edges + Q-score weights + labels, the
        +-n neighbour band (self loops, crossing genome seams), optional union assembly
        ``[sim ; nb]`` with weights ``[w ; 1...]``.  Without labels (no RIBAP table; the reference crashes at
        ``src/dataset.py:345``) the graph is the same with ``y = None`` and ``class_balance`` stays None."""
        src, dst, w, y = self.sim_edges
        dev = self.device
        N, n = self.num_genes, args.neighbours
        edge_index = torch.stack((src.long(), dst.long()))
        if y is not None:
            pos = y.sum()
            self.class_balance = ((y == 0).sum() / pos).item()                   # src/dataset.py:346
        x = torch.ones(N, device=dev) if self.categorical_nodes else torch.ones(N, 1, device=dev)
        if args.union_edge_weights:
            union = ops.union_index(edge_index, N, n)                            # band written into the tail
            g = Data(x, edge_index, ops.union_weights(w, union.size(1)), y)
            g.union_edge_index = union
        else:
            g = Data(x, edge_index, w, y)
            g.neighbour_edge_index = pp.neighbour_band(N, n, dev)
        if self.categorical_nodes:
            g.node_id = torch.arange(N, device=dev)
        if self.calculate_baseline:
            genome_d = torch.as_tensor(self.genome_of, device=dev)
            self.base_labels = pp.baseline_labels(src, dst, w, genome_d).tolist()
            self.base_labels_raw = self.raw_baseline_labels(self.raw_hits, src, dst, genome_d, N).tolist()
        return g

    @classmethod
    def raw_baseline_labels(cls, raw_hits, src, dst, genome_d, num_genes):
        """Raw baseline of the edges ``(src, dst)``: the max-candidate labels of the raw hit table incl. self hits
        (``src/helper.py:470-475``) after the same sort, dedupe and trivial-case filter as the graph.  Every
        (query, target genome) segment of the queries in ``src`` must be complete in ``raw_hits``."""
        q, t, b = (torch.as_tensor(a, device=src.device) for a in raw_hits)
        qs, ts, bs = ops.hits_sort_unique(q, t, b, num_genes)
        if not args.include_trivial:
            keep = cls._trivial_keep(qs, ts, genome_d)
            qs, ts, bs = qs[keep], ts[keep], bs[keep]
        raw = pp.baseline_labels(qs, ts, bs, genome_d)
        key_raw = qs.long() * num_genes + ts.long()
        return raw[torch.searchsorted(key_raw, src.long() * num_genes + dst.long())]

    @staticmethod
    def _trivial_keep(q, t, genome_of):
        g = genome_of.long()[t.long()]
        key = q.long() * (int(genome_of.max().item()) + 1) + g
        _, inv, cnt = torch.unique(key, return_inverse=True, return_counts=True)
        return cnt[inv] > 1

    # ------------------------------------------------------------------------------------------
    def generate_sub_graphs(self, groups):
        """One n-hop sub-graph per ortholog group (``src/dataset.py:222-322`` with ``get_connected_nodes`` /
        ``get_neighbour_graph`` of ``src/helper.py:327-417``), all groups at once on the device
        (``pangnn_b200.subgraphs.extract``).  -> (list-of-graphs view over the packed arena, class balance)."""
        src, dst, w, y = self.sim_edges
        if y is None:
            raise ValueError("training sub-graphs need labels: name the RIBAP groups table with -r")
        arena = subgraphs.extract(src, dst, w, y, self.num_genes, args.neighbours, groups,
                                  union=bool(args.union_edge_weights), gff_is_subset=self.gff_is_subset,
                                  chunks=args.cpus)
        return subgraphs.GraphList(arena, np.arange(arena.num_graphs)), arena.class_balance

    def split_data(self, split=(0.7, 0.15, 0.05), batch_size=32):
        """``src/dataset.py:172-213`` incl. its quirk: ``data[-int(len*split[2]):]`` is ALL graphs
        when there are fewer than ``1/split[2]`` of them."""
        n_train = int(len(self.data_lst) * split[0])
        n_val = int(len(self.data_lst) * split[1])
        n_test = int(len(self.data_lst) * split[2])
        order = list(range(len(self.data_lst)))              # the same permutation as shuffling the list itself
        random.Random(args.seed).shuffle(order)
        self.data_lst = self.data_lst[order] if hasattr(self.data_lst, "arena") else [self.data_lst[i] for i in order]
        log.info(f"Splitting data ({len(self.data_lst)}) into sets of train: {n_train}, test: {n_test}, val: {n_val} graphs.")
        self.train = self.data_lst[:n_train]
        self.val = self.data_lst[n_train:n_train + n_val]
        self.test = self.data_lst[-n_test:]

    def get(self, idx):
        return self.data_lst[idx]

    def len(self):
        return len(self.data_lst)
