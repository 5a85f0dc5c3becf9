"""Output side of the path (SURVEY.md §8f rank 4; ``src/postprocessing.py:5-36``): ortholog groups from the
model's predictions = connected components of the edges predicted positive, computed on the device
(``ops.connected_components``), and the group table the reference calls ``holiest_of_all_tables.csv``.

The reference's ``write_groups_file`` is unused and does not merge sets as written (every pair is appended
again after the scan); the behaviour here is the intended one, one line per group of at least two genes."""
import os

import torch

from . import ops


def ortholog_groups(edge_index, binary_prediction, num_genes):
    """-> (labels [N] int32: smallest gene id of the gene's group, groups: list of gene-id lists with >= 2 genes,
    ordered by smallest id)."""
    labels = ops.connected_components(edge_index[0], edge_index[1], num_genes, select=binary_prediction)
    order = torch.argsort(labels.long(), stable=True)
    sl = labels[order]
    head = torch.ones_like(sl, dtype=torch.bool)
    head[1:] = sl[1:] != sl[:-1]
    starts = torch.nonzero(head).squeeze(1)
    sizes = torch.diff(torch.cat((starts, starts.new_tensor([sl.numel()]))))
    keep = sizes > 1
    order_h, starts_h, sizes_h = order.cpu().tolist(), starts[keep].cpu().tolist(), sizes[keep].cpu().tolist()
    return labels, [order_h[a:a + n] for a, n in zip(starts_h, sizes_h)]


def write_groups_file(groups, gene_ids_lst=None, path=os.path.join("data", "holiest_of_all_tables.csv")):
    """``group_<i>, gene, gene, ...`` per line (``src/postprocessing.py:31-36``; ids are positions when the
    dataset has no string ids, as for simulated data)."""
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    with open(path, "w") as f:
        for i, grp in enumerate(groups):
            names = [gene_ids_lst[g] if gene_ids_lst is not None else str(g) for g in grp]
            f.write(f"group_{i}, {', '.join(names)}\n")
    return path


Q_SCORE_VS_LOGIT_COLUMNS = ("source_int_id", "target_int_id", "source_str_id", "target_str_id", "score", "logit", "homolog",
                            "q_score_baseline", "raw_baseline", "logit_baseline")


def write_q_score_vs_logit(edge_index, edge_attr, logits, labels, gene_lst=None, base_labels=None, base_labels_raw=None,
                           logit_baseline=None, path="q_score_vs_logit.csv", header=True, append=False):
    """The reference's only per-edge output table (``src/plot.py:473-504``, written from ``src/predict.py:88``):
    one row per SCORED edge, keyed by (source, target), with the input Q-score (``edge_attr[:E]`` — the literal
    slice of ``src/plot.py:456``), the output logit, the label and the three max-candidate baselines.  Same
    columns, order, dtypes (score / logit float64, homolog int64) and text format as ``DataFrame.to_csv(index=False)``.
    Tensors may live on the device; one D2H copy per column, rows formatted by pandas' C writer.  A column passed as
    None is written as -1 on every row: an absent baseline, or ``labels`` of a run without labels (``-r ''``).

    A table can be written in consecutive pieces: the first call with ``header=True``, the others with
    ``header=False, append=True``; the file is byte for byte the one a single call on the whole table writes."""
    import numpy as np
    import pandas as pd

    def host(t, dtype):
        if t is None:
            return None
        if torch.is_tensor(t):
            t = t.detach().cpu().numpy()
        return np.asarray(t).astype(dtype)
    E = int(logits.numel() if torch.is_tensor(logits) else len(logits))
    src, dst = host(edge_index[0], np.int64)[:E], host(edge_index[1], np.int64)[:E]
    cols = {"source_int_id": src, "target_int_id": dst}
    if gene_lst is not None:
        names = np.asarray(gene_lst, dtype=object)
        cols["source_str_id"], cols["target_str_id"] = names[src], names[dst]
    else:                                                                  # simulated data: ids are positions
        cols["source_str_id"], cols["target_str_id"] = src.astype(str), dst.astype(str)
    cols["score"] = host(edge_attr, np.float32)[:E].astype(np.float64)     # float32 values widened, as .tolist() does
    cols["logit"] = host(logits, np.float32).astype(np.float64)
    cols["homolog"] = (host(labels, np.float32)[:E].astype(np.int64) if labels is not None
                       else np.full(E, -1, dtype=np.int64))
    for name, v in (("q_score_baseline", base_labels), ("raw_baseline", base_labels_raw), ("logit_baseline", logit_baseline)):
        cols[name] = host(v, np.int64) if v is not None else np.full(E, -1, dtype=np.int64)
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    pd.DataFrame(cols)[list(Q_SCORE_VS_LOGIT_COLUMNS)].to_csv(path, index=False, header=header,
                                                              mode="a" if append else "w")
    return path
