"""Shared helpers for the parity tests."""
import ctypes as C
from contextlib import contextmanager
from types import SimpleNamespace

import numpy as np
import torch

from oracle.model import AlternateGCN as OracleGCN, Flags
from oracle.params import make_state_dict

VARIANT_FLAGS = {
    "default": dict(),
    "base": dict(base_model=True),
    "union_skip": dict(union_edge_weights=True, neighbours=3, skip_connections=True),
    "union_n4": dict(union_edge_weights=True, neighbours=4),
    "cosine": dict(decoder="cosine"),
}


def golden_graph(g, variant, device="cpu"):
    """Rebuild the graph object the golden model variant ran on."""
    t = lambda a, dt=None: torch.as_tensor(np.asarray(a), dtype=dt, device=device)
    graph = SimpleNamespace()
    graph.x = t(g["graph/x"], torch.float32)
    graph.edge_index = t(g["graph/edge_index"], torch.long)
    graph.y = t(g["graph/y"], torch.float32)
    key = f"model/{variant}"
    if f"{key}/union_edge_index" in g.files:
        graph.union_edge_index = t(g[f"{key}/union_edge_index"], torch.long)
        graph.edge_attr = t(g[f"{key}/edge_attr"], torch.float32)
    else:
        graph.edge_attr = t(g["graph/edge_attr"], torch.float32)
        nb = f"{key}/neighbour_edge_index"
        graph.neighbour_edge_index = t(g[nb] if nb in g.files else g["graph/neighbour_edge_index"],
                                       torch.long)
    return graph


def oracle_model(variant, seed=1234, **kw):
    flags = Flags(**VARIANT_FLAGS[variant], **kw)
    m = OracleGCN(flags)
    m.load_state_dict(make_state_dict(flags.node_dim, flags.hidden_dim, flags.skip_connections,
                                      seed=seed), strict=True)
    return m, flags


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny): the 1e-5 'relative (fp32)' bar of BASELINE.json is applied to
    the tensor's scale, since individual elements can be arbitrarily close to zero."""
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    scale = max(float(np.abs(b).max()) if b.size else 0.0, 1e-30)
    return float(np.abs(a - b).max() / scale) if b.size else 0.0


def assert_close(name, got, ref, tol):
    """Compact failure message (never dumps the arrays)."""
    err = rel_err(got, ref)
    if not err < tol:
        raise AssertionError(f"{name}: rel_err {err:.3e} >= {tol:.1e} (shape {np.shape(ref)})")


# Parameter / input gradients are long fp32 reductions (over all nodes / edges) of terms that cancel,
# and they pass through ReLU / ELU kinks where a last-ulp difference in a pre-activation legitimately
# flips a derivative.  The 1e-5 bar of BASELINE.json is stated for embeddings, probabilities and
# loss; gradients are held to 1e-4 of the tensor's scale against the fp32 reference.
GRAD_TOL = 1e-4


# ------------------------------------------------------------------------------------------------
# per-kernel fp64 suites (test_gpu_node_kernels_fp64.py, test_gpu_edge_kernels_fp64.py)
# ------------------------------------------------------------------------------------------------
def lib():
    from pangnn_b200 import _abi
    return _abi.load()


def ptr(t):
    """Device pointer of ``t``; NULL for None and for an empty tensor."""
    return C.c_void_p(t.data_ptr() if t is not None and t.numel() else 0)


def check(rc, what):
    from pangnn_b200 import _abi
    _abi.check(rc, what)


def nan_fill(*shape, device="cuda:0"):
    """fp32 buffer of quiet NaNs with distinct payloads: a stray store, or a lost one, shows bit for bit."""
    n = 1
    for s in shape:
        n *= s
    bits = (torch.arange(n, device=device, dtype=torch.int64) % 0x3FFFFF + 0x7FC00001).to(torch.int32)
    return bits.view(*shape).view(torch.float32)


def bits(t):
    return t.contiguous().view(torch.int32)


def scale_err(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300)) if ref.numel() else 0.0


def ratio(err, bar):
    """max of err / bar where bar > 0; inf where the bar is 0 and the error is not."""
    if err.numel() == 0:
        return 0.0
    r = torch.where(bar > 0, err / bar.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max())


class Table:
    """Per-case rows printed as one table before the bars are checked, so that a failure shows every number."""

    def __init__(self, title, cols):
        self.title, self.cols, self.rows, self.failures = title, cols, [], []

    def add(self, case, *vals, ok=True, why=""):
        self.rows.append((case, vals))
        if not ok:
            self.failures.append(f"{case}: {why}")

    def check(self):
        print(f"\n--- {self.title}")
        print(f"    {'case':<34}" + "".join(f"{c:>13}" for c in self.cols))
        for case, vals in self.rows:
            print(f"    {case:<34}" + "".join(f"{v:>13.3e}" if isinstance(v, float) else f"{v!s:>13}" for v in vals))
        assert not self.failures, "; ".join(self.failures[:8])


@contextmanager
def plain_fp32():
    """Library matmuls in true fp32 (no TF32) for the cuBLAS yardstick; restored afterwards."""
    prev = torch.backends.cuda.matmul.allow_tf32, torch.get_float32_matmul_precision()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev[0]
        torch.set_float32_matmul_precision(prev[1])
