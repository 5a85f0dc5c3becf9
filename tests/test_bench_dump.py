"""``bench.py --dump-outputs``: what the last timed step computed, written as float32 / float64 ``.npy`` files within
the size limit, the same on every call, with a fixed sample of the logits when there are too many edges."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from tests.helpers import rel_err


def _step(n_edges):
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(3, 4), torch.nn.ELU(), torch.nn.Linear(4, 1))
    logits = model(torch.randn(n_edges, 3)).squeeze(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(logits, (torch.arange(n_edges) % 2).float())
    loss.backward()
    return loss, logits.detach(), model


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_writes_the_step_outputs(tmp_path):
    loss, logits, model = _step(100)
    bench.dump_outputs(str(tmp_path / "a"), loss, logits, model)
    out = _read(str(tmp_path / "a"))
    names = {f"{kind}.{n}" for n, _ in model.named_parameters() for kind in ("param", "grad")}
    assert set(out) == {"loss", "logits"} | names
    assert all(v.dtype in (np.float32, np.float64) for v in out.values())
    assert out["loss"] == loss.item()
    assert np.array_equal(out["logits"], logits.numpy())
    for n, p in model.named_parameters():
        assert np.array_equal(out[f"param.{n}"], p.detach().numpy()) and np.array_equal(out[f"grad.{n}"], p.grad.numpy())


def test_dump_samples_many_logits_the_same_way_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LOGITS_FULL", 50)
    monkeypatch.setattr(bench, "DUMP_LOGITS_SAMPLE", 20)
    loss, logits, model = _step(100)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), loss, logits, model)
    a, b = _read(str(tmp_path / "a")), _read(str(tmp_path / "b"))
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["logits_index"]
    assert idx.dtype == np.float64 and idx.size == 20 and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["logits"], logits.numpy()[idx.astype(np.int64)])


def test_dump_refuses_more_than_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 100)
    loss, logits, model = _step(100)
    with pytest.raises(RuntimeError, match="limit"):
        bench.dump_outputs(str(tmp_path / "a"), loss, logits, model)
    assert not os.path.exists(tmp_path / "a")


@pytest.mark.gpu
def test_bench_dumps_its_last_timed_step(tmp_path):
    """``bench.py --dump-outputs`` on the c2 workload against the same seeded run trained here step by step: the dump
    is the state after the warm-up and timed steps, not after the inference / end-to-end legs that follow them."""
    from pangnn_b200 import ops, setup
    from pangnn_b200 import preprocessing as pp
    from pangnn_b200.data import Data
    from pangnn_b200.gnn import AlternateGCN
    from pangnn_b200.simulate import simulate_hits
    warmup, steps = 3, 2
    out = tmp_path / "dump"
    subprocess.run([sys.executable, bench.__file__, "--workload", "c2", "--steps", str(steps), "--warmup", str(warmup),
                    "--no_cpu", "--no_secondary", "--dump-outputs", str(out)], check=True, stdout=subprocess.DEVNULL)
    dump = _read(str(out))

    wl, dev = bench.WORKLOADS["c2"], torch.device("cuda:0")
    setup.reset()
    ops.clear_cache()
    try:
        for k, v in wl["flags"].items():
            setattr(setup.args, k, v)
        assert not setup.args.union_edge_weights                 # the graph below is bench.py's non-union assembly
        s = simulate_hits(*wl["sim"], seed=0)
        N = s["num_genes"]
        h = {k: torch.from_numpy(np.ascontiguousarray(s[k])) for k in ("q", "t", "bits", "genome_of", "group_of")}
        src, dst, w, y = pp.normalize_sim_scores(h["q"], h["t"], h["bits"], h["genome_of"], h["group_of"], num_nodes=N,
                                                 t_norm=0.8, include_trivial=False, device=dev)
        graph = Data(torch.ones(N, 1, device=dev), torch.stack((src.long(), dst.long())), w, y)
        graph.neighbour_edge_index = pp.neighbour_band(N, setup.args.neighbours, dev)
        pw = float(((y == 0).sum() / y.sum()).item())
        torch.manual_seed(0)
        model = AlternateGCN(dev, None, False).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        states = []
        for _ in range(warmup + steps + 1):
            opt.zero_grad(set_to_none=False)
            loss, logits = model.forward_loss(graph, pw)
            loss.backward()
            opt.step()
            st = {"loss": loss.detach().cpu().numpy(), "logits": logits.cpu().numpy()}
            for n, p in model.named_parameters():
                st[f"param.{n}"] = p.detach().cpu().numpy().copy()
                if p.grad is not None:
                    st[f"grad.{n}"] = p.grad.cpu().numpy().copy()
            states.append(st)
    finally:
        setup.reset()
        ops.clear_cache()
    last, later = states[warmup + steps - 1], states[-1]
    assert set(dump) == set(last)
    for k, v in dump.items():
        assert rel_err(v, last[k]) < 1e-6, k
    assert rel_err(dump["param.mlp.4.weight"], later["param.mlp.4.weight"]) > 1e-4   # one more step is told apart
