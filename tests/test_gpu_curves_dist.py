"""ROC and precision-recall curves over two GPUs (NCCL; skipped with fewer): ``metrics.roc_curve`` /
``metrics.precision_recall_curve`` on per-rank slices equal one GPU on the concatenation, bit for bit."""
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")]


def _slices():
    """400 000 scores with heavy ties and a saturated tail at 1.0f; rank 0 gets the first third, rank 1 the rest."""
    rng = np.random.default_rng(6)
    E = 400_000
    y = (rng.random(E) < 0.04).astype(np.float32)
    s = (np.round(rng.random(E) * 200) / 200 + 0.2 * y).astype(np.float32)
    s[rng.random(E) < 0.01] = 1.0
    return s, y, [(s[:E // 3], y[:E // 3]), (s[E // 3:], y[E // 3:])]


def _all(s, y):
    from pangnn_b200 import metrics
    out = {}
    for drop in (True, False):
        out[drop] = ([t.cpu() for t in metrics.roc_curve(s, y, drop_intermediate=drop)],
                     [t.cpu() for t in metrics.precision_recall_curve(s, y, drop_intermediate=drop)])
    return out


def _worker(rank, world, init_file, out_dir):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world, device_id=dev)
    try:
        _, _, parts = _slices()
        s, y = (torch.from_numpy(a).to(dev) for a in parts[rank])
        e = torch.zeros(0, device=dev)
        res = {"slices": _all(s, y), "empty_rank": _all(s if rank else e, y if rank else e)}
        torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_ranks():
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdv"), tmp), nprocs=2, join=True)
        yield [torch.load(os.path.join(tmp, f"r{r}.pt")) for r in range(2)]


def _equal(a, b):
    return all(x.dtype == w.dtype and torch.equal(x, w) for x3, w3 in zip(a, b) for x, w in zip(x3, w3))


def test_slices_equal_one_gpu_on_the_concatenation(two_ranks):
    s, y, _ = _slices()
    ref = _all(torch.from_numpy(s).cuda(), torch.from_numpy(y).cuda())
    tail = _all(torch.from_numpy(s[len(s) // 3:]).cuda(), torch.from_numpy(y[len(y) // 3:]).cuda())
    for r in two_ranks:
        for drop in (True, False):
            assert _equal(r["slices"][drop], ref[drop])
            assert _equal(r["empty_rank"][drop], tail[drop])
