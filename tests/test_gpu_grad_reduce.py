"""The peer-memory gradient average (csrc/grad_reduce.cu: ``ops.grad_push`` / ``ops.grad_reduce``) with ``W`` ranks
emulated in one process on one GPU: ``W`` buckets, ``W`` signal arrays and one control block per emulated rank, all
``W`` pushes queued before any reduce.  Results are bit-exact against numpy's fp32 rank-order sum times fp32(1/W),
over successive calls (both bucket halves, the epoch advance) and over replays of one captured CUDA graph."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SIZES = [1, 3, 64, 8192, 8256, 16384, 3, 1]
NULL = {2, 6}                                                   # gradients that are None on every rank


class Ranks:
    def __init__(self, world, dev):
        from pangnn_b200 import ops
        self.world, self.dev = world, dev
        self.half = ops.grad_bucket_floats(SIZES)
        self.buckets = [torch.full((2, self.half), float("nan"), device=dev) for _ in range(world)]
        self.signals = [torch.zeros(ops.GRAD_REDUCE_MAX_RANKS, dtype=torch.int32, device=dev) for _ in range(world)]
        self.ctrl = [torch.zeros(4, dtype=torch.int32, device=dev) for _ in range(world)]
        # gradients of rank r: odd offsets inside one allocation, so no tensor boundary is aligned
        self.store = [torch.zeros(sum(SIZES) + 7, device=dev) for _ in range(world)]
        self.grads = []
        for r in range(world):
            off, gl = 1, []
            for i, n in enumerate(SIZES):
                gl.append(None if i in NULL else self.store[r][off:off + n])
                off += n + (i % 2)
            self.grads.append(gl)

    def fill(self, gen):
        host = []
        for r in range(self.world):
            vals = [None if g is None else (torch.randn(g.numel(), generator=gen) * 10 ** float(torch.randint(-3, 4, (1,), generator=gen)))
                    for g in self.grads[r]]
            for g, v in zip(self.grads[r], vals):
                if g is not None:
                    g.copy_(v)
            host.append([None if v is None else v.numpy().astype(np.float32) for v in vals])
        return host

    def call(self):
        from pangnn_b200 import ops
        sig = [s.data_ptr() for s in self.signals]
        buck = [b.data_ptr() for b in self.buckets]
        for r in range(self.world):
            ops.grad_push(self.grads[r], SIZES, self.buckets[r], self.half, sig, r, self.ctrl[r])
        for r in range(self.world):
            ops.grad_reduce(self.grads[r], SIZES, buck, self.half, self.signals[r], r, self.ctrl[r], timeout_s=30.0)

    def check(self, host, calls):
        scale = np.float32(1.0 / self.world)
        for i in range(len(SIZES)):
            if i in NULL:
                continue
            acc = host[0][i].copy()
            for r in range(1, self.world):
                acc = (acc + host[r][i]).astype(np.float32)
            ref = (acc * scale).astype(np.float32)
            for r in range(self.world):
                got = self.grads[r][i].cpu().numpy()
                assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (self.world, r, i)
        for r in range(self.world):
            c = self.ctrl[r].tolist()
            assert c == [calls, 0, 0, 0], c                     # epoch advanced, tickets reset, status 0
            assert self.signals[r][:self.world].tolist() == [calls] * self.world
        assert float(self.store[0][0]) == 0.0                   # nothing written outside the tensors


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_grad_average_bit_exact_over_successive_calls(world):
    dev = torch.device("cuda", 0)
    R = Ranks(world, dev)
    gen = torch.Generator().manual_seed(world)
    for k in range(5):
        host = R.fill(gen)
        R.call()
        torch.cuda.synchronize()
        R.check(host, k + 1)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_grad_average_captured_and_replayed(world):
    dev = torch.device("cuda", 0)
    R = Ranks(world, dev)
    gen = torch.Generator().manual_seed(10 + world)
    host = R.fill(gen)
    R.call()                                                    # one eager call first: replays continue its epochs
    torch.cuda.synchronize()
    R.check(host, 1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        R.call()
    torch.cuda.synchronize()
    R.check(host, 1)                                            # capturing runs nothing
    for k in range(3):
        host = R.fill(gen)
        g.replay()
        torch.cuda.synchronize()
        R.check(host, 2 + k)
    host = R.fill(gen)
    R.call()                                                    # eager after the replays
    torch.cuda.synchronize()
    R.check(host, 5)


def test_grad_reduce_refuses_bad_arguments():
    from pangnn_b200 import _abi, ops
    dev = torch.device("cuda", 0)
    half = ops.grad_bucket_floats([4])
    bucket = torch.zeros(2, half, device=dev)
    sig = torch.zeros(8, dtype=torch.int32, device=dev)
    ctrl = torch.zeros(4, dtype=torch.int32, device=dev)
    g = [torch.zeros(4, device=dev)]
    before = ops.LAUNCHES["count"]
    cases = [
        (lambda: ops.grad_push([g[0]] * 33, [4] * 33, bucket, 33 * 4, [sig.data_ptr()], 0, ctrl), "count"),
        (lambda: ops.grad_push(g, [4], bucket, half, [sig.data_ptr()] * 9, 0, ctrl), "world"),
        (lambda: ops.grad_reduce(g, [4], [bucket.data_ptr()] * 2, half, sig, 2, ctrl), "rank"),
        (lambda: ops.grad_reduce(g, [4], [bucket.data_ptr()], half, sig, -1, ctrl), "rank"),
        (lambda: ops.grad_push(g, [4], bucket, 0, [sig.data_ptr()], 0, ctrl), "too small"),
        (lambda: ops.grad_reduce(g, [4], [bucket.data_ptr()] * 9, half, sig, 0, ctrl), "world"),
    ]
    for fn, needle in cases:
        with pytest.raises(_abi.PangnnError, match=needle):
            fn()
        assert needle in _abi.load().pangnn_last_error().decode()
    torch.cuda.synchronize()
    assert ops.LAUNCHES["count"] == before
    assert ctrl.tolist() == [0, 0, 0, 0] and sig.tolist() == [0] * 8
