#!/usr/bin/env python3
"""Tuning aid: times the fused scorer (train / inference forms) on C3-sized random inputs."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from pangnn_b200 import ops, _abi
dev = "cuda:0"
N, E, D = 1_000_000, 10_000_000, 64
torch.manual_seed(0)
pq = torch.randn(N, 2 * D, device=dev)
# C3-like locality: destination = random node of the next genome block of 100k
src = torch.sort(torch.randint(0, N, (E,), device=dev)).values
dst = ((src // 100_000 + 1) % 10) * 100_000 + torch.randint(0, 100_000, (E,), device=dev)
ei = torch.stack((src, dst))
gs = ops.GraphStruct(ei, N)
skip = torch.rand(E, device=dev) * 80 + 1
y = (torch.rand(E, device=dev) < 0.2).float()
w1c, b1, b2, b3 = (torch.randn(D, device=dev) * 0.1 for _ in range(3)).__iter__().__next__(), torch.randn(D, device=dev) * .1, torch.randn(D, device=dev) * .1, torch.randn(1, device=dev)
w2 = torch.randn(D, D, device=dev) / 8
w3 = torch.randn(1, D, device=dev) / 8
logits = torch.empty(E, device=dev); da1 = torch.empty(E, D, device=dev)
grads = torch.empty(ops.NGRADS, device=dev); loss = torch.zeros(1, dtype=torch.float64, device=dev)
ws = ops._ws(_abi.load().pangnn_edge_score_workspace_bytes(E), dev)
def train():
    ops.edge_score_train(pq, w1c, b1, w2, b2, w3, b3, gs, skip, y=y, pos_weight=4.0, scale=1.0 / E, logits=logits,
                         loss_sum=loss, da1=da1, grads=grads, ws=ws)
def infer():
    ops.edge_score_pq_fwd(pq, w1c, b1, w2, b2, w3, b3, gs, skip)
def timeit(f, reps=10):
    for _ in range(3): f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): f()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps
tt, ti = timeit(train), timeit(infer)
print(json.dumps({"train_ms": round(tt, 3), "train_GBs": round(E * 784 / tt / 1e6, 1), "infer_ms": round(ti, 3),
                  "infer_GBs": round(E * 528 / ti / 1e6, 1), "edges_per_s_train": E / tt * 1e3}))

# ---- accuracy at scale vs an fp64 evaluation of the same formulas (chunked to bound memory)
def fp64_ref():
    W2, W3 = w2.double(), w3.double().squeeze(0)
    dW2 = torch.zeros(D, D, dtype=torch.float64, device=dev)
    gb2 = torch.zeros(D, dtype=torch.float64, device=dev); gw3 = torch.zeros_like(gb2); gb1 = torch.zeros_like(gb2); gw1c = torch.zeros_like(gb2)
    lsum = torch.zeros((), dtype=torch.float64, device=dev); zs = []
    pw, scale = 4.0, 1.0 / E
    CH = 1_000_000
    for a in range(0, E, CH):
        s_, d_ = src[a:a + CH], dst[a:a + CH]
        a1 = pq[s_, :D].double() + pq[d_, D:].double() + skip[a:a + CH, None].double() * w1c.double() + b1.double()
        r1 = a1.clamp_min(0)
        a2 = r1 @ W2.t() + b2.double()
        r2 = a2.clamp_min(0)
        z = r2 @ W3 + b3.double()
        yy = y[a:a + CH].double()
        lsum += ((1 - yy) * z + (1 + (pw - 1) * yy) * (torch.log1p(torch.exp(-z.abs())) + (-z).clamp_min(0))).sum()
        dz = ((pw * yy + 1 - yy) * torch.sigmoid(z) - pw * yy) * scale
        da2 = dz[:, None] * W3 * (a2 > 0)
        dW2 += da2.t() @ r1; gb2 += da2.sum(0); gw3 += (dz[:, None] * r2).sum(0)
        da1 = (da2 @ W2) * (a1 > 0)
        gb1 += da1.sum(0); gw1c += (da1 * skip[a:a + CH, None].double()).sum(0)
        zs.append(z)
    return torch.cat(zs), lsum, dW2, gb2, gw3, gb1, gw1c
loss.zero_(); train(); torch.cuda.synchronize()
z, lsum, dW2, gb2, gw3, gb1, gw1c = fp64_ref()
rel = lambda got, ref: float((got.double() - ref).abs().max() / ref.abs().max())
g = ops.scorer_grads(grads)
print(json.dumps({"err_logits": rel(logits, z), "err_loss": abs(float(loss) - float(lsum)) / abs(float(lsum)),
                  "err_dW2": rel(g.dW2, dW2), "err_db2": rel(g.db2, gb2), "err_dw3": rel(g.dw3[0], gw3),
                  "err_db1": rel(g.db1, gb1), "err_dw1c": rel(g.dw1c, gw1c)}))
