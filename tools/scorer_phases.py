#!/usr/bin/env python3
"""Development aid: per-phase cycle breakdown of the scorer's training kernel (thread 0 of every CTA), from the
profiling build (`python -m pangnn_b200.build --prof`).  Not a bench: the counters add a few clock reads."""
import ctypes, os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["PANGNN_B200_LIB"] = os.path.join(ROOT, "pangnn_b200", "_lib", "libpangnn_b200_prof.so")
import torch
from pangnn_b200 import ops, _abi
dev = "cuda:0"
N, E, D = 1_000_000, int(os.environ.get("E", 10_000_000)), 64
torch.manual_seed(0)
pq = torch.randn(N, 2 * D, device=dev)
src = torch.sort(torch.randint(0, N, (E,), device=dev)).values
dst = ((src // 100_000 + 1) % 10) * 100_000 + torch.randint(0, 100_000, (E,), device=dev)
s32, d32 = src.int(), dst.int()
skip = torch.rand(E, device=dev) * 80 + 1
y = (torch.rand(E, device=dev) < 0.2).float()
w1c, b1, b2, b3 = (torch.randn(D, device=dev) * .1 for _ in range(3)).__next__(), torch.randn(D, device=dev) * .1, torch.randn(D, device=dev) * .1, torch.randn(1, device=dev)
w2, w3 = torch.randn(D, D, device=dev) / 8, torch.randn(1, D, device=dev) / 8
lib = _abi.load()
logits = torch.empty(E, device=dev); da1 = torch.empty(E, D, device=dev)
grads = torch.empty(ops.NGRADS, device=dev); loss = torch.zeros(1, dtype=torch.float64, device=dev)
ws = ops._ws(lib.pangnn_edge_score_workspace_bytes(E), dev)
def train():
    ops.edge_score_train(pq, w1c, b1, w2, b2, w3, b3, (s32, d32), skip, y=y, pos_weight=4.0, scale=1.0 / E,
                         logits=logits, loss_sum=loss, da1=da1, grads=grads, ws=ws)
prof = lib.pangnn_debug_scorer_prof
buf = (ctypes.c_ulonglong * 16)()
for _ in range(2): train()
prof(buf, 1)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); train(); e1.record(); torch.cuda.synchronize()
prof(buf, 1)
names = os.environ.get("PHASES", "loads+G3wait,r1+stores,arrive+L2pf,G1wait,epi1a+arrive,sync,epi1b+arrive,G2wait,epi2,-,-,-").split(",")
tiles = (E + 127) // 128
tot = sum(buf[i] for i in range(12))
print(f"kernel {e0.elapsed_time(e1):.3f} ms; tiles {tiles}; cycles per tile (thread 0, avg over CTAs):")
for i, n in enumerate(names):
    print(f"  {n:16s} {buf[i] / tiles:9.1f}  {100.0 * buf[i] / max(tot, 1):5.1f} %")
print(f"  {'total':16s} {tot / tiles:9.1f}")
