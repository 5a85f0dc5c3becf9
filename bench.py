#!/usr/bin/env python3
"""bench.py — throughput of the panGNN message-passing hot path on B200 (see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|...] [--impl reference] [--dump-outputs DIR]

A "step" is one whole-graph training step (fused fwd + BCE loss + bwd + Adam) over the
``generate_graphs()`` graph of a ``--simulate_dataset`` configuration of BASELINE.json.
Inputs and initial weights are seeded, so the same arguments give the same inputs on every run;
``--dump-outputs DIR`` writes what the last timed step computed (``dump_outputs``).
Prints ONE JSON line.  ``value`` = scored similarity edges per second with graph + CSR resident in
HBM; ``e2e`` = the same step through the public API from pinned HOST buffers (H2D of the batch,
CSR build, gcn_norm, step, loss read-back inside the timed region).  ``--impl reference`` times the
CPU oracle port of the reference model on the host cores.  The oracle is only ever the CPU arm.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # name: (simulate_dataset args, model flags)       — BASELINE.json configs[1..3]
    "c2": dict(sim=(10000, 2, 0.5, 10, 3), flags=dict(neighbours=1),
               desc="--simulate_dataset 10000 2 0.5 10 3 (whole graph)"),
    "c3": dict(sim=(100000, 10, 0.5, 50, 10),
               flags=dict(union_edge_weights=True, neighbours=3, skip_connections=True),
               desc="--simulate_dataset 100000 10 0.5 50 10 --union_edge_weights --neighbours 3 --skip_connections (whole graph)"),
    # configs[3]: multi-GPU only (--gpus 2 or 4: whole genomes per rank); G stays 20, strong scaling
    "c4": dict(sim=(200000, 20, 0.3, 100, 20), flags=dict(neighbours=1, categorical_node=True), fixed_G=True,
               desc="--simulate_dataset 200000 20 0.3 100 20 --categorical_node (whole graph, genome-partitioned)"),
    # configs[4] (pan-genome scale, 1e6 genes x 50 genomes, ~9.7e9 scored edges) at 1/10 of its genes per genome: the
    # same 50 genomes, per-gene candidate statistics (m = 98 negatives per gene and direction), synteny blocks and
    # flags; 9.7e8 scored edges, 1.2e8 per GPU on 8 GPUs.  The full size needs the per-rank build in 32-bit ids and
    # the scorer's per-edge spill in chunks (DESIGN.md §6b); multi-GPU only.
    "c5s": dict(sim=(100000, 50, 0.2, 500, 50), flags=dict(neighbours=1), fixed_G=True,
                desc="--simulate_dataset 100000 50 0.2 500 50 (configs[4] at 1/10 of its genes per genome; whole graph, genome-partitioned)"),
    "c5q": dict(sim=(250000, 50, 0.2, 500, 50), flags=dict(neighbours=1), fixed_G=True,
                desc="--simulate_dataset 250000 50 0.2 500 50 (configs[4] at 1/4 of its genes per genome; whole graph, genome-partitioned)"),
    "c5h": dict(sim=(500000, 50, 0.2, 500, 50), flags=dict(neighbours=1), fixed_G=True,
                desc="--simulate_dataset 500000 50 0.2 500 50 (configs[4] at 1/2 of its genes per genome; whole graph, genome-partitioned)"),
    "c5": dict(sim=(1000000, 50, 0.2, 500, 50), flags=dict(neighbours=1), fixed_G=True,
               desc="--simulate_dataset 1000000 50 0.2 500 50 (configs[4]; whole graph, genome-partitioned)"),
    "c3_default": dict(sim=(100000, 10, 0.5, 50, 10), flags=dict(neighbours=1),
                       desc="--simulate_dataset 100000 10 0.5 50 10 (two-graph default, whole graph)"),
}
# CPU arms run a bounded sample of the same workload: same genomes/flags, fewer genes per genome
CPU_SAMPLE_GENES = {"c2": 10000, "c3": 10000, "c3_default": 10000, "c4": 5000, "c5s": 2000, "c5q": 2000, "c5h": 2000, "c5": 2000}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML in a background
    thread (an `nvidia-smi -lms` child process measurably slowed the NCCL exchanges of the
    multi-GPU arm: 49 ms vs 19 ms per step at N=2)."""

    def __init__(self, index, period_s=0.2):
        self.index, self.period, self.rows, self._stop, self._t = index, period_s, [], threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip() != ""]
            if local < len(ids) and ids[local].strip().isdigit():
                return int(ids[local])
        return local

    def _sample(self):
        nv = self.nv
        sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        return sm, mx, r

    def _run(self):
        while not self._stop.is_set():
            try:
                self.rows.append(self._sample())
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        try:
            self.rows.append(self._sample())                 # at least one sample inside the region
        except Exception:
            pass
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        sm = [float(r[0]) for r in self.rows]
        mx = [float(r[1]) for r in self.rows]
        reasons = sorted({n for r in self.rows for n, bit in names.items() if r[2] & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons, "source": "NVML, 200 ms period"}


DUMP_MAX_BYTES = 64 << 20
DUMP_LOGITS_FULL = 12 << 20          # logits of up to this many edges are written whole (48 MB of float32)
DUMP_LOGITS_SAMPLE = 4 << 20         # above that, a fixed sample of this many edges


def dump_outputs(out_dir, loss, logits, model):
    """Write what one training step hands its caller as ``out_dir/<name>.npy``: ``loss``, the per-edge ``logits``,
    and every parameter after the optimiser step (``param.<name>``) with the gradient it was updated from
    (``grad.<name>``).  Two builds run with the same arguments can so be compared output for output.  Logits of
    more than DUMP_LOGITS_FULL edges are cut to a seeded sample; ``logits_index`` then holds the sampled edges'
    positions (float64, exact)."""
    arrays = {"loss": loss.detach().float().cpu().numpy()}
    z = logits.detach().float().cpu().numpy()
    if z.size > DUMP_LOGITS_FULL:
        idx = np.sort(np.random.default_rng(0).choice(z.size, DUMP_LOGITS_SAMPLE, replace=False))
        arrays["logits"], arrays["logits_index"] = z[idx], idx.astype(np.float64)
    else:
        arrays["logits"] = z
    for name, p in model.named_parameters():
        arrays[f"param.{name}"] = p.detach().float().cpu().numpy()
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad.detach().float().cpu().numpy()
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


def agg_bytes(E, N, F):
    """Algorithmic bytes of one aggregation launch (SURVEY.md §8d / DESIGN.md): per edge 4 (col) +
    4 (val) + 4F (gathered row), per node 4F (output row) + 8 (rowptr)."""
    return E * (8 + 4 * F) + N * 4 * F + 8 * (N + 1)


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference model) — also the `cpu_baseline` leg of the GPU arm
# ------------------------------------------------------------------------------------------------
def cpu_arm(workload, steps, warmup, budget_s=None):
    """``steps`` timed whole-graph steps after ``warmup``; with ``budget_s`` (the cpu_baseline leg of the GPU arm) each
    loop stops early once it has taken that many seconds, and ``steps`` of the result says how many were timed."""
    from types import SimpleNamespace
    from oracle import preprocess as op
    from oracle.model import AlternateGCN as OracleGCN, Flags, bce_with_logits
    from oracle.params import make_state_dict
    from pangnn_b200.simulate import simulate_hits
    wl = WORKLOADS[workload]
    n, G, f, frags, shuf = wl["sim"]
    n_s = min(n, CPU_SAMPLE_GENES[workload])
    torch.set_num_threads(os.cpu_count() or 1)
    s = simulate_hits(n_s, G, f, frags, shuf, seed=0)
    q, t, b = op.dedupe_last(s["q"].astype(np.int64), s["t"].astype(np.int64), s["bits"])
    q, t, b = op.remove_trivial_cases(q, t, b, s["genome_of"])
    src, dst, w = op.normalize_sim_scores(q, t, b, s["genome_of"])
    y = op.map_labels(src, dst, s["group_of"])
    flags = Flags(**wl["flags"])
    N = s["num_genes"]
    ei = np.stack((src, dst))
    nb = op.neighbour_band(N, flags.neighbours)
    g = SimpleNamespace(x=torch.ones(N, 1), edge_index=torch.from_numpy(ei), y=torch.from_numpy(y))
    if flags.union_edge_weights:
        uei, uw = op.union_whole_graph(ei, w, nb)
        g.union_edge_index, g.edge_attr = torch.from_numpy(uei), torch.from_numpy(uw)
    else:
        g.neighbour_edge_index, g.edge_attr = torch.from_numpy(nb), torch.from_numpy(w.astype(np.float32))
    model = OracleGCN(flags)
    model.load_state_dict(make_state_dict(skip_connections=flags.skip_connections), strict=True)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    pw = op.class_balance(y)
    E = int(src.size)

    def step():
        opt.zero_grad()
        loss = bce_with_logits(model(g), g.y, pw)
        loss.backward()
        opt.step()
        return loss.item()

    t0 = time.perf_counter()
    for _ in range(warmup):
        step()
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    times = []
    for _ in range(steps):
        t1 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t1)
        if budget_s is not None and sum(times) > budget_s:
            break
    dt = float(np.median(times))
    sample = (f"--simulate_dataset {n_s} {G} {f} {frags} {shuf} with the workload's flags: N={N}, "
              f"E_scored={E}, {len(times)} whole-graph steps (fwd+loss+bwd+Adam), median")
    return {"value": E / dt, "unit": "edges/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": sample, "ms_per_step": dt * 1e3, "steps": len(times)}, E


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def gpu_arm(a):
    import torch.distributed as dist
    from pangnn_b200 import ops, setup
    from pangnn_b200 import preprocessing as pp
    from pangnn_b200.data import Data
    from pangnn_b200.gnn import AlternateGCN
    from pangnn_b200.simulate import simulate_hits

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = WORKLOADS[a.workload]
    n, G, f, frags, shuf = wl["sim"]
    setup.reset()
    for k, v in wl["flags"].items():
        setattr(setup.args, k, v)
    flags = setup.args
    if world > 1:
        return partitioned_arm(a, wl, world, rank, local, dev)

    # ---- input: the simulated pan-genome, host side
    s = simulate_hits(n, G, f, frags, shuf, seed=0)
    N = s["num_genes"]
    host = {k: torch.from_numpy(np.ascontiguousarray(s[k])).pin_memory() for k in ("q", "t", "bits", "genome_of", "group_of")}

    def preprocess():
        return pp.normalize_sim_scores(host["q"], host["t"], host["bits"], host["genome_of"], host["group_of"],
                                       num_nodes=N, t_norm=0.8, include_trivial=False, device=dev)

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    src, dst, w, y = preprocess()
    torch.cuda.synchronize()
    prep_s = time.perf_counter() - t0
    E = int(src.numel())

    def assemble(src, dst, w, y):
        """src/dataset.py:325-395 on the device: band (a8) + union assembly (a11)."""
        ei = torch.stack((src.long(), dst.long()))
        x = torch.ones(N, 1, device=dev)
        if flags.union_edge_weights:
            union = ops.union_index(ei, N, flags.neighbours)
            g = Data(x, ei, ops.union_weights(w, union.size(1)), y)
            g.union_edge_index = union
        else:
            g = Data(x, ei, w, y)
            g.neighbour_edge_index = pp.neighbour_band(N, flags.neighbours, dev)
        return g

    graph = assemble(src, dst, w, y)
    pw = float(((y == 0).sum() / y.sum()).item())
    torch.manual_seed(0)
    model = AlternateGCN(dev, None, False).to(dev)                 # random init of the reference architecture
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    params = [p for p in model.parameters()]

    def allreduce_grads():
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in params if p.grad is not None])
            dist.all_reduce(flat)
            flat /= world
            off = 0
            for p in params:
                if p.grad is not None:
                    p.grad.copy_(flat[off:off + p.numel()].view_as(p))
                    off += p.numel()

    step_out = {}

    def step(g):
        opt.zero_grad(set_to_none=False)
        loss, logits = model.forward_loss(g, pw)
        loss.backward()
        allreduce_grads()
        opt.step()
        if a.dump_outputs:
            step_out["loss"], step_out["logits"] = loss.detach(), logits
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """k calls of fn bracketed by barrier+sync; device time via CUDA events; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- value: inputs resident in HBM (graph, CSR, norm built during warm-up)
    for _ in range(a.warmup):
        step(graph)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = ops.LAUNCHES["count"]
    ms = timed(lambda: step(graph), a.steps)
    launches = ops.LAUNCHES["count"] - l0
    clk = clocks.stop() if rank == 0 else None
    value = E * world * a.steps / (ms * 1e-3)
    if a.dump_outputs:                                      # here, before the legs below train the model further
        dump_outputs(a.dump_outputs, step_out["loss"], step_out["logits"], model)

    if a.profile:
        a.no_cpu = True
    # ---- inference edges/s (forward only, no_grad)
    def infer():
        with torch.no_grad():
            return model(graph)
    for _ in range(0 if a.profile else 2):
        infer()
    ms_inf = timed(infer, 1 if a.profile else a.steps)

    # ---- e2e: public API from pinned host buffers, everything rebuilt per step
    # The host batch is what the host-side preprocessing hands over: the SCORED edges (int64 edge_index as on
    # the PyG surface, Q-score weights, labels) and x.  The neighbour band (a8) and the union assembly (a11)
    # are rows of the hot path and run on the device inside the timed region (AlternateGCN.prepare).
    gh = Data(torch.ones(N, 1), torch.stack((src.long(), dst.long())).cpu(), w.cpu(), y.cpu()).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in gh.__dict__.values() if torch.is_tensor(v))
    e2e_steps = 1 if a.profile else max(3, min(a.steps, 10))
    last = {}

    from pangnn_b200.data import PrefetchLoader

    def e2e_run(k):
        """k steps, each from the pinned host batch: H2D + band / union assembly + CSR builds of step i+1 overlap
        step i (one batch of look-ahead, as a prefetching DataLoader gives); loss.item() every step."""
        ops.clear_cache()
        loader = PrefetchLoader([gh] * k, model, dev)
        for g in loader:
            loss = step(g)                                  # queue the step,
            loader.prefetch_next()                          # then the next batch's copy + structure build beside it
            last["loss"] = loss.item()                      # D2H read of the step's loss (pangnn.py:218)
    if not a.profile:
        e2e_run(3)
        e2e_run(e2e_steps)                                  # a full-length untimed repetition (allocator steady state)
    e2e_reps = [timed(lambda: e2e_run(e2e_steps), 1) for _ in range(1 if a.profile else 5)]
    ms_e2e = float(np.median(e2e_reps))                     # median of 5 repetitions of e2e_steps steps each

    def e2e_serial():                                       # the same step without look-ahead, for the record
        ops.clear_cache()
        g = model.prepare(gh.to_pipelined(dev, order=model.transfer_order(scored_only=True)))
        last["loss"] = step(g).item()
    ms_e2e_serial = None
    if not a.profile:
        e2e_serial()
        ms_e2e_serial = timed(e2e_serial, 3) / 3
    e2e_val = E * world * e2e_steps / (ms_e2e * 1e-3)
    ops.clear_cache()
    step(graph)                                             # restore the resident structures

    # ---- roofline of the dominant kernel: normalised aggregation at the widest layer, timed alone
    ei_c = graph.union_edge_index if flags.union_edge_weights else graph.edge_index
    gs = ops.graph_struct(ei_c, N)
    ent = gs.norm(graph.edge_attr, need_src=False)
    F = flags.hidden_dim
    xin = torch.randn(N, F, device=dev)
    out = torch.empty(N, F, device=dev)
    bias = torch.zeros(F, device=dev)
    agg = lambda: ops.gcn_aggregate(gs.dst.rowptr, gs.dst.col, ent["dst"], xin, N, bias, ops.ACT_ELU, out=out)
    for _ in range(3):
        agg()
    reps = 3 if a.profile else 20
    ms_agg = timed(agg, reps) / reps
    Ec = int(ei_c.size(1))
    abytes = agg_bytes(Ec, N, F)
    peak, peak_src = peaks()
    achieved = abytes / (ms_agg * 1e-3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "agg_traffic.json")
    if os.path.exists(prof):
        traffic = json.load(open(prof)).get(a.workload)

    # ---- the other large kernel of the step, timed alone the same way: the fused scorer (training and inference
    #      forms) on this graph's scored edges; algorithmic bytes per edge from SURVEY §8d (784 / 528 B)
    others = []
    if not a.profile and flags.decoder == "mlp":
        from pangnn_b200 import _abi
        lib, P, D = _abi.load(), ops._p, ops.SCORER_D
        gsc = ops.graph_struct(graph.edge_index, N)
        s32, d32 = gsc.endpoints32
        pq = torch.randn(N, 2 * D, device=dev)
        m = model.mlp
        skip = graph.edge_attr[:E].contiguous() if flags.skip_connections else None
        w1c = m[0].weight[:, 2 * D].contiguous() if skip is not None else None
        w2, w3 = m[2].weight.detach().contiguous(), m[4].weight.detach().contiguous()
        b1, b2, b3 = m[0].bias.detach(), m[2].bias.detach(), m[4].bias.detach()
        logits = torch.empty(E, device=dev)
        da1 = torch.empty(E, D, device=dev)
        grads = torch.empty(ops.NGRADS, device=dev)
        lsum = torch.zeros(1, dtype=torch.float64, device=dev)
        ws = ops._ws(lib.pangnn_edge_score_workspace_bytes(E), dev)
        sc_train = lambda: _abi.check(lib.pangnn_edge_score_bwd(
            P(pq), P(s32), P(d32), P(skip), P(w1c), P(b1), P(w2), P(b2), P(w3), P(b3), E, None, P(graph.y), pw, 1.0 / E,
            P(da1), P(grads), P(logits), P(lsum), P(ws), ws.numel(), ops._stream()), "edge_score_bwd")
        sc_infer = lambda: _abi.check(lib.pangnn_edge_score_fwd(
            P(pq), P(s32), P(d32), P(skip), P(w1c), P(b1), P(w2), P(b2), P(w3), P(b3), E, None, 1.0, P(logits), None,
            None, 0, ops._stream()), "edge_score_fwd")
        for name, fn, bpe in (("edge_score_tc (training form: logits + loss + all gradients)", sc_train, 784),
                              ("edge_score_tc (inference form)", sc_infer, 528)):
            for _ in range(3):
                fn()
            t_ms = timed(fn, 10) / 10
            ach = E * bpe / (t_ms * 1e-3) / 1e9
            tr = (json.load(open(prof)).get(a.workload + ("_scorer_train" if bpe == 784 else "_scorer_infer"))
                  if os.path.exists(prof) else None)
            others.append({"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                           "algorithmic_bytes": E * bpe, "traffic": tr,
                           "frac_dram": (tr / (t_ms * 1e-3) / 1e9 / peak) if tr else None,
                           "us_per_launch": t_ms * 1e3, "timed": "alone, burst peak"})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- side measurement: configs[1] (N = 2e4, whole graph in L2, launch-latency-bound) for the record
    secondary = None
    if a.workload == "c3" and not a.profile and not a.no_secondary:
        try:
            secondary = small_config_leg("c2", dev, steps=max(a.steps, 20), warmup=max(a.warmup, 5))
        finally:
            setup.reset()
            for k, v in wl["flags"].items():
                setattr(setup.args, k, v)
    cpu, _ = cpu_arm(a.workload, steps=3, warmup=1, budget_s=45.0) if (world == 1 and not a.no_cpu) else (None, None)
    line = {
        "metric": "train_edges_per_s", "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "per_gpu": {"N": N, "E_scored": E, "E_conv": Ec},
                   "step": "whole-graph fwd + BCE(pos_weight) + bwd + Adam (fused scorer/loss kernel)",
                   "l2": "inputs larger than L2 (no flush needed)" if N * F * 4 > 126e6 else "graph fits in L2; not flushed",
                   "parallelism": f"dp{world}: one simulated pan-genome per GPU, weight-gradient all-reduce (NCCL)" if world > 1 else "single GPU",
                   "preprocess_s": prep_s},
        "inference_edges_per_s": E * world * a.steps / (ms_inf * 1e-3),
        "e2e": {"value": e2e_val, "unit": "edges/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps, "ms_per_step_without_lookahead": ms_e2e_serial,
                "repetitions_ms_per_step": [t / e2e_steps for t in e2e_reps],
                "includes": "every step: H2D of the scored-edge batch from pinned host memory (int64 edge_index [2,E], weights, labels, x; copy stream), neighbour band + union assembly on the device (a8, a11), CSR builds x2 orientations, gcn_norm, step, loss.item(); PrefetchLoader: copy + structure build of step i+1 overlap step i on side streams"},
        "gpu_launches": launches,
        "clocks": clk,
        # `frac` follows SURVEY §8d's no-reuse model (every gathered row counted as HBM traffic) and therefore exceeds
        # 1 when L2 serves the gathers; `frac_dram` = the DRAM bytes ncu measured for this kernel on this workload
        # (profiles/agg_traffic.json) over the same time — the honest HBM utilisation — and `frac_compulsory` the
        # lower bound (every input / output byte once)
        "roofline": {"bound": "hbm", "kernel": f"gcn_aggregate F={F} (+bias+ELU)", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic,
                     "frac_dram": (traffic / (ms_agg * 1e-3) / 1e9 / peak) if traffic else None,
                     "frac_compulsory": (8.0 * Ec + 8.0 * N * F + 4.0 * N) / (ms_agg * 1e-3) / 1e9 / peak,
                     "algorithmic_bytes": abytes, "us_per_launch": ms_agg * 1e3, "timed": "alone, burst peak",
                     "traffic_source": "profiles/agg_traffic.json (ncu --set full, one launch)" if traffic else None},
        "roofline_other_kernels": others,
        "cpu_baseline": cpu,
        "secondary": secondary,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def small_config_leg(workload, dev, steps, warmup):
    """Whole-graph training step + inference of a small configuration (fits in L2; launch-bound), same API."""
    from pangnn_b200 import ops, setup
    from pangnn_b200 import preprocessing as pp
    from pangnn_b200.data import Data
    from pangnn_b200.gnn import AlternateGCN
    from pangnn_b200.simulate import simulate_hits
    wl = WORKLOADS[workload]
    n, G, f, frags, shuf = wl["sim"]
    setup.reset()
    for k, v in wl["flags"].items():
        setattr(setup.args, k, v)
    flags = setup.args
    s = simulate_hits(n, G, f, frags, shuf, seed=0)
    N = s["num_genes"]
    src, dst, w, y = pp.normalize_sim_scores(s["q"], s["t"], s["bits"], s["genome_of"], s["group_of"], num_nodes=N,
                                             t_norm=0.8, include_trivial=False, device=dev)
    ei = torch.stack((src.long(), dst.long()))
    nb = pp.neighbour_band(N, flags.neighbours, dev)
    g = Data(torch.ones(N, 1, device=dev), ei, w, y)
    g.neighbour_edge_index = nb
    pw = float(((y == 0).sum() / y.sum()).item())
    torch.manual_seed(0)
    model = AlternateGCN(dev, None, False).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def step():
        opt.zero_grad(set_to_none=False)
        loss, _ = model.forward_loss(g, pw)
        loss.backward()
        opt.step()

    def infer():
        with torch.no_grad():
            model(g)

    def timed(fn, k):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k
    for _ in range(warmup):
        step()
    ms = timed(step, steps)
    infer()
    ms_inf = timed(infer, steps)
    E = int(src.numel())
    out = {"workload": wl["desc"], "N": N, "E_scored": E, "ms_per_step": ms, "train_edges_per_s": E / ms * 1e3,
           "inference_edges_per_s": E / ms_inf * 1e3,
           "note": "graph fits in L2; one step is ~90 kernel launches of a few microseconds each (launch-latency-bound)"}
    try:                                                      # the same step captured once and replayed as a CUDA graph
        from pangnn_b200.graphs import GraphedStep
        gopt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        gstep = GraphedStep(model, g, gopt, pw)
        ms_g = timed(gstep, steps)
        out["cuda_graph"] = {"ms_per_step": ms_g, "train_edges_per_s": E / ms_g * 1e3, "loss": float(gstep.loss.item())}
    except Exception as e:                                    # reported, never fatal for the main line
        out["cuda_graph"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if workload == "c2":
        try:
            out["subgraph_regime"] = subgraph_regime_leg(wl, dev)
        except Exception as e:
            out["subgraph_regime"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


def subgraph_regime_leg(wl, dev, batch_size=32):
    """The reference's OWN training regime on configs[1] (`pangnn.py --simulate_dataset 10000 2 0.5 10 3 --train -b 32`:
    one sub-graph per ortholog group, ~285 scored edges per step; SURVEY F7): ms per batch of the eager step (device
    collation) and of the same step replayed as one CUDA graph per size bucket (pangnn_b200.graphs.GraphedBatchStep)."""
    import gc, tempfile
    from pangnn_b200 import ops, setup, train
    from pangnn_b200.data import DeviceLoader
    from pangnn_b200.graphs import GraphedBatchStep
    n, G, f, frags, shuf = wl["sim"]
    setup.reset()
    ops.clear_cache()
    tmp = tempfile.mkdtemp(prefix="pangnn_bench_")
    argv = ["--simulate_dataset", str(n), str(G), str(f), str(frags), str(shuf), "--train", "-e", "0", "-b", str(batch_size),
            "-o", tmp, "-m", os.path.join(tmp, "absent.pkl"), "--seed", "0"]
    t0 = time.perf_counter()
    res = train.run(setup.parse(argv), device=str(dev))
    build_s = time.perf_counter() - t0
    ds, model = res["dataset"], res["model"]
    pw = float(ds.class_balance)
    loader = DeviceLoader(ds.train, batch_size=batch_size, shuffle=True, device=dev, seed=0)

    def epoch(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        nb = ne = 0
        for packed, ids, ids_dev in loader.iter_ids():
            ne += fn(packed, ids, ids_dev)
            nb += 1
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / max(nb, 1) * 1e3, nb, ne

    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def eager(packed, ids, ids_dev):
        b = packed.collate(ids, ids_dev)
        opt.zero_grad(set_to_none=True)
        loss, logits = model.forward_loss(b, pw)
        loss.backward()
        opt.step()
        loss.item()                                          # pangnn.py:218 reads the loss every step
        return int(logits.numel())
    epoch(eager)
    ms_eager, nb, ne = epoch(eager)
    del opt
    gc.collect()
    gopt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
    stepper = GraphedBatchStep(model, gopt, pw)

    def graphed(packed, ids, ids_dev):
        loss, logits = stepper.step_ids(packed, ids, ids_dev)
        loss.item()
        return int(logits.numel())
    epoch(graphed)                                           # captures the buckets
    epoch(graphed)
    ms_graph, _, _ = epoch(graphed)
    setup.reset()
    ops.clear_cache()
    return {"regime": f"-b {batch_size} sub-graph batches, {len(ds.train)} sub-graphs, {ne / max(nb, 1):.0f} scored edges per batch",
            "dataset_build_s": build_s, "eager_ms_per_batch": ms_eager, "cuda_graph_ms_per_batch": ms_graph,
            "cuda_graph_scored_edges_per_s": ne / max(nb, 1) / ms_graph * 1e3, "buckets": len(stepper.buckets),
            "stats": dict(stepper.stats)}


def weak_scaling_fraction(n, G0, f0, G):
    """--simulate_dataset's `fraction_pos_edges` for a G-genome pan-genome that keeps the per-gene
    negative-candidate mean m of the (G0, f0) workload (src/simulate.py:120-129 ties m to G)."""
    from pangnn_b200.simulate import negatives_mean
    m0 = negatives_mean(n, G0, f0)
    f = 1.0 / (1.0 + 2.0 * (m0 + 0.5) / (G - 1))
    assert negatives_mean(n, G, f) == m0, (m0, negatives_mean(n, G, f))
    return f


def partitioned_arm(a, wl, world, rank, local, dev):
    """N > 1: ONE simulated pan-genome of G0 * N genomes, node set partitioned by genome (rank r owns
    genomes [r G0, (r+1) G0)), halo rows exchanged once per layer over NVLink peer memory (or NCCL), weight
    gradients all-reduced once per step (pangnn_b200/dist.py).  Weak scaling: genomes per GPU fixed.  The
    line also carries configs[3] (C4, --categorical_node, G = 20 fixed: strong scaling) as ``secondary``."""
    import torch.distributed as dist
    from pangnn_b200 import ops, setup
    # ---- parity gate: the transport about to be timed must reproduce the reference-derived goldens at THIS world
    #      size (and the single-GPU path on a simulated slab) before any number is taken; rc 3 on failure
    gate = None
    if not a.no_gate:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import parity_gate
        gate = parity_gate.run(rank, world, dev)
        setup.reset()
        for k, v in wl["flags"].items():
            setattr(setup.args, k, v)
        ops.clear_cache()
    line = partition_leg(a, wl, world, rank, local, dev, a.steps, a.warmup, full=not a.no_e2e, device_sim=a.device_sim)
    secondary = None
    if a.workload == "c3" and not a.no_secondary:
        torch.cuda.empty_cache()
        wl4 = WORKLOADS["c4"]
        setup.reset()
        for k, v in wl4["flags"].items():
            setattr(setup.args, k, v)
        ops.clear_cache()
        try:
            sec = partition_leg(a, wl4, world, rank, local, dev, steps=5, warmup=3, full=False, device_sim=True)
            if rank == 0:
                secondary = {k: sec[k] for k in ("value", "unit", "ms_per_step", "scaling", "inference_edges_per_s", "steps")}
                secondary.update(metric="train_edges_per_s", workload=sec["config"]["workload"], total=sec["config"]["total"],
                                 per_gpu=sec["config"]["per_gpu"], parallelism=sec["config"]["parallelism"],
                                 preprocess_s=sec["config"]["preprocess_s"], input="device Philox generator (pangnn_simulate_edges)")
        except Exception as e:                                   # reported, never fatal for the main line
            secondary = {"workload": WORKLOADS["c4"]["desc"], "error": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0:
        line["parity_gate"] = gate
        line["secondary"] = secondary
        emit(line)
    dist.destroy_process_group()


def partition_leg(a, wl, world, rank, local, dev, steps, warmup, full, device_sim):
    """One partitioned workload: build, warm-up, timed training steps, inference; with ``full`` also the end-to-end
    leg and the roofline kernel.  -> the JSON line (dict) on every rank."""
    import torch.distributed as dist
    from pangnn_b200 import dist as pdist, ops, setup
    from pangnn_b200.gnn import AlternateGCN
    flags = setup.args
    n, G0, f0, frags, shuf = wl["sim"]
    if wl.get("fixed_G"):                                         # strong scaling: the configuration as published
        G, f = G0, f0
    else:
        G = G0 * world
        f = weak_scaling_fraction(n, G0, f0, G)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pg = pdist.PartitionedGraph.from_simulation(n, G, f, frags, shuf, rank, world, dev, seed=0, device_generator=device_sim)
    torch.cuda.synchronize()
    prep_s = time.perf_counter() - t0
    E_local, E_total = int(pg.y.numel()), pg.num_edges_total
    pw = pg.class_balance
    torch.manual_seed(0)
    cat = bool(getattr(flags, "categorical_node", False))
    model = AlternateGCN(dev, n * G if cat else None, cat).to(dev)
    for p in model.parameters():                                  # same weights on every rank
        dist.broadcast(p.data, 0)
    dm = pdist.DistModel(model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def step(g):
        opt.zero_grad(set_to_none=False)
        loss, _ = dm.forward_loss(g, pw)
        loss.backward()
        dm.allreduce_grads()
        opt.step()
        return loss

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(warmup):
        step(pg)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = ops.LAUNCHES["count"]
    ms = timed(lambda: step(pg), steps)
    launches = ops.LAUNCHES["count"] - l0
    clk = clocks.stop() if rank == 0 else None
    value = E_total * steps / (ms * 1e-3)

    for _ in range(2):
        dm(pg)
    ms_inf = timed(lambda: dm(pg), steps)
    halo = torch.tensor([float(pg.conv.plan.n_halo), float(pg.scored.plan.n_halo),
                         float(torch.cuda.max_memory_allocated(dev)) / 2**30], device=dev)
    dist.all_reduce(halo, op=dist.ReduceOp.MAX)
    lg = pg.conv
    Ec = int(lg.gs.num_edges)
    F = flags.hidden_dim
    line = {
        "metric": "train_edges_per_s", "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "strong" if wl.get("fixed_G") else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"] if wl.get("fixed_G") else
                   wl["desc"].replace(f"{n} {G0} {f0}", f"{n} {G} {f:.4f}") +
                   f" — {G0} genomes per GPU; fraction_pos_edges chosen so that the per-gene negative mean m stays that of the 1-GPU workload",
                   "total": {"N": n * G, "E_scored": E_total},
                   "per_gpu": {"N": pg.n_own, "E_scored": E_local, "E_conv": Ec,
                               "halo_rows_conv": int(halo[0].item()), "halo_rows_scorer": int(halo[1].item()),
                               "max_memory_allocated_gib": round(float(halo[2].item()), 2)},
                   "step": "whole-graph fwd + BCE(pos_weight) + bwd + Adam (fused scorer/loss kernel)",
                   "l2": "inputs larger than L2 (no flush needed)" if pg.n_own * F * 4 > 126e6 else "graph fits in L2; not flushed",
                   "parallelism": f"genome partition x{world}: halo rows exchanged per layer ("
                                  + ("NVLink peer memory: pushed from the tcgen05 GEMM epilogue into the neighbours' symmetric "
                                     "buffers, halo gradients pulled from them" if pg.conv.plan.p2p is not None
                                     else "NCCL grouped send/recv")
                                  + "), weight-gradient all-reduce (NCCL) once per step",
                   "preprocess_s": prep_s,
                   "input": "device Philox generator (pangnn_simulate_edges)" if device_sim else "host generator (numpy)"},
        "inference_edges_per_s": E_total * steps / (ms_inf * 1e-3),
        "gpu_launches": launches, "clocks": clk, "cpu_baseline": None,
    }
    if not full:
        del pg, dm, model, opt
        return line

    # ---- e2e: every rank's LOCAL batch from pinned host buffers (edge lists in own + halo ids,
    # weights, labels), CSR x2 + gcn_norm (incl. the `dis` halo exchange) rebuilt per step
    host = pg.to_host_pinned()
    h2d = torch.tensor([float(host.nbytes)], device=dev)
    dist.all_reduce(h2d)
    e2e_steps = max(3, min(steps, 10))

    def e2e_run(k):
        """k steps, each from this rank's pinned host batch; copy + CSR builds of step i+1 overlap step i."""
        main = torch.cuda.current_stream()
        pending = pg.prefetch_from(host, dev, main)
        for i in range(k):
            g, ev = pending
            main.wait_event(ev)
            loss = step(g)
            pending = pg.prefetch_from(host, dev, main) if i + 1 < k else None
            loss.item()
    e2e_run(3)
    reps = [timed(lambda: e2e_run(e2e_steps), 1) / e2e_steps for _ in range(5)]
    ms_e2e = float(np.median(reps))
    e2e_val = E_total / (ms_e2e * 1e-3)

    # ---- roofline kernel on this rank's conv graph (rows = owned nodes, sources = own + halo)
    val_dst, _ = lg.norm(True)
    xin = torch.randn(lg.n_ext, F, device=dev)
    out = torch.empty(lg.n_own, F, device=dev)
    bias = torch.zeros(F, device=dev)
    agg = lambda: ops.gcn_aggregate(lg.gs.dst.rowptr, lg.gs.dst.col, val_dst, xin, lg.n_own, bias, ops.ACT_ELU, out=out)
    for _ in range(3):
        agg()
    ms_agg = timed(agg, 20) / 20
    abytes = agg_bytes(Ec, lg.n_own, F)
    peak, peak_src = peaks()
    achieved = abytes / (ms_agg * 1e-3) / 1e9
    line["e2e"] = {"value": e2e_val, "unit": "edges/s", "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": 4 * world,
                   "ms_per_step": ms_e2e, "steps": e2e_steps, "repetitions_ms_per_step": reps,
                   "includes": "per rank: H2D of the local batch (int64 edge lists, weights, labels), CSR build x2 orientations, "
                               "gcn_norm with its halo exchange, step, loss.item(); halo plans are kept; copy + CSR builds of step i+1 "
                               "overlap step i on side streams (one batch of look-ahead); median of 5 repetitions"}
    line["roofline"] = {"bound": "hbm", "kernel": f"gcn_aggregate F={F} (+bias+ELU), rank 0's partition", "achieved": achieved,
                        "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "traffic": None,
                        "algorithmic_bytes": abytes, "us_per_launch": ms_agg * 1e3, "timed": "alone, burst peak"}
    del pg, dm, model, opt, host
    return line


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpu, E = cpu_arm(a.workload, steps=a.steps, warmup=max(1, min(a.warmup, 2)))
    wl = WORKLOADS[a.workload]
    line = {"impl": "reference", "metric": "train_edges_per_s", "value": cpu["value"], "unit": "edges/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": cpu["steps"], "warmup": a.warmup,
            "ms_per_step": cpu["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "note": "reference model (oracle port: torch CPU index_select/index_add_ GCNConv, "
                       "as src/gnn.py over restated PyG) on the host cores, bounded sample"},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def emit(line):
    """The contract is ONE JSON line on stdout; libraries (NCCL banner) also write to fd 1, so fd 1
    is pointed at stderr for the whole run and restored only for this line."""
    sys.stdout.flush()
    os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no_cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no_gate", action="store_true", help="N > 1: skip the multi-GPU parity gate (development only)")
    ap.add_argument("--no_e2e", action="store_true",
                    help="N > 1: resident step and inference only (the end-to-end leg keeps two batches alive: look-ahead)")
    ap.add_argument("--no_secondary", action="store_true", help="skip the secondary workload leg (c2 at N = 1, c4 at N > 1)")
    ap.add_argument("--device_sim", action="store_true",
                    help="N > 1: generate the main workload's hit table with the device Philox generator too")
    ap.add_argument("--profile", action="store_true",
                    help="ncu mode: warm-up + timed steps + aggregation loop only (no e2e / inference / CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="single GPU: write the loss, logits, parameters and gradients of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: the single-GPU path only (--impl ours, one process)")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        reference_arm(a)
    else:
        gpu_arm(a)
