#!/usr/bin/env python
"""Headline benchmark: SPGNN-3 (st_pgat_spgnn_3) training step on synthetic airway-tree batches.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--trees B] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one iteration of the reference's GCN_STEPS loop (job_runner.py:1892-1919) over one batch of B trees
per GPU: zero_grad, forward (7 GATConv + head, train mode with dropout), masked weighted CE, backward,
gradient all-reduce (N > 1) and the SGD-momentum update.  Prints ONE JSON line (rank 0).

  value     graphs/s, whole job, batch resident in HBM (CUDA events, max over ranks)
  e2e       graphs/s through the public API from pinned HOST buffers: H2D of the scan batch in the loader's lossless
            wire format (zero-suppressed fvs, edge lists, fvs_out, labels), device decode + graph build + positional
            encoding + the training step, D2H of the loss — every step.  e2e_dense_format: the same with the dense
            stage-1 layout (adj / fvs as in the pickles); h2d_only: the copy alone
  roofline  dominant kernel by time share, algorithmic flops (or bytes) per launch / CUDA-event duration
  cpu_baseline  the oracle (PyTorch-CPU restatement of the DGL op sequence; DGL itself is not installable) on
            a bounded sample of the same workload, on this box's host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HEADLINE = "st_pgat_spgnn_3"                           # BASELINE.json configs[1]; the other presets are extra lines
LR, MOMENTUM = 5e-4, 0.9                               # train.py:14 default lr; st_pgat_spgnn_3.py:124-128
SEED = 1234
ORACLE_KIND = {"models.GATNet": "gat", "models.GCNNet": "gcn", "models.GINNet": "gin", "models.SAGENet": "sage",
               "models.GATPositionSPGNNNet": "spgnn"}


def workload(name):
    """(model kwargs, oracle kind, dotted class name, SAMPLING_RATE) of an exp_settings preset (SURVEY.md App. A)."""
    from spgnn_b200.settings import PRESETS
    st = PRESETS[name]
    model = dict(st["MODEL"])
    method = model.pop("method")
    return model, ORACLE_KIND[method], method, st["SAMPLING_RATE"]


def metric_name(name):
    return "spgnn3_train_graphs_per_s" if name == HEADLINE else f"{name}_train_graphs_per_s"


def workload_text(name, ragged=False):
    return f"{name} train step (fwd+bwd+SGD), synthetic bifurcating airway trees " + \
        ("n in [241, 361], mean 301" if ragged else "n=301")


# C-ABI call -> its dominant kernel in the ncu capture (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py)
NCU_KERNEL = {"planes_linear_bwd_weight": "tn_planes_kernel", "planes_linear_fwd": "nt_planes_kernel",
              "planes_linear_bwd_input": "nt_planes_kernel", "wide_linear": "wide_kernel",
              "gat_layer_fwd": "gat_tree_fwd_kernel", "gat_layer_bwd": "gat_tree_bwd_kernel",
              "gat_aggx_fwd": "aggx_fwd_kernel", "split_planes": "split_planes_kernel"}


def ncu_traffic(op, trees):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, mean over the launches of one training
    step) of the kernel behind C-ABI call `op`, from the committed ncu --set full capture; None when there is no
    capture at this batch size."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    k = d.get("kernels", {}).get(NCU_KERNEL.get(op, ""))
    if not k or d.get("trees") != trees or d.get("csrc_sha16") != csrc_sha16():
        return None                     # no capture at this size, or captured from other kernel sources: stale
    return k["dram_bytes_per_launch"]


def csrc_sha16():
    """sha256 (first 16 hex) over the CUDA sources: profiles/ncu_traffic.json carries the value of the build it was
    captured from (scripts/ncu_traffic.py) and is ignored when the kernels have changed since."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "spgnn_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                    str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(int(float(r[0])) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        mx = max((int(float(r[1])) for r in self.rows if r[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_oracle_rate(trees, steps, warmup, threads, name=HEADLINE):
    """graphs/s of the CPU oracle on one train step (fwd+bwd+SGD) of preset `name` over `trees` synthetic trees
    (same generator, same model)."""
    import numpy as np
    import torch
    from oracle import dgl_ops, models as om, pe as ope
    from spgnn_b200 import synth
    torch.set_num_threads(threads)
    model, kind, _, rate = workload(name)
    scans = synth.make_scans(0, trees, seed=SEED)
    gs = []
    for s in scans:
        g = dgl_ops.graph_from_adj(s.adj)
        g.ndata["fvs"] = torch.from_numpy(s.fvs)
        if kind == "spgnn":
            anc = ope.anchors_39(s.fvs_out, s.adj)
            g.ndata["pos_enc"] = torch.from_numpy(ope.dist_pos_enc(s.adj, anc)[0])
        gs.append(g)
    bg = dgl_ops.batch(gs)
    y = torch.from_numpy(np.concatenate([s.labels for s in scans]))
    torch.manual_seed(0)
    net = om.GNNNet(kind, model)
    net.init_like_reference()
    net.train()
    opt = torch.optim.SGD(net.parameters(), lr=LR, momentum=MOMENTUM)
    cw = torch.tensor([0.2] + [0.8] * 21)
    gen = torch.Generator().manual_seed(0)

    def step():
        opt.zero_grad()
        mask = (y != 0) | (torch.rand(y.numel(), generator=gen) < rate)
        out = net(bg)
        loss = om.cross_entropy_masked(out[0], y, mask, cw)
        loss.backward()
        opt.step()
        return float(loss.detach())

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return trees / dt, dt, int(bg.num_nodes)


def cpu_config0_and_pe(threads):
    """BASELINE.json configs[0] as stated — st_gat_3 INFERENCE on the CPU over 64 synthetic trees, one graph at a time
    as GCNTest.run does (job_runner.py:840-911: graph → logits → softmax → per-class arg-max) — and BASELINE.md C3:
    the reference's host-side positional encoding of one tree (job_runner.py:1759-1777: networkx all-pairs shortest
    paths + diameter + the distal-leaf search, literal networkx calls), which dominates its wall clock."""
    import numpy as np
    import torch
    from oracle import dgl_ops, models as om, pe as ope
    from spgnn_b200 import synth
    torch.set_num_threads(threads)
    model, kind, _, _ = workload("st_gat_3")
    scans = synth.make_scans(0, 64, seed=SEED, ragged=True)
    torch.manual_seed(0)
    net = om.GNNNet(kind, model)
    net.init_like_reference()
    net.eval()
    graphs = []
    for s in scans:
        g = dgl_ops.graph_from_adj(s.adj)
        g.ndata["fvs"] = torch.from_numpy(s.fvs)
        graphs.append(g)
    with torch.no_grad():
        net(graphs[0])
        t0 = time.perf_counter()
        for g in graphs:
            om.decide_per_tree(net(g)[0], g.batch_num_nodes())
        dt = time.perf_counter() - t0
    out = {"gat3_eval_graphs_per_s": len(graphs) / dt, "gat3_eval_ms_per_graph": dt / len(graphs) * 1e3,
           "gat3_eval_what": "st_gat_3 eval, 64 ragged synthetic trees, one graph per forward (BASELINE config 0)"}
    try:
        import networkx as nx
        t0 = time.perf_counter()
        for s in scans[:3]:
            a = np.array(s.adj, dtype=np.int64)
            np.fill_diagonal(a, 0)
            G = nx.Graph(a)
            dict(nx.all_pairs_shortest_path_length(G))
            nx.diameter(G)
            ope.anchors_39(s.fvs_out, s.adj, tie_rule="reference")
        out["networkx_pe_ms_per_tree"] = (time.perf_counter() - t0) / 3 * 1e3
    except Exception as e:                                  # networkx missing on the box: say so
        out["networkx_pe_ms_per_tree"] = None
        out["networkx_pe_error"] = repr(e)
    return out


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle restatement; DGL is not installable) on host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    trees = args.cpu_trees
    rate, dt, nodes = cpu_oracle_rate(trees, max(1, args.steps), max(1, min(args.warmup, 2)), cores, args.workload)
    extra = cpu_config0_and_pe(cores) if args.workload == HEADLINE else None
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": rate, "unit": "graphs/s",
        "n_gpus": args.gpus, "steps": max(1, args.steps), "warmup": max(1, min(args.warmup, 2)),
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "nodes_per_s": rate * nodes / trees,
        "config": {"workload": workload_text(args.workload), "trees_per_step": trees, "nodes_per_step": nodes},
        "cpu_baseline": {"value": rate, "unit": "graphs/s", "cores": cores, "kind": "port",
                         "sample": f"{trees} trees/step (bounded sample of the 4096-tree batch); oracle = PyTorch-CPU "
                                   f"restatement of the DGL-0.7 op sequence, torch threads = {cores}"},
        "e2e": {"value": rate, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_other_configs": extra,
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
DUMP_LOGIT_ROWS = 1 << 16


def dump_outputs(out_dir, net, loss, logits):
    """What the last timed train step left to its caller, as float32 .npy files (about 26 MB for the headline), so
    that two builds run with the same arguments can be compared output for output:
      loss.npy           the step's masked weighted cross-entropy (scalar)
      logits_sample.npy  forward logits of DUMP_LOGIT_ROWS nodes drawn without replacement by numpy's default_rng(SEED),
                         in ascending node order (the full [N, 22] tensor is 108 MB at 4096 trees)
      params.npy         every parameter after the step's SGD update, flattened in net.parameters() order
      grads.npy          the step's gradients in the same layout (zeros for a parameter without one)
    Two runs of one build are not bit-identical: on a B200 (1000 W limit) the headline's loss matched exactly, the
    logits to 5e-6 and the gradients to 8e-6 of their largest entry, so compare with a tolerance."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = logits.shape[0]
    rows = np.sort(np.random.default_rng(SEED).choice(n, size=min(n, DUMP_LOGIT_ROWS), replace=False))
    params = list(net.parameters())
    arrays = {
        "loss": loss.reshape(()),
        "logits_sample": logits[torch.from_numpy(rows).to(logits.device)],
        "params": torch.cat([p.detach().reshape(-1) for p in params]),
        "grads": torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1)
                            for p in params]),
    }
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from spgnn_b200 import models as sm, ops, pe as spe, runner, synth_device
    from spgnn_b200._lib import lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gemm_mode is not None:
        ops.GEMM_MODE = args.gemm_mode
    B = args.trees
    L = lib()

    # -------- synthetic batch on device (this rank's shard of the global batch), positional encoding on device
    batch = synth_device.make_batch(first_tree=rank * B, count=B, seed=SEED, ragged=args.ragged)
    g = batch.graph
    model, kind, method, rate = workload(args.workload)
    pe_dim = model.get("pos_enc_dim", 0) if kind == "spgnn" else 0
    if pe_dim:
        spe.distance_pos_enc(g, pos_enc_dim=pe_dim)
    N, E = g.num_nodes, g.num_edges

    torch.manual_seed(0)
    net = getattr(sm, method.split(".")[-1])(**model).to(dev)
    net.init()
    net.train()
    net.set_gcn_only()
    opt = runner.FlatSGD(net.parameters(), lr=LR, momentum=MOMENTUM)
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device=dev)
    ops.manual_seed(SEED)

    def step():
        return runner.train_step(net, g, opt, cw, rate)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    last = {}
    hook = None
    if args.dump_outputs and rank == 0:          # keeps a reference to each step's logits, no copy inside the timed loop
        hook = net.register_forward_hook(lambda m, i, o: last.__setitem__("logits", o[0].detach()))
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = L.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    barrier()
    if hook is not None:
        hook.remove()
        dump_outputs(args.dump_outputs, net, loss, last.pop("logits"))
    ms = e0.elapsed_time(e1) / args.steps
    launches = L.launch_count() - l0                     # this library's kernel launches inside the timed region
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    loss_val = float(loss.item())

    # -------- inference (the metric's "infer" half): eval-mode forward + per-tree decision, no collectives
    net.eval()
    for _ in range(2):
        runner.infer(net, g)
    barrier()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for _ in range(args.steps):
        runner.infer(net, g)
    i1.record()
    barrier()
    t = torch.tensor([i0.elapsed_time(i1) / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    infer_ms = float(t.item())
    net.train()

    # -------- BASELINE config 5: 1M synthetic trees streamed — every step takes a NEW batch generated on device from
    # (seed, global tree index): synthesis, CSR/CSC build and positional encoding are inside the timed region
    stream_line = None
    if args.stream_steps > 0:
        def stream_step(i):
            first = (i * world + rank) * B                   # contiguous blocks of global tree indices per rank
            bb = synth_device.make_batch(first_tree=first, count=B, seed=SEED, ragged=args.ragged)
            if pe_dim:
                spe.distance_pos_enc(bb.graph, pos_enc_dim=pe_dim)
            return runner.train_step(net, bb.graph, opt, cw, rate)

        stream_step(0)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(args.stream_steps):
            stream_step(1 + i)
        s1.record()
        barrier()
        t = torch.tensor([s0.elapsed_time(s1) / args.stream_steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sms = float(t.item())
        rate_s = world * B / (sms / 1e3)
        stream_line = {"value": rate_s, "unit": "graphs/s", "ms_per_step": sms, "steps": args.stream_steps,
                       "seconds_per_1M_trees": 1e6 / rate_s,
                       "what": "every step: device synthesis of a fresh 4096-tree batch per GPU from (seed, global tree "
                               "index) + graph build + positional encoding + train step (BASELINE config 5)"}

    # -------- per-kernel profile pass (CUDA events around every C-ABI call; separate from the timed region)
    # Every rank takes these steps (a step holds two collectives: the CE sums and the gradient all-reduce); only rank
    # 0 keeps the per-call events.
    roof, roof_agg, shares, abi_ms = None, None, None, None
    if rank == 0:
        L.profile = []
    n_prof = max(1, min(3, args.steps))
    for _ in range(n_prof):
        step()
    barrier()
    if rank == 0:
        prof, L.profile = L.profile, None
        agg = {}
        for name, key, a, b in prof:
            d = agg.setdefault(name, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0, "impl": 0.0})
            d["ms"] += a.elapsed_time(b)
            d["n"] += 1
            if key:
                d[key[0]] += key[1]
                d["impl"] += key[2] if len(key) > 2 else key[1]      # bytes the implementation moves by design
        total = sum(d["ms"] for d in agg.values())
        shares = {k: round(d["ms"] / total, 4) for k, d in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])[:8]}
        abi_ms = total / n_prof          # GPU time inside this library's calls per step (the rest is launch gaps)
        pk = peaks()

        def traffic(name):
            return ncu_traffic(name, B) if args.workload == HEADLINE else None     # the capture is of the headline

        def roofline(name):
            d = agg.get(name)
            if not d or d["ms"] == 0:
                return None
            sec = d["ms"] / 1e3
            if d["flops"] == 0 and d["bytes"] == 0:
                return {"kernel": name, "bound": None, "achieved": None, "launches": d["n"], "avg_ms": d["ms"] / d["n"],
                        "share_of_step": d["ms"] / total, "note": "no algorithmic-work figure registered for this call"}
            if d["flops"] > 0:
                ach = d["flops"] / sec / 1e12
                return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                        "frac": ach / pk["tf_sust"], "traffic": traffic(name), "launches": d["n"],
                        "avg_ms": d["ms"] / d["n"],
                        "peak_source": pk["src"] + " bf16 dense, sustained", "share_of_step": d["ms"] / total,
                        "note": "fp32-accurate projection; algorithmic flops 2*M*N*K"}
            ach = d["bytes"] / sec / 1e9
            return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": ach / pk["hbm"], "traffic": traffic(name), "launches": d["n"],
                    "avg_ms": d["ms"] / d["n"], "algorithmic_bytes_per_launch": d["bytes"] / d["n"],
                    "implementation_bytes_per_launch": d["impl"] / d["n"],
                    "frac_implementation_bytes": d["impl"] / sec / 1e9 / pk["hbm"],
                    "peak_source": pk["src"] + " copy bandwidth", "share_of_step": d["ms"] / total,
                    "frac_of_nominal_8TBs": ach / 8000.0}
        dominant = max(agg.items(), key=lambda kv: kv[1]["ms"])[0]
        roof = roofline(dominant)
        agg_calls = {"gat": ("gat_layer_fwd", "gat_layer_bwd"), "spgnn": ("gat_layer_fwd", "gat_layer_bwd"),
                     "gcn": ("spmm", None), "gin": ("spmm", None), "sage": ("sage_maxpool_fwd", "sage_maxpool_bwd")}[kind]
        roof_agg = {"fwd": roofline(agg_calls[0]), "bwd": roofline(agg_calls[1]) if agg_calls[1] else None}
        if agg_calls[1] is None and roof_agg["fwd"]:
            roof_agg["fwd"]["note"] = "forward and backward (transposed graph) aggregations are the same call"

    # -------- end to end through the public API from pinned host buffers
    e2e = e2e_dense = h2d_only = None
    if not args.no_e2e:
        def e2e_run(hb, n):
            # public API: DeviceBatchLoader copies batch i+1 from pinned host memory on a copy stream while step i
            # computes; EVERY step's inputs cross PCIe inside the timed region and every step's loss is read back.
            for gg in runner.DeviceBatchLoader((hb for _ in range(n)), pos_enc_dim=pe_dim, device=dev):
                ls = runner.train_step(net, gg, opt, cw, rate)
                float(ls.item())                         # D2H read of the loss
                del gg

        def e2e_measure(hb, n, what):
            # 3 untimed steps: the first end-to-end steps grow the allocator's pools (two batches are alive at once:
            # cudaMalloc of multi-GB blocks serialises with the GPU) — steady state from the third step on
            torch.cuda.empty_cache()                     # pools shaped by the end-to-end pattern, not by the legs before
            e2e_run(hb, 3)
            barrier()
            t0 = time.perf_counter()
            e2e_run(hb, n)
            barrier()
            t = torch.tensor([(time.perf_counter() - t0) / n], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return {"value": world * B / float(t.item()), "unit": "graphs/s", "h2d_bytes_per_step": hb.nbytes(),
                    "d2h_bytes_per_step": 4, "ms_per_step": float(t.item()) * 1e3, "steps": n, "host_format": what,
                    "pipeline": "H2D of batch i+1 overlaps step i (copy stream); first batch's copy is inside the "
                                "timed region"}

        # the loader's wire format (csrc/wire.cu): fvs zero-suppressed (a ReLU output), adjacency as edge lists —
        # lossless, decoded on the device into the same tensors; packing happens once when a batch is read
        hb = runner.host_batch_from_graph(g, packed=True)
        e2e = e2e_measure(hb, args.e2e_steps, "packed: zero-suppressed fvs + int32 edge lists + uint8 labels (lossless)")
        e2e["host_pack_seconds_per_batch"] = hb.pack_seconds
        e2e["host_pack_threads"] = os.cpu_count()
        # the link alone: the same buffers copied with no compute behind them (names the limiter of the e2e number)
        bufs = None
        barrier()
        t0 = time.perf_counter()
        for _ in range(5):
            bufs = runner._upload(hb, dev)
        barrier()
        t = torch.tensor([(time.perf_counter() - t0) / 5], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        h2d_only = {"gb_per_s_per_gpu": hb.nbytes() / float(t.item()) / 1e9, "ms_per_batch": float(t.item()) * 1e3,
                    "bytes": hb.nbytes(), "ranks_copying_at_once": world}
        del bufs, hb
        # the same step fed with the dense stage-1 layout (one fp32 [N, 1024] + one uint8 [n, n] per scan): 5.5 GB/step
        hbd = runner.host_batch_from_graph(g, packed=False)
        e2e_dense = e2e_measure(hbd, max(3, args.e2e_steps // 3), "dense stage-1 pickle layout")
        del hbd

    # -------- the reference's own regime (TRAIN_BATCH_SIZE = 64 scans, GCN_STEPS = 300 steps on one batch,
    # job_runner.py:1892-1919; inference one scan at a time, :840-911): launch-bound, so the step is replayed from a
    # CUDA graph (runner.GraphedTrainStep)
    small = None
    if rank == 0 and world == 1 and not args.no_small and B > 64:
        sb = synth_device.make_batch(first_tree=0, count=64, seed=SEED, ragged=True).graph
        if pe_dim:
            spe.distance_pos_enc(sb, pos_enc_dim=pe_dim)

        def timed(fn, n):
            fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n, (time.perf_counter() - t0) / n * 1e3

        eager_ms, eager_wall = timed(lambda: runner.train_step(net, sb, opt, cw, rate), 30)
        gs = runner.GraphedTrainStep(net, sb, opt, cw, rate, warmup=2)
        graph_ms, graph_wall = timed(gs, 100)
        gs.reset_salt()
        one = synth_device.make_batch(first_tree=7, count=1, seed=SEED, ragged=True).graph
        if pe_dim:
            spe.distance_pos_enc(one, pos_enc_dim=pe_dim)
        net.eval()
        inf_ms, inf_wall = timed(lambda: runner.infer(net, one), 30)
        net.train()
        small = {"trees": 64, "nodes": sb.num_nodes, "train_step_eager_ms": eager_ms, "train_step_cuda_graph_ms": graph_ms,
                 "train_graphs_per_s_cuda_graph": 64 / (graph_ms / 1e3), "train_graphs_per_s_eager": 64 / (eager_ms / 1e3),
                 "single_scan_inference_ms": inf_wall, "single_scan_inference_gpu_ms": inf_ms,
                 "what": "64 ragged trees per step (the reference's TRAIN_BATCH_SIZE); CUDA-graph replay of the whole "
                         "train step with per-replay dropout/sampling masks; inference latency of ONE scan (graph → "
                         "logits → per-class arg-max), host wall clock"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:     # reported at N=1 only (at N>1 the ranks share the host cores)
        cores = os.cpu_count() or 1
        crate, dt, nodes = cpu_oracle_rate(args.cpu_trees, 2, 1, cores, args.workload)
        cpu = {"value": crate, "unit": "graphs/s", "cores": cores, "kind": "port",
               "sample": f"{args.cpu_trees} trees/step x 2 steps (+1 warm-up) of the same {args.workload} train step; oracle = "
                         f"PyTorch-CPU restatement of the DGL-0.7 op sequence (DGL not installable), {cores} threads",
               "ms_per_step": dt * 1e3}

    if rank == 0:
        gps = world * B / (ms / 1e3)
        line = {
            "metric": metric_name(args.workload), "value": gps, "unit": "graphs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "nodes_per_s": gps * N / B,
            "infer": {"value": world * B / (infer_ms / 1e3), "unit": "graphs/s", "ms_per_step": infer_ms,
                      "nodes_per_s": world * N / (infer_ms / 1e3),
                      "what": "eval-mode forward (7 GATConv + head) + per-tree per-class arg-max, batch resident in HBM"},
            "config": {"workload": workload_text(args.workload, args.ragged),
                       "trees_per_gpu": B, "nodes_per_gpu": N, "edges_per_gpu": E, "parallelism": f"dp{world} by graph",
                       "l2": "inputs (5.2 GB/GPU) larger than L2, no flush needed", "gemm_mode": ops.GEMM_MODE,
                       "loss": loss_val},
            "roofline": roof, "roofline_agg": roof_agg, "kernel_time_shares": shares, "abi_ms_per_step": abi_ms,
            "cpu_baseline": cpu, "e2e": e2e, "e2e_dense_format": e2e_dense, "h2d_only": h2d_only,
            "stream_1M_trees": stream_line, "small_batch": small, "gpu_launches": int(launches),
            "gpu_launches_per_step": int(launches) // args.steps, "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()                      # rank 0 may still be timing the CPU baseline: leave together
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--trees", type=int, default=4096, help="trees per GPU per step (BASELINE config 2)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=HEADLINE, help="exp_settings preset; the default is the headline "
                    "(BASELINE.json configs[1]); st_gat_3|st_gat_6|st_gat_6_nr|st_gcn_3|st_gin_3|st_sage_3 give the "
                    "extra lines of configs[2..3] (profiles/), never the driver's bench line")
    ap.add_argument("--cpu-trees", type=int, default=64)
    ap.add_argument("--e2e-steps", type=int, default=40, help="end-to-end steps (the first batch's H2D copy is inside the "
                    "timed region and is not overlapped by anything: 51 ms spread over these steps)")
    ap.add_argument("--ragged", action="store_true", help="tree sizes n in [241, 361] (mean 301) instead of n = 301")
    ap.add_argument("--stream-steps", type=int, default=10, help="extra steps on freshly generated batches (config 5)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-small", action="store_true", help="skip the 64-tree / single-scan latency leg")
    ap.add_argument("--gemm-mode", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last "
                    "one computed (loss, a fixed sample of logits, updated parameters, gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
