"""SAGENet (st_sage_3 widths) with each of DGL 0.7's SAGEConv aggregators: one JSON line per aggregator.

    python scripts/sage_aggregators.py [--trees 4096] [--steps 5] [--warmup 2] [--out FILE]

Per aggregator (model kwargs from ``bench.workload("st_sage_3")`` with ``aggregator_type`` overridden):
  * full-batch training step (forward, masked CE, backward, SGD) and eval-mode inference on ``--trees`` synthetic
    bifurcating trees of n = 301, from CUDA events after warm-up; if the training step does not fit in device
    memory the tree count is halved until it does, and the line says at which count it was measured;
  * one sampled mini-batch step (64 seeds, fanouts [2, 2, 2, 2], GCNTrainSAGE's inner step);
  * ``torch.cuda.max_memory_allocated`` over the aggregator's runs;
  * for lstm: the layer-0 reducer (D = 1024) forward + backward on its own, with the time of the cell and dP
    kernels against their algorithmic bytes and of the recurrent planes GEMMs against their flops (events around
    every C-ABI call).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from spgnn_b200 import models as sm, ops, runner, sampling, synth_device  # noqa: E402
from spgnn_b200._lib import lib  # noqa: E402

COPY_PEAK_GBS = 6545.0          # B200 device-to-device copy bandwidth this project measures kernels against


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def full_batch(model, trees, steps, warmup):
    batch = synth_device.make_batch(0, trees, seed=bench.SEED, ragged=False)
    g = batch.graph
    torch.manual_seed(0)
    net = sm.SAGENet(**model).cuda()
    net.init()
    opt = runner.FlatSGD(net.parameters(), lr=bench.LR, momentum=bench.MOMENTUM)
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device="cuda")
    net.train()
    train_ms = timed(lambda: runner.train_step(net, g, opt, cw, 0.05), steps, warmup)
    net.eval()
    with torch.no_grad():
        infer_ms = timed(lambda: net(g), steps, warmup)
    return dict(trees=trees, nodes=g.num_nodes, edges=g.num_edges, train_ms=train_ms, infer_ms=infer_ms,
                train_graphs_per_s=trees / train_ms * 1e3)


def minibatch(model, steps, warmup):
    batch = synth_device.make_batch(0, 64, seed=bench.SEED, ragged=False)
    g = batch.graph
    torch.manual_seed(0)
    net = sm.SAGENet(**model).cuda()
    net.init()
    net.train()
    opt = runner.FlatSGD(net.parameters(), lr=bench.LR, momentum=bench.MOMENTUM)
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(3)
    seeds = torch.randperm(g.num_nodes, device="cuda", generator=gen)[:64]
    blocks = sampling.MultiLayerNeighborSampler([2, 2, 2, 2]).sample_blocks(g, seeds, gen)
    x = g.ndata["fvs"][blocks[0].src_ids]
    y = g.ndata["y"][seeds]

    def step():
        opt.zero_grad()
        out, _ = net.forward_batch(blocks, x)
        ops.masked_cross_entropy(out, y, cw, rate=1.0).backward()
        opt.step()

    return dict(seeds=64, fanouts=[2, 2, 2, 2], step_ms=timed(step, 20 * steps, warmup))


def lstm_layer0(trees, steps):
    """Layer 0's reducer (P [N, 4096] -> [N, 1024]) forward + backward with events around every C-ABI call."""
    g = synth_device.make_batch(0, trees, seed=bench.SEED, ragged=False).graph
    D = 1024
    gen = torch.Generator(device="cuda").manual_seed(1)
    P = (torch.randn(g.num_nodes, 4 * D, device="cuda", generator=gen) * 0.5).requires_grad_()
    W = (torch.randn(4 * D, D, device="cuda", generator=gen) / D ** 0.5).requires_grad_()
    gout = torch.randn(g.num_nodes, D, device="cuda", generator=gen)

    def run():
        ops.LstmReduceFn.apply(P, W, g).backward(gout)

    run()
    torch.cuda.synchronize()
    L = lib()
    L.profile = []
    for _ in range(steps):
        run()
    torch.cuda.synchronize()
    prof, L.profile = L.profile, None
    agg = {}
    for name, key, e0, e1 in prof:
        d = agg.setdefault(name, dict(ms=0.0, n=0, bytes=0.0, flops=0.0))
        d["ms"] += e0.elapsed_time(e1) / steps
        d["n"] += 1
        if key:
            d[key[0]] += key[1] / steps
    out = {}
    for name, d in agg.items():
        r = dict(ms_per_step=d["ms"], launches_per_step=d["n"] / steps)
        if d["bytes"]:
            r["algorithmic_GBs"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9
            r["frac_of_copy_peak"] = r["algorithmic_GBs"] / COPY_PEAK_GBS
        if d["flops"]:
            r["algorithmic_TFs"] = d["flops"] / (d["ms"] * 1e-3) / 1e12
        out[name] = r
    o = ops.lstm_order(g)
    return dict(trees=trees, nodes=g.num_nodes, steps_n_t=o.steps, calls=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--aggs", default="pool,mean,gcn,lstm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sage_aggregators.py measures on a CUDA device; none is available")
    model, _, _, _ = bench.workload("st_sage_3")
    lines = []
    for agg in a.aggs.split(","):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        m = dict(model, aggregator_type=agg)
        trees, fb = a.trees, None
        while fb is None:
            try:
                fb = full_batch(m, trees, a.steps, a.warmup)
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                trees //= 2
        rec = dict(workload="st_sage_3", aggregator_type=agg, card=card(), full_batch=fb,
                   full_batch_fits_requested_trees=trees == a.trees, minibatch=minibatch(m, a.steps, a.warmup),
                   max_memory_allocated_GB=torch.cuda.max_memory_allocated() / 1e9)
        if agg == "lstm":
            torch.cuda.empty_cache()
            rec["lstm_layer0_reducer"] = lstm_layer0(trees, a.steps)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
