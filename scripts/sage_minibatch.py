"""GCNTrainSAGE's mini-batch (st_sage_3): the torch neighbour sampler against the device sampler, one JSON line per
(batch size, sampler).

    python scripts/sage_minibatch.py [--scans 2 64] [--batches 30] [--repeats 5] [--out FILE]

For a GCNTrainSAGE batch of ``--scans`` synthetic ragged scans (the runner's input: 2 scans at st_sage_3's
TRAIN_BATCH_SIZE; 64 scans for a larger graph): mini-batches of NODE_BATCH_SIZE = 64 seeds from a random 30 % of the
nodes (node_sample_rate), fanouts node_ks = [2, 2, 2, 2].  Per sampler:
  * ms per mini-batch of the sampler alone (blocks + node-data gathers) and of the whole step (sampler + SAGENet
    forward_batch + class-weighted CE + backward + FlatSGD step), host clock over ``--batches`` mini-batches ending in
    a device synchronise.  The two samplers run alternately, ``--repeats`` times each, in the same process; the line
    gives the median and the spread (min, max) of the repeats;
  * kernel launches per mini-batch of the sampler (torch.profiler, CUDA kernels, in a separate pass) and
    synchronising calls per mini-batch (torch.cuda.set_sync_debug_mode("warn")).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from spgnn_b200 import models as sm, ops, runner, sampling, synth_device  # noqa: E402
from spgnn_b200.settings import PRESETS  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def torch_sampler(fanouts):
    s = sampling.MultiLayerNeighborSampler(fanouts)

    def sample(g, seeds):
        blocks = s.sample_blocks(g, seeds)
        for k, v in g.ndata.items():                         # NodeDataLoader's gathers
            blocks[0].srcdata[k] = v[blocks[0].src_ids]
            blocks[-1].dstdata[k] = v[seeds]
        return blocks
    return sample


def device_sampler(fanouts):
    s = sampling.DeviceBlockSampler(fanouts)
    return lambda g, seeds: s.sample_blocks(g, seeds)


def minibatches(g, n, bs, rate, gen):
    out = []
    while len(out) < n:
        nids = torch.randperm(g.num_nodes, device="cuda", generator=gen)[:int(g.num_nodes * rate)]
        out += [nids[i:i + bs] for i in range(0, nids.numel(), bs)]
    return out[:n]


def run(g, seed_sets, sample, step):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for seeds in seed_sets:
        blocks = sample(g, seeds)
        if step is not None:
            step(blocks)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / len(seed_sets)


def counts(g, seed_sets, sample):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for seeds in seed_sets:
            sample(g, seeds)
        torch.cuda.synchronize()
    kernels = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                  and not e.name.startswith(("Memcpy", "Memset")))
    syncs = 0
    for seeds in seed_sets:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            torch.cuda.set_sync_debug_mode("warn")
            try:
                sample(g, seeds)
            finally:
                torch.cuda.set_sync_debug_mode("default")
        syncs += sum("synchroniz" in str(x.message) for x in w)
    return kernels / len(seed_sets), syncs / len(seed_sets)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, nargs="+", default=[2, 64])
    ap.add_argument("--batches", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    p = PRESETS["st_sage_3"]
    model = {k: v for k, v in p["MODEL"].items() if k != "method"}
    fanouts, rate, bs = model["node_ks"], model["node_sample_rate"], p["NODE_BATCH_SIZE"]
    dev_card = card()
    lines = []
    for scans in args.scans:
        g = synth_device.make_batch(0, scans, ragged=True).graph
        g.max_degree()
        torch.manual_seed(0)
        ops.manual_seed(0)
        net = sm.SAGENet(**model).cuda()
        net.train()
        opt = runner.FlatSGD(net.parameters(), lr=1e-4, momentum=0.9)
        cw = torch.tensor([0.1, 0.2] + [0.8] * 20, device="cuda")

        def step(blocks):
            opt.zero_grad()
            out, _ = net.forward_batch(blocks, blocks[0].srcdata["fvs"])
            ops.masked_cross_entropy(out, blocks[-1].dstdata["y"], cw, rate=1.0).backward()
            opt.step()

        gen = torch.Generator(device="cuda").manual_seed(1)
        seed_sets = minibatches(g, args.batches, bs, rate, gen)
        samplers = {"torch": torch_sampler(fanouts), "device": device_sampler(fanouts)}
        for s in samplers.values():                              # warm-up: modules, allocator, cached norms
            run(g, seed_sets[:3], s, step)
        t = {(k, w): [] for k in samplers for w in ("sampler", "step")}
        for _ in range(args.repeats):
            for name, s in samplers.items():
                t[(name, "sampler")].append(run(g, seed_sets, s, None))
                t[(name, "step")].append(run(g, seed_sets, s, step))
        for name, s in samplers.items():
            kern, syncs = counts(g, seed_sets[:10], s)
            line = dict(script="sage_minibatch", sampler=name, scans=scans, nodes=g.num_nodes, seeds_per_minibatch=bs,
                        fanouts=fanouts, minibatches=len(seed_sets), repeats=args.repeats,
                        sampler_ms_median=round(statistics.median(t[(name, "sampler")]), 4),
                        sampler_ms_min=round(min(t[(name, "sampler")]), 4),
                        sampler_ms_max=round(max(t[(name, "sampler")]), 4),
                        step_ms_median=round(statistics.median(t[(name, "step")]), 4),
                        step_ms_min=round(min(t[(name, "step")]), 4), step_ms_max=round(max(t[(name, "step")]), 4),
                        kernels_per_minibatch=kern, syncs_per_minibatch=syncs, card=dev_card)
            lines.append(line)
            print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
