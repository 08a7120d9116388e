"""Cost of the device optimisers: one JSON line per measurement.

    python scripts/optimizer_step.py [--iters 200] [--steps 20] [--out FILE]

  * the optimiser step alone on the SPGNN-3 bucket (2,501,078 floats, st_pgat_spgnn_3's parameters with fixed
    random gradients): runner.FlatSGD (momentum 0.9), runner.FlatAdam, FlatAdam as AdamW with amsgrad, and
    torch.optim.Adam(fused=True) on the same parameters.  Each is timed three ways with CUDA events: eager steps
    back to back (host launch cost included; the ~70-80 MB working set then sits in the 126 MB L2), the step
    replayed from a CUDA graph back to back, and the graph with a 512 MB buffer written between steps so that the
    step reads its operands from HBM (events around the step only).  torch's fused Adam is captured with
    capturable=True.  ``bytes`` is what the update must move at least (read and write of every state vector, read
    of the gradient), ``hbm_gbs`` that over the flushed time;
  * the st_pgat_spgnn_3 training step with SGD and with Adam: 64 ragged trees replayed from a CUDA graph
    (runner.GraphedTrainStep, the reference's batch size) and 4096 ragged trees eager (bench.py's headline
    workload), the two optimisers alternated twice in one process.
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
from spgnn_b200 import models as sm, ops, pe as spe, runner, synth_device  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def spgnn3_net():
    model, _, method, rate = bench.workload(bench.HEADLINE)
    torch.manual_seed(0)
    net = getattr(sm, method.split(".")[-1])(**model).cuda()
    net.init()
    net.train()
    net.set_gcn_only()
    return net, rate


OPTIMISERS = {
    "FlatSGD": lambda ps: runner.FlatSGD(ps, lr=bench.LR, momentum=bench.MOMENTUM),
    "FlatAdam": lambda ps: runner.FlatAdam(ps, lr=1e-3),
    "FlatAdam_AdamW_amsgrad": lambda ps: runner.FlatAdam(ps, lr=1e-3, weight_decay=1e-2, amsgrad=True,
                                                         decoupled=True),
    "torch_Adam_fused": lambda ps: torch.optim.Adam(ps, lr=1e-3, fused=True, capturable=True),
}
STATE_VECTORS = {"FlatSGD": 2, "FlatAdam": 3, "FlatAdam_AdamW_amsgrad": 4, "torch_Adam_fused": 3}   # p, buffers


def events(fn, iters, flush=None):
    """ms per call of fn: events around the whole loop, or around each call with ``flush`` run between calls."""
    ms = 0.0
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2 * (iters if flush else 1))]
    torch.cuda.synchronize()
    if flush is None:
        e[0].record()
        for _ in range(iters):
            fn()
        e[1].record()
        torch.cuda.synchronize()
        return e[0].elapsed_time(e[1]) / iters
    for i in range(iters):
        flush()
        e[2 * i].record()
        fn()
        e[2 * i + 1].record()
    torch.cuda.synchronize()
    for i in range(iters):
        ms += e[2 * i].elapsed_time(e[2 * i + 1])
    return ms / iters


def optimiser_alone(name, iters):
    net, _ = spgnn3_net()
    params = list(net.parameters())
    n = sum(p.numel() for p in params)
    opt = OPTIMISERS[name](params)
    gen = torch.Generator(device="cuda").manual_seed(5)
    grads = [torch.randn(p.shape, device="cuda", generator=gen) * 1e-3 for p in params]
    for p, g in zip(params, grads):
        p.grad = g.clone()

    def step():
        opt.step()                    # FlatSGD / FlatAdam: p.grad is the gradient bucket's slot after the first step

    for _ in range(5):
        step()
    eager = events(step, iters)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        step()
    graphed = events(graph.replay, iters)
    scratch = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    flushed = events(graph.replay, iters, flush=lambda: scratch.fill_(1))
    nbytes = 4 * n * (2 * STATE_VECTORS[name] + 1)
    return dict(what="optimiser step alone", optimiser=name, floats=n, eager_ms=eager, graph_ms=graphed,
                graph_hbm_ms=flushed, bytes=nbytes, hbm_gbs=nbytes / flushed / 1e6)


def training_steps(steps, reps):
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device="cuda")
    small = synth_device.make_batch(first_tree=0, count=64, seed=bench.SEED, ragged=True).graph
    spe.distance_pos_enc(small, pos_enc_dim=39)
    big = synth_device.make_batch(first_tree=0, count=4096, seed=bench.SEED, ragged=True).graph
    spe.distance_pos_enc(big, pos_enc_dim=39)
    out = []
    for rep in range(reps):
        for name in ("FlatSGD", "FlatAdam"):
            net, rate = spgnn3_net()
            opt = OPTIMISERS[name](net.parameters())
            ops.manual_seed(bench.SEED)
            gs = runner.GraphedTrainStep(net, small, opt, cw, rate, warmup=3)
            g64 = events(gs, 10 * steps)
            gs.reset_salt()
            for _ in range(3):
                runner.train_step(net, big, opt, cw, rate)
            b4096 = events(lambda: runner.train_step(net, big, opt, cw, rate), steps)
            out.append(dict(what="st_pgat_spgnn_3 training step", optimiser=name, rep=rep,
                            graph_64_trees_ms=g64, eager_4096_trees_ms=b4096,
                            graphs_per_s_4096=4096 / b4096 * 1e3))
            del gs, opt, net
            torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("optimizer_step.py measures on a CUDA device; none found")
    gpu = card()
    lines = [dict(optimiser_alone(name, args.iters), gpu=gpu) for name in OPTIMISERS]
    lines += [dict(d, gpu=gpu) for d in training_steps(args.steps, args.reps)]
    text = "\n".join(json.dumps(d) for d in lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
