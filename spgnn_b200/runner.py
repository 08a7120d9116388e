"""Callers of the hot path, kept on device: batch assembly from host buffers, the training step of
/root/reference/job_runner.py:1863-1920 (GCNTrainSPGNN.train) / :1368-1416 (GCNTrain.train) and the SGD or Adam update.

One process per GPU; trees shard by graph (they are independent components, SURVEY.md §8e): inference needs no
collective, training adds ONE NCCL all-reduce of the flat gradient bucket per step, and the masked weighted
cross-entropy is normalised by the GLOBAL Σw so that G-GPU training equals one big batch (sum order aside).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import dist as sdist, graph as sg, ops, pe as spe
from ._lib import lib, ptr, stream

CLASS_WEIGHTS_22 = [0.2] + [0.8] * 21      # exp_settings/st_pgat_spgnn_3.py:70-74 via job_runner.py:1867


class _FlatBucket:
    """The parameters as views into ONE contiguous fp32 buffer and a second one their gradients are gathered into:
    a step is one multi-tensor gather, one all-reduce (when world_size > 1) and the optimiser's fused update over
    the buffer.  ``zero_grad`` drops the gradients (``p.grad = None``), so autograd hands over each parameter's
    gradient without an accumulation kernel per parameter — at the reference's own batch size (64 trees) a step is
    launch-bound and those ~40 tiny kernels are a tenth of it."""

    def __init__(self, params, process_group=None):
        self.params = [p for p in params if p.requires_grad]
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.g_views, self.offsets = [], []
        o = 0
        for p in self.params:
            k = p.numel()
            self.flat_p[o:o + k].copy_(p.data.reshape(-1))
            p.data = self.flat_p[o:o + k].view_as(p.data)
            self.g_views.append(self.flat_g[o:o + k].view_as(p.data))
            self.offsets.append((o, k))
            p.grad = None
            o += k
        self.steps = 0
        self.numel = n

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    def _gather(self):
        """p.grad of every parameter -> its slot of the flat bucket (one multi-tensor copy).  Returns the list of
        parameters that have a gradient; afterwards their p.grad IS the slot, so callers see the (reduced) values."""
        dst, src, live, dead = [], [], [], []
        for i, (p, v) in enumerate(zip(self.params, self.g_views)):
            g = p.grad
            if g is None:
                dead.append(v)
                continue
            live.append(i)
            if g.data_ptr() != v.data_ptr():
                dst.append(v)
                src.append(g)
        if dead:
            torch._foreach_zero_(dead)                  # absent gradients contribute zeros to the all-reduce
        if dst:
            if hasattr(torch, "_foreach_copy_"):
                torch._foreach_copy_(dst, src)
            else:
                for d, g in zip(dst, src):
                    d.copy_(g)
        for i in live:
            self.params[i].grad = self.g_views[i]
        return live

    def set_lr(self, lr):
        self.lr = float(lr)


class FlatSGD(_FlatBucket):
    """torch.optim.SGD semantics (momentum, dampening, weight_decay, nesterov; the reference builds
    ``torch.optim.SGD(model.parameters(), **settings.OPTIMIZER)``, job_runner.py:239-249) over the flat bucket: one
    fused update kernel per contiguous run of live parameters.  As in torch, a parameter whose ``grad`` is None is
    skipped entirely (no momentum-only update, no weight decay) and its momentum buffer starts at the first gradient
    it receives."""

    def __init__(self, params, lr, momentum=0.0, dampening=0.0, weight_decay=0.0, nesterov=False, process_group=None):
        self.lr, self.momentum = float(lr), float(momentum)
        self.dampening, self.weight_decay, self.nesterov = float(dampening), float(weight_decay), bool(nesterov)
        if self.nesterov and (self.momentum <= 0.0 or self.dampening != 0.0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")        # torch's own check
        super().__init__(params, process_group)
        self.buf = torch.zeros(self.numel, dtype=torch.float32, device=self.flat_p.device)
        self.has_buf = [False] * len(self.params)       # momentum buffer initialised (torch: state['momentum_buffer'])

    def _runs(self, live):
        """Maximal contiguous ranges of the bucket whose parameters are live and share the first-step flag."""
        runs = []
        for i in live:
            o, k = self.offsets[i]
            first = not self.has_buf[i]
            if runs and runs[-1][0] + runs[-1][1] == o and runs[-1][2] == first:
                runs[-1] = (runs[-1][0], runs[-1][1] + k, first)
            else:
                runs.append((o, k, first))
            self.has_buf[i] = True
        return runs

    def step(self):
        live = self._gather()
        sdist.allreduce_sum_(self.flat_g, self.group)      # the ONE gradient collective of a step (no-op at world 1)
        esz = 4
        for o, k, first in self._runs(live):
            lib().sgd_step(self.flat_p.data_ptr() + o * esz, self.flat_g.data_ptr() + o * esz,
                           self.buf.data_ptr() + o * esz, k, self.lr, self.momentum, self.dampening, self.weight_decay,
                           int(self.nesterov), 1.0, int(first), stream())
        self.steps += 1

    # ---- torch.optim.SGD-shaped state (job_runner.py:341 saves optimizer.state_dict() under "optimizer_dict")
    def state_dict(self):
        state = {}
        for i, (o, k) in enumerate(self.offsets):
            if self.has_buf[i] and self.momentum != 0.0:
                state[i] = {"momentum_buffer": self.buf[o:o + k].view_as(self.params[i].data).detach().cpu().clone()}
        group = dict(lr=self.lr, momentum=self.momentum, dampening=self.dampening, weight_decay=self.weight_decay,
                     nesterov=self.nesterov, params=list(range(len(self.params))))
        return {"state": state, "param_groups": [group], "steps": self.steps}

    def load_state_dict(self, sd):
        group = sd["param_groups"][0]
        self.lr = float(group.get("lr", self.lr))
        self.momentum = float(group.get("momentum", self.momentum))
        self.dampening = float(group.get("dampening", self.dampening))
        self.weight_decay = float(group.get("weight_decay", self.weight_decay))
        self.nesterov = bool(group.get("nesterov", self.nesterov))
        self.has_buf = [False] * len(self.params)
        self.buf.zero_()
        for i, st in sd.get("state", {}).items():
            i = int(i)
            mb = st.get("momentum_buffer") if isinstance(st, dict) else None
            if mb is None or i >= len(self.params) or mb.numel() != self.offsets[i][1]:
                continue
            o, k = self.offsets[i]
            self.buf[o:o + k].copy_(mb.reshape(-1).to(self.buf.device, torch.float32))
            self.has_buf[i] = True
        self.steps = int(sd.get("steps", max(self.steps, 1 if any(self.has_buf) else 0)))


class FlatAdam(_FlatBucket):
    """torch.optim.Adam semantics (betas, eps, weight_decay, amsgrad, maximize), or torch.optim.AdamW with
    ``decoupled=True``, over the flat bucket (``spgnn_adam_step``).  As in torch, every parameter has its own step
    count and a parameter whose ``grad`` is None is skipped: its count does not advance and no decay is applied.
    The counts (``step_t``, int64 per parameter) live in device memory and the kernel advances them, so a
    GraphedTrainStep replay takes the bias corrections of the step it really is.  A step is two launches whatever
    the number of parameters: the count increment and one update over a device table of chunks of the live
    parameters, built once per set of live parameters and kept (a captured graph may still read it)."""

    CHUNK = 4096                                        # elements per block of the update kernel

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False,
                 maximize=False, decoupled=False, process_group=None):
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.weight_decay, self.amsgrad, self.maximize = float(weight_decay), bool(amsgrad), bool(maximize)
        self.decoupled = bool(decoupled)
        if not (self.lr >= 0.0 and self.eps >= 0.0 and self.weight_decay >= 0.0):         # torch's own checks
            raise ValueError(f"Adam: lr, eps and weight_decay must be >= 0 (got {lr}, {eps}, {weight_decay})")
        if not all(0.0 <= b < 1.0 for b in self.betas):
            raise ValueError(f"Adam: betas must be in [0, 1) (got {betas})")
        super().__init__(params, process_group)
        dev = self.flat_p.device
        self.exp_avg = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.max_exp_avg_sq = torch.zeros_like(self.exp_avg) if self.amsgrad else None
        self.step_t = torch.zeros(len(self.params), dtype=torch.int64, device=dev)
        self._tables = {}

    def _table(self, live):
        """(int64 device tensor [chunks x {offset, length, parameter}, then the live indices], number of chunks)"""
        key = tuple(live)
        if key not in self._tables:
            rows = []
            for i in live:
                o, k = self.offsets[i]
                for c in range(0, k, self.CHUNK):
                    rows += [o + c, min(self.CHUNK, k - c), i]
            self._tables[key] = (torch.tensor(rows + list(live), dtype=torch.int64, device=self.flat_p.device),
                                 len(rows) // 3)
        return self._tables[key]

    def step(self):
        live = self._gather()
        sdist.allreduce_sum_(self.flat_g, self.group)      # the ONE gradient collective of a step (no-op at world 1)
        if live:
            table, n_chunks = self._table(live)
            lib().adam_step(ptr(self.flat_p), ptr(self.flat_g), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                            ptr(self.max_exp_avg_sq), ptr(self.step_t), ptr(table), n_chunks,
                            table.data_ptr() + 8 * 3 * n_chunks, len(live), self.lr, self.betas[0], self.betas[1],
                            self.eps, self.weight_decay, int(self.amsgrad), int(self.maximize), int(self.decoupled),
                            stream())
        self.steps += 1

    # ---- the layout of torch.optim.Adam / AdamW.state_dict(), which job_runner.py saves under "optimizer_dict"
    def _buffers(self):
        names = [("exp_avg", self.exp_avg), ("exp_avg_sq", self.exp_avg_sq)]
        return names + ([("max_exp_avg_sq", self.max_exp_avg_sq)] if self.amsgrad else [])

    def state_dict(self):
        counts = self.step_t.tolist()
        state = {}
        for i, (o, k) in enumerate(self.offsets):
            if counts[i]:                               # torch creates a parameter's state at its first gradient
                st = {"step": torch.tensor(float(counts[i]), dtype=torch.float32)}
                for name, buf in self._buffers():
                    st[name] = buf[o:o + k].view_as(self.params[i].data).detach().cpu().clone()
                state[i] = st
        group = dict(lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.weight_decay, amsgrad=self.amsgrad,
                     maximize=self.maximize, foreach=None, capturable=False, differentiable=False, fused=None,
                     decoupled_weight_decay=self.decoupled, params=list(range(len(self.params))))
        return {"state": state, "param_groups": [group], "steps": self.steps}

    def load_state_dict(self, sd):
        """A state dict of this class or of torch.optim.Adam / AdamW (CPU or CUDA tensors, ``step`` a tensor or a
        number).  As in torch, the saved group's hyper-parameters replace the current ones."""
        groups = sd["param_groups"]
        if len(groups) != 1 or len(groups[0]["params"]) != len(self.params):
            raise ValueError(f"FlatAdam: expected one parameter group of {len(self.params)} parameters")
        group = groups[0]
        self.lr = float(group.get("lr", self.lr))
        self.betas = tuple(float(b) for b in group.get("betas", self.betas))
        self.eps = float(group.get("eps", self.eps))
        self.weight_decay = float(group.get("weight_decay", self.weight_decay))
        self.amsgrad = bool(group.get("amsgrad", self.amsgrad))
        self.maximize = bool(group.get("maximize", self.maximize))
        self.decoupled = bool(group.get("decoupled_weight_decay", self.decoupled))
        self.max_exp_avg_sq = torch.zeros_like(self.exp_avg) if self.amsgrad else None
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        counts = [0] * len(self.params)
        for i, st in sd.get("state", {}).items():
            i = int(i)
            o, k = self.offsets[i]
            for name, buf in self._buffers():
                t = st[name]
                if t.numel() != k:
                    raise ValueError(f"FlatAdam: state {i} '{name}' has {t.numel()} elements, the parameter {k}")
                buf[o:o + k].copy_(t.reshape(-1).to(buf.device, torch.float32))
            counts[i] = int(round(float(st["step"])))
        self.step_t.copy_(torch.tensor(counts, dtype=torch.int64))
        self.steps = int(sd.get("steps", max(counts)))


def _allreduce_sums(group=None):
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None

    def fn(sums):
        return sdist.allreduce_sum_(sums, group)       # (Σ w·nll, Σ w) over all ranks: the loss is the GLOBAL mean
    return fn


def train_step(net, g, opt, class_w, sampling_rate, mask=None, group=None):
    """One iteration of the reference's GCN_STEPS loop (job_runner.py:1892-1919): zero_grad, forward, masked
    weighted CE (labelled nodes always kept, label-0 nodes with probability ``sampling_rate``), backward, step."""
    opt.zero_grad()
    out = net(g)
    loss = ops.masked_cross_entropy(out[0], g.ndata["y"], class_w, mask=mask, rate=sampling_rate,
                                    reduce_fn=_allreduce_sums(group))
    loss.backward()
    opt.step()
    # detached: a caller that keeps the loss must not keep the step's autograd graph (and the parameters'
    # AccumulateGrad nodes, bound to the stream they were created on) alive into the next step / a graph capture
    return loss.detach()


class GraphedTrainStep:
    """The GCN_STEPS loop of the reference (job_runner.py:1892-1919: 300 steps on ONE batch) as a CUDA graph.

    At the reference's own batch size (64 scans, ~19 k nodes) a step is ~115 kernel launches of a few microseconds
    each: the GPU waits for the host.  The step is captured once per batch and replayed: the learning rate, the
    momentum-buffer state and every pointer are frozen in the graph, the dropout / sampling masks are NOT — the first
    nodes of the graph bump a device-side step counter and copy it into the library's seed salt
    (``spgnn_seed_salt_set``), so replay k draws the masks of seed + k.  FlatAdam's step counts (its bias corrections)
    are not frozen either: they live in device memory and its kernel advances them.  ``loss`` is a device tensor
    refreshed by every replay.  Re-capture (a new object) when the batch or the learning rate changes; world_size > 1 stays eager."""

    def __init__(self, net, g, opt, class_w, sampling_rate, warmup=3, group=None):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            raise RuntimeError("GraphedTrainStep: data-parallel steps are not captured (use train_step)")
        self.net, self.g, self.opt = net, g, opt
        dev = class_w.device
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
        g.max_degree()                                  # the builder's flags: read once, before the capture
        g.check_no_zero_in_degree()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):        # eager: allocator pools, momentum buffers, lazy attributes
                train_step(net, g, opt, class_w, sampling_rate)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.lr = opt.lr
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self.counter.add_(1)
            lib().seed_salt_set(ptr(self.counter), stream())
            self.loss = train_step(net, g, opt, class_w, sampling_rate)
        self.replays = 0

    def __call__(self):
        if self.opt.lr != self.lr:
            raise RuntimeError("GraphedTrainStep: the learning rate changed since the capture; build a new one")
        self.graph.replay()
        self.replays += 1
        self.opt.steps += 1
        return self.loss

    def reset_salt(self):
        """Back to eager semantics for whatever runs next on this device (salt 0)."""
        self.counter.zero_()
        lib().seed_salt_set(ptr(self.counter), stream())


@torch.no_grad()
def infer(net, g):
    """GCNTestSPGNN.run's device part (job_runner.py:2052 + :158-165): logits → per-tree per-class arg-max node."""
    out = net(g)
    return out[0], ops.segmented_argmax(out[0], g)


class HostBatch:
    """A batch of scans in (pinned) host memory, ready for the H2D copy of job_runner.py:1872-1875.

    ``packed=False``: the stage-1 pickle layout concatenated over scans (job_runner.py:796-805): adj uint8 blocks,
    fvs fp32 [N, fv], fvs_out fp32 [N, 22], labels int64 [N] — 4.5 MB per 301-node scan.
    ``packed=True`` (default): the lossless wire format of csrc/wire.cu — ``fvs`` zero-suppressed (it is a ReLU
    output: bit mask + non-zero values), the adjacency as int32 edge lists in DGL edge order, labels as uint8 when
    they fit — about half the bytes; the device decodes into bit-identical tensors.  Packing is loader work done
    once per batch when it is read (``pack_threads`` host threads, ``pack_seconds`` records it)."""

    def __init__(self, n_nodes, adj_cat, fvs, fvs_out, labels, pin=True, packed=False, pack_threads=0):
        import time
        f = (lambda t: t.pin_memory()) if pin else (lambda t: t)
        self.packed = bool(packed)
        self.n_nodes = f(torch.as_tensor(n_nodes, dtype=torch.int64))
        self.max_nodes = int(self.n_nodes.max())
        self.fvs_out = f(fvs_out)
        self.fv_dim = int(fvs.shape[1])
        self.pack_seconds = 0.0
        if not self.packed:
            self.adj_cat, self.fvs, self.labels = f(adj_cat), f(fvs), f(labels)
            return
        t0 = time.perf_counter()
        L = lib()
        fvs = fvs.contiguous()
        rows, cols = fvs.shape
        row_off = torch.empty(rows + 1, dtype=torch.int64)
        nnz = int(L.host_pack_rows_count(fvs.data_ptr(), fvs.stride(0), rows, cols, row_off.data_ptr(), pack_threads))
        if nnz < 0:
            raise RuntimeError("spgnn_host_pack_rows_count failed: " + L.last_error())
        self.f_row_off = f(row_off)
        self.f_mask = f(torch.empty(rows, (cols + 31) // 32, dtype=torch.int32))
        self.f_vals = f(torch.empty(max(nnz, 1), dtype=torch.float32))
        L.host_pack_rows_fill(fvs.data_ptr(), fvs.stride(0), rows, cols, self.f_row_off.data_ptr(),
                              self.f_mask.data_ptr(), self.f_vals.data_ptr(), pack_threads)
        self.f_nnz = nnz
        # adjacency blocks -> int32 edge lists (row-major order of the off-diagonal non-zeros = DGL edge order)
        adj_cat = adj_cat.contiguous()
        nn_ = self.n_nodes.contiguous()
        B = nn_.numel()
        e_off = torch.empty(B + 1, dtype=torch.int64)
        ne = int(L.host_adj_edges_count(adj_cat.data_ptr(), nn_.data_ptr(), B, e_off.data_ptr(), pack_threads))
        if ne < 0:
            raise RuntimeError("spgnn_host_adj_edges_count failed: " + L.last_error())
        self.e_off = f(e_off)
        self.e_src = f(torch.empty(max(ne, 1), dtype=torch.int32))[:ne]
        self.e_dst = f(torch.empty(max(ne, 1), dtype=torch.int32))[:ne]
        md = torch.zeros(1, dtype=torch.int32)
        L.host_adj_edges_fill(adj_cat.data_ptr(), nn_.data_ptr(), B, self.e_off.data_ptr(), self.e_src.data_ptr(),
                              self.e_dst.data_ptr(), md.data_ptr(), pack_threads)
        self.max_degree = int(md.item())              # includes the self loop the device appends to every node
        small = labels.numel() == 0 or (int(labels.min()) >= 0 and int(labels.max()) < 256)
        self.labels = f(labels.to(torch.uint8) if small else labels)
        self.pack_seconds = time.perf_counter() - t0

    def tensors(self):
        if self.packed:
            return (self.n_nodes, self.e_off, self.e_src, self.e_dst, self.f_row_off, self.f_mask, self.f_vals,
                    self.fvs_out, self.labels)
        return (self.n_nodes, self.adj_cat, self.fvs, self.fvs_out, self.labels)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in self.tensors())


def _upload(hb: HostBatch, dev):
    return tuple(t.to(dev, non_blocking=True) for t in hb.tensors())


def _assemble(hb: HostBatch, bufs, dev, pos_enc_dim, pe_kind, defer_checks=False):
    if hb.packed:
        n_nodes, e_off, e_src, e_dst, f_row_off, f_mask, f_vals, fvs_out, labels = bufs
        L = lib()
        B, N, NE = n_nodes.numel(), int(f_mask.shape[0]), int(e_src.numel())
        node_off = sg.device_scan(n_nodes)
        sl = torch.empty(NE + N, dtype=torch.int64, device=dev)
        dl = torch.empty(NE + N, dtype=torch.int64, device=dev)
        n_edges = torch.empty(B, dtype=torch.int64, device=dev)
        L.edges_expand(ptr(e_src), ptr(e_dst), ptr(e_off), ptr(node_off), B, NE, N, ptr(sl), ptr(dl), ptr(n_edges),
                       stream())
        fvs = ops.empty_padded(N, hb.fv_dim, dev)
        L.unpack_rows(ptr(f_mask), ptr(f_vals), ptr(f_row_off), N, hb.fv_dim, ptr(fvs), fvs.stride(0), stream(),
                      _key=("bytes", 4.0 * hb.f_nnz + 4.0 * N * hb.fv_dim + N * (hb.fv_dim // 8 + 8)))
        labels = labels.to(torch.int64)
        # everything the builder would read back is known from packing: no device→host read on this path
        g = sg.Graph.from_edge_lists(n_nodes, n_edges, sl, dl, max_nodes=hb.max_nodes, check=False, num_nodes=N,
                                     max_degree=hb.max_degree, zero_in_degree=0)
    else:
        n_nodes, adj, fvs, fvs_out, labels = bufs
        n_edges, sl, dl = sg._edges_from_dense(adj, n_nodes, dev)
        g = sg.Graph.from_edge_lists(n_nodes, n_edges, sl, dl, max_nodes=hb.max_nodes, check=False)
    g.ndata["fvs"], g.ndata["fvs_out"], g.ndata["y"] = fvs, fvs_out, labels
    if pos_enc_dim:
        if pe_kind == "dist":
            spe.distance_pos_enc(g, pos_enc_dim=pos_enc_dim, check=not defer_checks)
        else:
            g.ndata["pos_enc"] = spe.rw_pos_enc(g, pos_enc_dim)
    return g


def batch_to_device(hb: HostBatch, pos_enc_dim=39, device=None, pe_kind="dist"):
    """Host buffers → device graph batch with features and positional encoding: the per-batch part of
    GCNTrainSPGNN.train (job_runner.py:1872-1882) — H2D copies, from_adj_to_graph for every scan, PE, dgl.batch."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    return _assemble(hb, _upload(hb, dev), dev, pos_enc_dim, pe_kind)


class DeviceBatchLoader:
    """Iterates device batches over an iterable of :class:`HostBatch`, with the H2D copy of batch i+1 running on
    a copy stream while the caller computes on batch i (the reference copies synchronously inside the loop,
    job_runner.py:1872-1875).  Every batch is copied from (pinned) host memory each time it is yielded; graph
    build and positional encoding run on the caller's stream once that batch's copy has landed."""

    def __init__(self, host_batches, pos_enc_dim=39, device=None, pe_kind="dist"):
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.it = iter(host_batches)
        self.pos_enc_dim, self.pe_kind = pos_enc_dim, pe_kind
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self._pending = None
        self._last = None
        self._issue()

    def _issue(self):
        try:
            hb = next(self.it)
        except StopIteration:
            self._pending = None
            return
        cur = torch.cuda.current_stream(self.dev)
        # destination blocks come from the copy stream's pool; record_stream hands them to the caller's stream
        with torch.cuda.stream(self.copy_stream):
            bufs = _upload(hb, self.dev)
            done = torch.cuda.Event()
            done.record(self.copy_stream)
        for t in bufs:
            t.record_stream(cur)
        self._pending = (hb, bufs, done)

    def __iter__(self):
        return self

    def __next__(self):
        if self._last is not None:         # connectivity flag of the PREVIOUS batch: long finished, the read is free
            if int(self._last.item()):
                raise RuntimeError("Found infinite path length because the graph is not connected (nx.diameter in "
                                   "the reference) — in the batch before this one")
            self._last = None
        if self._pending is None:
            raise StopIteration
        hb, bufs, done = self._pending
        torch.cuda.current_stream(self.dev).wait_event(done)
        # decode + graph build + positional encoding are queued WITHOUT a device→host read, and only then is the next
        # batch's copy issued: submitting a multi-GB cudaMemcpyAsync takes the host milliseconds during which kernel
        # launches crawl (scripts/e2e_timeline.py: 24 ms instead of 4 ms to launch a step) — with the GPU already
        # holding this batch's build work, that submission costs no GPU idle time
        g = _assemble(hb, bufs, self.dev, self.pos_enc_dim, self.pe_kind, defer_checks=True)
        self._last = getattr(g, "_pe_flags", None)
        self._issue()                      # next batch's copy overlaps this batch's graph build + step
        return g


def host_batch_from_graph(g, pin=True, packed=False):
    """Device batch → HostBatch (bench/test helper: produces the host-side inputs of the end-to-end path)."""
    n = g.batch_num_nodes()
    adj_off = sg.device_scan(n * n)
    adj = torch.zeros(int(adj_off[-1].item()), dtype=torch.uint8, device=g.device)
    gid = torch.repeat_interleave(torch.arange(g.batch_size, device=g.device), g.batch_num_edges())
    adj[adj_off[gid] + g.src_local * n[gid] + g.dst_local] = 1
    return HostBatch(n.cpu(), adj.cpu(), g.ndata["fvs"].cpu(), g.ndata["fvs_out"].cpu(), g.ndata["y"].cpu(), pin=pin,
                     packed=packed)
