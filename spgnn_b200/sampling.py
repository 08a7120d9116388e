"""Neighbour-sampled mini-batches for the SAGE training path of the reference (SURVEY.md §8f rank 4).

Replaces what ``GCNTrainSAGE.train`` (/root/reference/job_runner.py:1460-1514) takes from DGL:
``dgl.dataloading.MultiLayerNeighborSampler(node_ks)``, ``dgl.dataloading.NodeDataLoader(g, nids, sampler,
batch_size=NODE_BATCH_SIZE, shuffle=True)`` and the message-flow-graph ``block`` objects that
``SAGE.forward_batch`` (models.py:685-689) feeds to ``SAGEConv``.

DGL semantics kept (0.7.x ``sample_neighbors(replace=False)`` + ``to_block``):
  * per layer, every seed keeps ``min(fanout, in_degree)`` of its in-edges, drawn uniformly without replacement;
  * a block's destination nodes are the seeds in order, its source nodes are the seeds FIRST and then every other
    endpoint once (so ``h_dst = h_src[:num_dst]``); blocks are built output layer first, each layer's source
    nodes being the previous layer's seeds; ``blocks[0].srcdata`` / ``blocks[-1].dstdata`` carry the node data.
The random stream is torch's, not DGL's: parity with DGL is distributional (which edges are drawn), exact for
everything computed from a given set of blocks.

Two implementations of the same semantics:
  * ``MultiLayerNeighborSampler`` / ``NodeDataLoader``: torch tensor arithmetic on the graph's device (or the host),
    drawing from a torch generator - 44 synchronising calls and 338 launches per st_sage_3 mini-batch;
  * ``DeviceBlockSampler`` / ``DeviceNodeDataLoader``: every layer's draw, ``to_block`` and CSC / CSR build in one
    CUDA kernel (csrc/sampling.cu) plus one row gather per node-data key, with ONE device->host read per mini-batch
    (the block sizes and the kernel's error word).  Its random stream is a counter hash of (seed, salt, layer, CSC
    slot) - the same distribution, a different stream (as for the dropout masks).  ``GCNTrainSAGE`` uses it.
The layer arithmetic on the blocks is this repo's CUDA kernels either way.
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import SpgnnError, lib, ptr, require_cuda, stream


class Block:
    """Bipartite message-flow graph: edges go from ``num_src_nodes`` source rows to ``num_dst_nodes`` destination
    rows; destination node i is source node i.  In-CSC by destination and out-CSR by source (int32), the layout
    the aggregation kernels read (``out_slot`` = position of the edge in the in-CSC)."""

    is_block = True

    def __init__(self, src_local, dst_local, src_ids, num_dst):
        dev = src_local.device
        self.num_src_nodes, self.num_dst_nodes = int(src_ids.numel()), int(num_dst)
        self.src_ids = src_ids                                   # global node ids; [:num_dst] are the seeds
        self.dst_ids = src_ids[:self.num_dst_nodes]
        E = int(src_local.numel())
        # edges arrive grouped by destination in ascending order (the sampler emits them that way)
        if E > 1 and bool((dst_local[1:] < dst_local[:-1]).any()):
            order = torch.sort(dst_local, stable=True)[1]
            src_local, dst_local = src_local[order], dst_local[order]
        self.in_ptr = torch.zeros(self.num_dst_nodes + 1, dtype=torch.int32, device=dev)
        self.in_ptr[1:] = torch.cumsum(torch.bincount(dst_local, minlength=self.num_dst_nodes), 0).to(torch.int32)
        self.in_src = src_local.to(torch.int32)
        order = torch.sort(src_local, stable=True)[1]
        self.out_ptr = torch.zeros(self.num_src_nodes + 1, dtype=torch.int32, device=dev)
        self.out_ptr[1:] = torch.cumsum(torch.bincount(src_local, minlength=self.num_src_nodes), 0).to(torch.int32)
        self.out_dst = dst_local[order].to(torch.int32)
        self.out_slot = order.to(torch.int32)
        self.srcdata, self.dstdata = {}, {}

    @classmethod
    def from_csr(cls, src_ids, num_dst, in_ptr, in_src, out_ptr, out_dst, out_slot):
        """A block around a prebuilt in-CSC / out-CSR (int32, the layout ``__init__`` computes), adopted as given."""
        b = object.__new__(cls)
        b.num_src_nodes, b.num_dst_nodes = int(src_ids.numel()), int(num_dst)
        b.src_ids, b.dst_ids = src_ids, src_ids[:b.num_dst_nodes]
        b.in_ptr, b.in_src, b.out_ptr, b.out_dst, b.out_slot = in_ptr, in_src, out_ptr, out_dst, out_slot
        b.srcdata, b.dstdata = {}, {}
        return b

    # ---- the surface of a DGL block the reference touches (job_runner.py:1499-1501)
    def number_of_src_nodes(self):
        return self.num_src_nodes

    def number_of_dst_nodes(self):
        return self.num_dst_nodes

    def number_of_edges(self):
        return int(self.in_src.numel())

    @property
    def num_edges(self):
        return int(self.in_src.numel())

    @property
    def device(self):
        return self.in_ptr.device

    def int(self):
        return self                                              # indices are int32 already

    def to(self, device=None, **_):
        if device is None or torch.device(device) == self.device:
            return self
        b = object.__new__(Block)
        b.__dict__.update(self.__dict__)
        for k in ("src_ids", "dst_ids", "in_ptr", "in_src", "out_ptr", "out_dst", "out_slot"):
            setattr(b, k, getattr(self, k).to(device))
        b.srcdata = {k: v.to(device) for k, v in self.srcdata.items()}
        b.dstdata = {k: v.to(device) for k, v in self.dstdata.items()}
        return b

    def check_no_zero_in_degree(self):
        if bool((self.in_ptr[1:] == self.in_ptr[:-1]).any()):
            raise SpgnnError("There are 0-in-degree nodes in the block")

    def edges(self):
        """(src_local, dst_local) int64 in in-CSC order."""
        deg = (self.in_ptr[1:] - self.in_ptr[:-1]).long()
        dst = torch.repeat_interleave(torch.arange(self.num_dst_nodes, device=self.device), deg)
        return self.in_src.long(), dst


def sample_neighbors(g, seeds, fanout, generator=None):
    """For every seed keep min(fanout, in_degree) in-edges, uniformly without replacement (fanout < 0: all).
    Returns (src global ids, dst index into ``seeds``), grouped by destination in ascending order."""
    dev = g.in_ptr.device
    seeds = seeds.to(dev).long()
    S = int(seeds.numel())
    beg = g.in_ptr[seeds].long()
    deg = g.in_ptr[seeds + 1].long() - beg
    total = int(deg.sum())
    seg = torch.repeat_interleave(torch.arange(S, device=dev), deg)
    start = torch.cumsum(deg, 0) - deg                           # first edge of each seed in the enumeration
    off = torch.arange(total, device=dev) - start[seg]
    slot = beg[seg] + off
    if fanout >= 0 and total > 0:
        key = torch.rand(total, generator=generator, device=dev, dtype=torch.float64)
        order = torch.sort(seg.to(torch.float64) + key)[1]       # random order inside every seed's segment
        rank = torch.arange(total, device=dev) - start[seg[order]]
        keep = order[rank < fanout]
        keep = torch.sort(keep)[0]                               # back to ascending (destination, edge id) order
        seg, slot = seg[keep], slot[keep]
    return g.in_src[slot].long(), seg


def to_block(g, src, dst_index, seeds):
    """DGL ``to_block``: destination nodes = seeds (in order), source nodes = seeds first, then the other endpoints."""
    dev = src.device
    seeds = seeds.to(dev).long()
    S = int(seeds.numel())
    pos = torch.full((g.num_nodes,), -1, dtype=torch.int64, device=dev)
    pos[seeds] = torch.arange(S, device=dev)
    extra = torch.unique(src[pos[src] < 0])
    pos[extra] = S + torch.arange(int(extra.numel()), device=dev)
    return Block(pos[src], dst_index, torch.cat([seeds, extra]), S)


class MultiLayerNeighborSampler:
    """``dgl.dataloading.MultiLayerNeighborSampler(fanouts)``: one block per layer, ``fanouts[i]`` for layer i."""

    def __init__(self, fanouts, replace=False, return_eids=False):
        if replace:
            raise SpgnnError("MultiLayerNeighborSampler: only replace=False (what the reference uses)")
        self.fanouts = [int(f) if f is not None else -1 for f in fanouts]

    def sample_blocks(self, g, seeds, generator=None):
        blocks = []
        seeds = torch.as_tensor(seeds, device=g.in_ptr.device).long()
        for fanout in reversed(self.fanouts):
            src, dst_index = sample_neighbors(g, seeds, fanout, generator)
            block = to_block(g, src, dst_index, seeds)
            blocks.insert(0, block)
            seeds = block.src_ids
        return blocks


class NodeDataLoader:
    """``dgl.dataloading.NodeDataLoader(g, nids, sampler, batch_size=, shuffle=, drop_last=)``: iterates
    ``(input_nodes, seeds, blocks)`` with ``blocks[0].srcdata`` / ``blocks[-1].dstdata`` filled from ``g.ndata``."""

    def __init__(self, g, nids, block_sampler, device=None, batch_size=1, shuffle=False, drop_last=False,
                 num_workers=0, generator=None, **_):
        self.g, self.sampler = g, block_sampler
        self.nids = torch.as_tensor(nids, device=g.in_ptr.device).long()
        self.batch_size, self.shuffle, self.drop_last = int(batch_size), bool(shuffle), bool(drop_last)
        self.generator = generator

    def __len__(self):
        n = int(self.nids.numel())
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        nids = self.nids
        if self.shuffle:
            perm = torch.randperm(int(nids.numel()), generator=self.generator, device=nids.device)
            nids = nids[perm]
        for i in range(len(self)):
            seeds = nids[i * self.batch_size:(i + 1) * self.batch_size]
            blocks = self.sampler.sample_blocks(self.g, seeds, self.generator)
            input_nodes = blocks[0].src_ids
            for k, v in self.g.ndata.items():
                blocks[0].srcdata[k] = v[input_nodes]
                blocks[-1].dstdata[k] = v[seeds]
            yield input_nodes, seeds, blocks


# ------------------------------------------------------------------------------------------------ device sampler
_INT32_MAX = 2 ** 31 - 1
_SMEM_KEYS = 4096            # csrc/sampling.cu kSmemKeys: sorts up to this many keys need no global scratch
_ERRORS = {1: "a block outgrew the capacity computed for it", 2: "a seed id is outside [0, num_nodes)",
           3: "a seed id is repeated", 4: "the graph's in_src holds an id outside [0, num_nodes)"}


def block_capacities(num_nodes, num_edges, num_seeds, fanouts, max_degree=None):
    """Upper bounds of every block's sizes, known on the host before the draw: ``[(dst, src, edges)]`` per layer,
    input layer first.  Layer l keeps at most ``dst_l * fanout_l`` edges (``max_degree`` per destination when
    fanout < 0) and never more than the graph has; every kept edge adds at most one source; no block has more sources
    than the graph has nodes; a layer's destinations are the next layer's sources.  Refuses bounds above int32."""
    caps, d = [], int(num_seeds)
    for f in reversed([int(f) for f in fanouts]):
        if f < 0:
            if max_degree is None:
                raise SpgnnError("block_capacities: fanout -1 needs the graph's max_degree()")
            f = int(max_degree)
        e = min(d * f, int(num_edges))
        src = min(int(num_nodes), d + e)
        if max(d, src, e) > _INT32_MAX - 1:
            raise SpgnnError(f"block_capacities: a block of up to {src} sources / {e} edges exceeds int32 indexing")
        caps.insert(0, (d, src, e))
        d = src
    return caps


def _pow2(n):
    return 1 << max(int(n) - 1, 0).bit_length()


class DeviceBlockSampler:
    """``MultiLayerNeighborSampler(fanouts)`` on the device: the blocks of all layers from one kernel launch, their
    sizes from one device->host read.  Every block tensor is a view of a buffer allocated at the host-known capacity
    (:func:`block_capacities`), trimmed to the sizes read back.  ``seed`` / ``salt`` select the draw (a counter
    hash: the same (graph, seeds, fanouts, seed, salt) gives the same blocks); ``seed=None`` takes the next seed of
    ``ops.next_seed()``.  Calls on one graph are stream-ordered on the current stream (they share its ``pos``
    scratch)."""

    def __init__(self, fanouts, replace=False):
        if replace:
            raise SpgnnError("DeviceBlockSampler: only replace=False (what the reference uses)")
        self.fanouts = [int(f) if f is not None else -1 for f in fanouts]
        if not 1 <= len(self.fanouts) <= 8:
            raise SpgnnError(f"DeviceBlockSampler: 1 to 8 layers, got {len(self.fanouts)}")

    def sample_blocks(self, g, seeds, seed=None, salt=0, gather=True):
        """Blocks for the distinct node ids ``seeds`` (int64 CUDA tensor); with ``gather`` every ``g.ndata`` key is
        gathered into ``blocks[0].srcdata`` and ``blocks[-1].dstdata``."""
        from . import ops
        require_cuda(seeds)
        dev = g.in_ptr.device
        seeds = seeds.to(device=dev, dtype=torch.int64).contiguous()
        S, L = int(seeds.numel()), len(self.fanouts)
        if S == 0:
            raise SpgnnError("DeviceBlockSampler: no seeds")
        max_deg = g.max_degree() if min(self.fanouts) < 0 else None
        caps = block_capacities(g.num_nodes, g.num_edges, S, self.fanouts, max_deg)
        # one int32 buffer (in_ptr, in_src, out_ptr, out_dst, out_slot per layer, then the edge-destination scratch)
        # and one int64 buffer (src_ids per layer, then the sizes)
        lens32 = [n for cd, cs, ce in caps for n in (cd + 1, ce, cs + 1, ce, ce)]
        edst_cap = max(max(ce for _, _, ce in caps), 1)
        buf32 = torch.empty(sum(lens32) + edst_cap, dtype=torch.int32, device=dev)
        buf64 = torch.empty(sum(cs for _, cs, _ in caps) + 2 * L + 1, dtype=torch.int64, device=dev)
        v32 = list(torch.split(buf32, lens32 + [edst_cap]))
        v64 = list(torch.split(buf64, [cs for _, cs, _ in caps] + [2 * L + 1]))
        sizes = v64[L]
        need = max(max(ce, cs - cd) for cd, cs, ce in caps)
        keys = torch.empty(_pow2(need), dtype=torch.int64, device=dev) if need > _SMEM_KEYS else None
        pos = g.__dict__.get("_sample_pos")
        if pos is None:                                           # all -1; every call leaves it that way
            pos = g.__dict__["_sample_pos"] = torch.full((g.num_nodes,), -1, dtype=torch.int32, device=dev)
        bufs = np.array([[ptr(t) for t in v32[5 * l:5 * l + 5]] + [ptr(v64[l])] for l in range(L)], dtype=np.int64)
        fan = np.array(self.fanouts, dtype=np.int64)
        cap_arr = np.array(caps, dtype=np.int64)
        lib().sample_blocks(ptr(g.in_ptr), ptr(g.in_src), g.num_nodes, ptr(seeds), S, L, fan.ctypes.data,
                            cap_arr.ctypes.data, bufs.ctypes.data, ops.next_seed() if seed is None else int(seed),
                            int(salt) & 0xFFFFFFFFFFFFFFFF, ptr(pos), ptr(v32[-1]), edst_cap, ptr(keys),
                            0 if keys is None else keys.numel(), ptr(sizes), stream())
        src_data, dst_data = {}, {}
        if gather:
            for k, v in g.ndata.items():
                src_data[k] = _gather(v, v64[0], sizes, caps[0][1])
                dst_data[k] = _gather(v, seeds, None, S)
        host = sizes.tolist()                                     # the one device->host read of the mini-batch
        if host[2 * L]:
            raise SpgnnError(f"DeviceBlockSampler: {_ERRORS.get(host[2 * L], 'error ' + str(host[2 * L]))}")
        blocks = []
        for l in range(L):
            n_src, E = host[2 * l], host[2 * l + 1]
            n_dst = host[2 * l + 2] if l + 1 < L else S
            in_ptr, in_src, out_ptr, out_dst, out_slot = v32[5 * l:5 * l + 5]
            blocks.append(Block.from_csr(v64[l][:n_src], n_dst, in_ptr[:n_dst + 1], in_src[:E], out_ptr[:n_src + 1],
                                         out_dst[:E], out_slot[:E]))
        n0 = blocks[0].num_src_nodes
        blocks[0].srcdata.update({k: v[:n0] for k, v in src_data.items()})
        blocks[-1].dstdata.update(dst_data)
        return blocks


def _gather(x, idx, count, cap):
    """x[idx[:min(cap, *count)]] into a buffer of ``cap`` rows (csrc/sampling.cu gather_rows)."""
    require_cuda(x)
    if x.dim() == 0 or (x.dim() > 1 and not x[0].is_contiguous()):
        x = x.contiguous()
    row_bytes = x[0].numel() * x.element_size()
    if row_bytes % 4 or (x.stride(0) * x.element_size()) % 4 or x.data_ptr() % 4:
        raise SpgnnError(f"node data of {row_bytes} bytes per row: rows must be whole 32-bit words")
    out = torch.empty((cap,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    lib().gather_rows(ptr(x), x.stride(0) * x.element_size() // 4, x.shape[0], ptr(idx), ptr(count), cap,
                      row_bytes // 4, ptr(out), row_bytes // 4, stream())
    return out


class DeviceNodeDataLoader:
    """``NodeDataLoader`` over a :class:`DeviceBlockSampler`: iterates ``(input_nodes, seeds, blocks)`` with
    ``blocks[0].srcdata`` / ``blocks[-1].dstdata`` filled from ``g.ndata``.  ``nids`` (distinct node ids) are checked
    on the host once, when the loader is built; the shuffle is a ``torch.randperm`` drawn on the device.  Each
    mini-batch costs one device->host read (the block sizes)."""

    def __init__(self, g, nids, block_sampler, device=None, batch_size=1, shuffle=False, drop_last=False,
                 num_workers=0, generator=None, **_):
        self.g, self.sampler = g, block_sampler
        dev = g.in_ptr.device
        if isinstance(nids, torch.Tensor) and nids.is_cuda:
            lo, hi = (int(v) for v in torch.stack([nids.min(), nids.max()]).tolist()) if nids.numel() else (0, 0)
            self.nids = nids.to(device=dev, dtype=torch.int64)
        else:
            host = np.asarray(nids.cpu() if isinstance(nids, torch.Tensor) else nids, dtype=np.int64).reshape(-1)
            lo, hi = (int(host.min()), int(host.max())) if host.size else (0, 0)
            self.nids = torch.from_numpy(host).pin_memory().to(dev, non_blocking=True)
        if lo < 0 or hi >= g.num_nodes:
            raise SpgnnError(f"DeviceNodeDataLoader: node ids [{lo}, {hi}] outside [0, {g.num_nodes})")
        self.batch_size, self.shuffle, self.drop_last = int(batch_size), bool(shuffle), bool(drop_last)
        self.generator = generator

    def __len__(self):
        n = int(self.nids.numel())
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        nids = self.nids
        if self.shuffle:
            nids = nids[torch.randperm(int(nids.numel()), generator=self.generator, device=nids.device)]
        for i in range(len(self)):
            seeds = nids[i * self.batch_size:(i + 1) * self.batch_size]
            blocks = self.sampler.sample_blocks(self.g, seeds)
            yield blocks[0].src_ids, seeds, blocks
