"""The device neighbour sampler (csrc/sampling.cu, sampling.DeviceBlockSampler) restated in numpy, and that
restatement checked on the CPU: against the torch sampler (same blocks when nothing is drawn, same inclusion
frequencies when something is), against the block invariants, and the host-side capacity bounds against the sizes
of exhaustively enumerated seed sets.  tests/test_gpu_device_sampler.py compares the kernel with the restatement
bit for bit."""
import itertools

import numpy as np
import torch

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


# ------------------------------------------------------------------------------------------------ the restatement
def mix64(x):
    """common.cuh mix64 (splitmix64 finaliser) on uint64 arrays."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def layer_base(seed, salt, layer):
    s = np.array([salt & 0xFFFFFFFFFFFFFFFF], dtype=np.uint64) ^ np.uint64(((layer + 1) << 56) & 0xFFFFFFFFFFFFFFFF)
    return mix64(np.array([seed & 0xFFFFFFFFFFFFFFFF], dtype=np.uint64) ^ mix64(s))[0]


def draw(in_ptr, u, fanout, base):
    """CSC slots kept for destination u: all when fanout < 0 or fanout >= degree, else the `fanout` smallest
    (key, slot) pairs with key = mix64(base ^ slot); ascending slot order."""
    slots = np.arange(in_ptr[u], in_ptr[u + 1], dtype=np.int64)
    if fanout < 0 or slots.size <= fanout:
        return slots
    keys = mix64(np.uint64(base) ^ slots.astype(np.uint64))
    pick = np.lexsort((slots, keys))[:fanout]                  # key first, ties to the lower slot
    return np.sort(slots[pick])


def sample_blocks(in_ptr, in_src, seeds, fanouts, seed, salt):
    """The blocks the kernel builds, input layer first: dicts of src_ids, in_ptr, in_src (local), out_ptr, out_dst,
    out_slot (numpy, int64)."""
    in_ptr, in_src = np.asarray(in_ptr, np.int64), np.asarray(in_src, np.int64)
    cur = np.asarray(seeds, np.int64)
    blocks = []
    for l in reversed(range(len(fanouts))):
        base = layer_base(seed, salt, l)
        kept = [draw(in_ptr, int(u), fanouts[l], base) for u in cur]
        cnt = np.array([k.size for k in kept], np.int64)
        slots = np.concatenate(kept) if kept else np.zeros(0, np.int64)
        src = in_src[slots]
        dst = np.repeat(np.arange(cur.size), cnt)
        extras = np.unique(src[~np.isin(src, cur)])             # ascending global id
        src_ids = np.concatenate([cur, extras])
        local = np.empty(src.size, np.int64)
        lookup = {int(u): i for i, u in enumerate(src_ids)}
        for e, u in enumerate(src):
            local[e] = lookup[int(u)]
        order = np.argsort(local, kind="stable")                 # out-CSR: stable counting sort by source
        blocks.insert(0, dict(src_ids=src_ids, in_ptr=np.concatenate([[0], np.cumsum(cnt)]), in_src=local,
                              out_ptr=np.concatenate([[0], np.cumsum(np.bincount(local, minlength=src_ids.size))]),
                              out_dst=dst[order], out_slot=order, num_dst=cur.size))
        cur = src_ids
    return blocks


def check_invariants(blocks, in_ptr, in_src, seeds):
    """src_ids[:S] are the destinations (the seeds for the last block), the extras are unique, ascending and
    disjoint from them, every kept edge is a graph edge drawn once, layers chain, and the out-CSR is the in-CSC
    transposed with out_slot pointing back into it (numpy arrays)."""
    in_ptr, in_src = np.asarray(in_ptr, np.int64), np.asarray(in_src, np.int64)
    dst_ids = np.asarray(seeds, np.int64)
    for b in reversed(blocks):
        src_ids, S = b["src_ids"], dst_ids.size
        assert np.array_equal(src_ids[:S], dst_ids)
        ex = src_ids[S:]
        assert np.all(ex[1:] > ex[:-1]) and not np.isin(ex, dst_ids).any()
        ip, isrc = b["in_ptr"], b["in_src"]
        assert ip.size == S + 1 and ip[0] == 0 and np.all(np.diff(ip) >= 0) and isrc.size == ip[-1]
        for i, u in enumerate(dst_ids):
            nbrs = src_ids[isrc[ip[i]:ip[i + 1]]]
            graph_nbrs = in_src[in_ptr[u]:in_ptr[u + 1]]
            assert np.isin(nbrs, graph_nbrs).all()
            assert np.unique(nbrs).size == nbrs.size or np.unique(graph_nbrs).size < graph_nbrs.size
        used = np.zeros(src_ids.size, bool)
        used[isrc] = True
        assert used[S:].all()                                   # every extra is the source of a kept edge
        op, od, osl = b["out_ptr"], b["out_dst"], b["out_slot"]
        assert op.size == src_ids.size + 1 and op[-1] == isrc.size and np.all(np.diff(op) >= 0)
        assert np.array_equal(np.sort(osl), np.arange(isrc.size))
        src_of_out = np.repeat(np.arange(src_ids.size), np.diff(op))
        assert np.array_equal(isrc[osl], src_of_out)
        dst_of_in = np.repeat(np.arange(S), np.diff(ip))
        assert np.array_equal(dst_of_in[osl], od)
        for s in range(src_ids.size):                            # stable: in-CSC order inside every source
            assert np.all(np.diff(osl[op[s]:op[s + 1]]) > 0)
        dst_ids = src_ids


# ------------------------------------------------------------------------------------------------ graphs
def csc(num_nodes, src, dst):
    """in-CSC (in_ptr, in_src) with ascending edge id per destination, as spgnn_batch_build writes it."""
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    order = np.argsort(dst, kind="stable")
    in_ptr = np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=num_nodes))])
    return in_ptr, src[order]


def tree_edges(n, max_children, rng, self_loops=True):
    parent = [-1]
    kids = np.zeros(n, np.int64)
    for i in range(1, n):
        p = int(rng.choice(np.flatnonzero(kids[:i] < max_children)))
        kids[p] += 1
        parent.append(p)
    src, dst = [], []
    for i in range(1, n):
        src += [i, parent[i]]
        dst += [parent[i], i]
    if self_loops:
        src += list(range(n))
        dst += list(range(n))
    return src, dst


class _HostGraph:
    def __init__(self, num_nodes, in_ptr, in_src):
        self.num_nodes = num_nodes
        self.in_ptr = torch.from_numpy(np.asarray(in_ptr)).to(torch.int32)
        self.in_src = torch.from_numpy(np.asarray(in_src)).to(torch.int32)


# ------------------------------------------------------------------------------------------------ tests
def test_restatement_meets_the_block_invariants():
    rng = np.random.default_rng(0)
    src, dst = tree_edges(200, 6, rng)
    in_ptr, in_src = csc(200, src, dst)
    seeds = rng.permutation(200)[:40]
    for fanouts in ([0], [1], [2], [50], [-1], [2, 2, 2, 2], [1, 3, -1, 2], [0, 2, 1, 2]):
        for salt in range(3):
            check_invariants(sample_blocks(in_ptr, in_src, seeds, fanouts, 11, salt), in_ptr, in_src, seeds)


def test_restatement_equals_the_torch_sampler_when_nothing_is_drawn():
    """fanout -1 / fanout >= every degree keeps every edge: the blocks are fixed, and both samplers must build the
    same ones (extras order, local ids, CSC and CSR)."""
    from spgnn_b200 import sampling
    rng = np.random.default_rng(1)
    src, dst = tree_edges(150, 4, rng)
    in_ptr, in_src = csc(150, src, dst)
    hg = _HostGraph(150, in_ptr, in_src)
    seeds = rng.permutation(150)[:30]
    for fanouts in ([-1], [-1, -1, -1], [10, -1, 10]):
        mine = sample_blocks(in_ptr, in_src, seeds, fanouts, 5, 0)
        ref = sampling.MultiLayerNeighborSampler(fanouts).sample_blocks(hg, torch.from_numpy(seeds))
        for a, b in zip(mine, ref):
            assert np.array_equal(a["src_ids"], b.src_ids.numpy())
            for k in ("in_ptr", "in_src", "out_ptr", "out_dst", "out_slot"):
                assert np.array_equal(a[k], getattr(b, k).numpy().astype(np.int64)), k


def test_restatement_and_torch_sampler_keep_each_in_edge_equally_often():
    """Different random streams, same distribution: over many draws each in-edge of a degree-d destination is kept
    min(f, d)/d of the time by both samplers (d = 7: six children and a self loop)."""
    from spgnn_b200 import sampling
    d, f, n = 7, 2, 3000
    src = list(range(1, d)) + [0]
    dst = [0] * d
    in_ptr, in_src = csc(d, src, dst)
    hg = _HostGraph(d, in_ptr, in_src)
    gen = torch.Generator().manual_seed(3)
    mine = np.zeros(d)
    theirs = np.zeros(d)
    for salt in range(n):
        mine[draw(in_ptr, 0, f, layer_base(9, salt, 0)) - in_ptr[0]] += 1
        s, _ = sampling.sample_neighbors(hg, torch.tensor([0]), f, gen)
        theirs[[int(np.flatnonzero(in_src == u)[0]) for u in s.tolist()]] += 1
    want = n * f / d
    from scipy.stats import chisquare
    assert chisquare(mine, np.full(d, want)).pvalue > 1e-3, mine
    assert chisquare(theirs, np.full(d, want)).pvalue > 1e-3, theirs
    assert np.abs(mine - theirs).max() < 6 * np.sqrt(want)


def test_capacities_bound_every_seed_set_and_salt():
    """block_capacities against brute force: every seed set of a few small graphs (all subsets of a given size) under
    several salts, and the bound reached where every draw adds new nodes (disjoint in-neighbourhoods)."""
    from spgnn_b200 import sampling
    rng = np.random.default_rng(2)
    graphs = []
    s, d = tree_edges(9, 3, rng)
    graphs.append((9, s, d))
    graphs.append((8, [1, 2, 3, 4, 5, 6, 7], [0] * 7))                           # a star, zero-in-degree leaves
    graphs.append((7, [0, 1, 2, 3, 4, 5], [1, 2, 3, 4, 5, 6]))                   # a chain: node 0 has no in-edge
    for N, s, d in graphs:
        in_ptr, in_src = csc(N, s, d)
        maxdeg = int(max(np.diff(in_ptr).max(), np.bincount(s, minlength=N).max()))
        for fanouts in ([1], [2, 1], [-1, 2], [3, 0, -1]):
            for S in (1, 2, 3):
                caps = sampling.block_capacities(N, len(s), S, fanouts, maxdeg)
                for seeds in itertools.combinations(range(N), S):
                    for salt in range(3):
                        bl = sample_blocks(in_ptr, in_src, np.array(seeds), fanouts, 1, salt)
                        for b, (cd, cs, ce) in zip(bl, caps):
                            assert b["num_dst"] <= cd and b["src_ids"].size <= cs and b["in_src"].size <= ce
    # attained: 4 destinations with 3 private in-neighbours each, fanout 2, one layer -> 4 + 8 sources, 8 edges
    s = [4 + 3 * i + k for i in range(4) for k in range(3)]
    d = [i for i in range(4) for _ in range(3)]
    in_ptr, in_src = csc(16, s, d)
    (cd, cs, ce), = sampling.block_capacities(16, len(s), 4, [2])
    b, = sample_blocks(in_ptr, in_src, np.arange(4), [2], 0, 0)
    assert (cd, cs, ce) == (4, 12, 8) == (b["num_dst"], b["src_ids"].size, b["in_src"].size)


def test_capacities_refuse_what_int32_cannot_index():
    import pytest
    from spgnn_b200 import sampling
    from spgnn_b200._lib import SpgnnError
    with pytest.raises(SpgnnError):
        sampling.block_capacities(2 ** 33, 2 ** 34, 2 ** 31, [2])
    with pytest.raises(SpgnnError):
        sampling.block_capacities(100, 300, 10, [-1])                             # fanout -1 needs max_degree
    assert sampling.block_capacities(100, 300, 10, [-1], max_degree=4) == [(10, 50, 40)]
