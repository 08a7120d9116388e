"""The SAGEConv lstm reducer (ops.LstmReduceFn: the device sort of csrc/sage_lstm.cu, the fused cell kernels, the
recurrent planes GEMMs and the dP gather) called directly, forward and backward, against an fp64 LSTM over every
destination's in-edge messages in in-CSC order: long recurrences whose steps hold one to three rows at unaligned row
offsets, feature widths that are not multiples of 64, zero in-degrees, sampled blocks with sources that send nothing,
and both sides of the in-degree limit of the sort."""
import numpy as np
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu

MAX_SORT_DEGREE = 12287          # the largest in-degree the device sort accepts
TOL = 1e-4
GRAD_TOL = 2e-4


@pytest.fixture(scope="module")
def mods():
    from spgnn_b200 import graph as sg, ops, sampling
    from spgnn_b200._lib import SpgnnError, lib
    return dict(sg=sg, ops=ops, sampling=sampling, SpgnnError=SpgnnError, lib=lib)


def lstm_ref(P, W, in_ptr, in_src, n_dst):
    """h_T of an LSTM (zero initial state, gates i, f, g, o) over P[in_src[in_ptr[v] + t]], t < in-degree of v, for
    every destination v; rows are taken by descending in-degree so that step t is a prefix of them."""
    D = W.shape[1]
    deg = in_ptr[1:n_dst + 1] - in_ptr[:n_dst]
    order = torch.sort(-deg, stable=True)[1]
    ds = deg[order]
    out_rows, out_h = [], []
    h = torch.zeros(0, D, dtype=P.dtype)
    c = torch.zeros(0, D, dtype=P.dtype)
    for t in range(int(deg.max()) if n_dst else 0):
        n_t = int((ds > t).sum())
        rows = order[:n_t]
        z = P[in_src[in_ptr[rows] + t]]
        if t > 0:
            z = z + h[:n_t] @ W.t()
        i, f, g, o = torch.sigmoid(z[:, :D]), torch.sigmoid(z[:, D:2 * D]), torch.tanh(z[:, 2 * D:3 * D]), \
            torch.sigmoid(z[:, 3 * D:])
        c = (f * c[:n_t] + i * g) if t > 0 else i * g
        h = o * torch.tanh(c)
        end = ds[:n_t] == t + 1
        out_rows.append(rows[end])
        out_h.append(h[end])
    out = torch.zeros(n_dst, D, dtype=P.dtype)
    if out_rows:
        out = out.index_copy(0, torch.cat(out_rows), torch.cat(out_h))
    return out


def _graph(mods, kind, rng):
    sg, sampling = mods["sg"], mods["sampling"]
    if kind == "hub":
        # node 0 receives 300 messages, nodes 1..3 receive 2, 3, 9, every node a self loop on top: 301 steps, most of
        # them one row, the first few two or three rows that start at row offsets that are not multiples of 8
        n = 400
        src = list(range(1, 301)) + [5, 6] + [7, 8, 9] + list(range(10, 19)) + list(range(n))
        dst = [0] * 300 + [1, 1] + [2, 2, 2] + [3] * 9 + list(range(n))
        perm = rng.permutation(len(src))
        return sg.from_edges(np.array(src)[perm], np.array(dst)[perm], n)
    if kind == "mixed":
        n = 3000
        deg = rng.integers(0, 13, n)
        dst = np.repeat(np.arange(n), deg)
        src = rng.integers(0, n, dst.size)
        perm = rng.permutation(dst.size)
        return sg.from_edges(src[perm], dst[perm], n)
    # sampled block: 300 destinations (the first source rows), 900 sources, sources 700.. send nothing
    n_dst, n_src = 300, 900
    deg = rng.integers(0, 11, n_dst)
    dst = torch.from_numpy(np.repeat(np.arange(n_dst), deg)).cuda()
    src = torch.from_numpy(rng.integers(0, 700, dst.numel())).cuda()
    return sampling.Block(src, dst, torch.arange(n_src, device="cuda") + 5000, n_dst)


def _n_dst(g):
    return g.num_dst_nodes if getattr(g, "is_block", False) else g.num_nodes


def _n_src(g):
    return g.num_src_nodes if getattr(g, "is_block", False) else g.num_nodes


def _run(mods, g, D, seed):
    """Device forward + backward and the fp64 reference of both; returns (device, reference) triples
    (out, dP, dW_hh)."""
    ops = mods["ops"]
    n_src, n_dst = _n_src(g), _n_dst(g)
    gen = torch.Generator().manual_seed(seed)
    P = torch.randn(n_src, 4 * D, generator=gen)
    W = torch.randn(4 * D, D, generator=gen) / D ** 0.5
    go = torch.randn(n_dst, D, generator=gen)
    Pc, Wc = P.cuda().requires_grad_(), W.cuda().requires_grad_()
    out = ops.LstmReduceFn.apply(Pc, Wc, g)
    out.backward(go.cuda())
    P64, W64 = P.double().requires_grad_(), W.double().requires_grad_()
    in_ptr, in_src = g.in_ptr.long().cpu(), g.in_src.long().cpu()
    ref = lstm_ref(P64, W64, in_ptr, in_src, n_dst)
    ref.backward(go.double())
    return (out.detach().cpu(), Pc.grad.cpu(), Wc.grad.cpu()), (ref.detach(), P64.grad, W64.grad)


def _check(dev, ref, tag):
    assert rel_err(dev[0], ref[0]) < TOL, (tag, "out")
    assert rel_err(dev[1], ref[1]) < GRAD_TOL, (tag, "dP")
    assert rel_err(dev[2], ref[2]) < GRAD_TOL, (tag, "dW_hh")


@pytest.mark.parametrize("D", [4, 36, 64, 260])
@pytest.mark.parametrize("kind", ["hub", "mixed", "block"])
def test_lstm_reducer_against_fp64(mods, kind, D):
    rng = np.random.default_rng(D + len(kind))
    g = _graph(mods, kind, rng)
    dev, ref = _run(mods, g, D, seed=D * 13 + len(kind))
    o = mods["ops"].lstm_order(g)
    deg = (g.in_ptr[1:_n_dst(g) + 1] - g.in_ptr[:_n_dst(g)]).cpu()
    assert o.steps == [int((deg > t).sum()) for t in range(int(deg.max()))]
    if kind == "hub":
        assert len(o.steps) == 301 and sum(s == 1 for s in o.steps) == 291
        assert {2, 3} <= set(o.steps) and any(off % 8 for off, s in zip(o.off, o.steps) if s in (2, 3))
    elif kind == "mixed":
        assert len(o.steps) == 12 and int((deg == 0).sum()) > 0
        assert torch.equal(dev[0][deg == 0], torch.zeros(int((deg == 0).sum()), D))
    else:
        silent = (g.out_ptr[1:] == g.out_ptr[:-1]).cpu()
        assert g.num_src_nodes > g.num_dst_nodes and bool(silent[700:].all())
        assert torch.equal(dev[1][silent], torch.zeros(int(silent.sum()), 4 * D))
        assert dev[0].shape == (g.num_dst_nodes, D)
    _check(dev, ref, (kind, D))


def _star(mods, degree):
    """Node 0 receives one message from each of nodes 1..degree; nothing else."""
    return mods["sg"].from_edges(np.arange(1, degree + 1), np.zeros(degree, dtype=np.int64), degree + 1)


def test_the_sort_at_its_largest_in_degree(mods):
    """In-degree 12287, the largest the device sort takes: its scatter then stages 12289 counters (48 KB + 4 bytes of
    shared memory).  12287 LSTM steps of one row each, against fp64."""
    g = _star(mods, MAX_SORT_DEGREE)
    dev, ref = _run(mods, g, 4, seed=1)
    o = mods["ops"].lstm_order(g)
    assert len(o.steps) == MAX_SORT_DEGREE and set(o.steps) == {1}
    assert o.perm.cpu()[0] == 0
    _check(dev, ref, "star")


def test_the_sort_refuses_a_larger_in_degree_before_launching(mods):
    g = _star(mods, MAX_SORT_DEGREE + 1)
    L = mods["lib"]()
    before = L.launch_count()
    with pytest.raises(mods["SpgnnError"], match="in-degree above the sort's key range"):
        mods["ops"].lstm_order(g)
    assert L.launch_count() == before
    assert "_lstm_order" not in g.__dict__
