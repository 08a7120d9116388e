"""SAGEConv's mean / gcn / lstm aggregators: the oracle (DGL 0.7's op sequence, tests/sage_oracle.py) against
formulations it shares no code with, in fp64 — ``torch.sparse.mm`` with D^-1 A for mean, a scipy CSR (A + I) /
(deg + 1) for gcn, a per-node loop over ``nn.LSTMCell`` in edge-list order for lstm — on trees, on a sampled-style
Block and on a hand-made Block with an empty destination; plus the parameter surface of ``nn.SAGEConv`` and
``SAGENet`` against the oracle's (no GPU needed: modules are only constructed)."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import dgl_ops
from sage_oracle import SAGEConv, gnn_net
from spgnn_b200 import synth

AGGS = ("mean", "gcn", "lstm")


def _tree_graph(tree, fdim):
    sc = synth.make_scan(tree, k=9, fv_dim=fdim)
    g = dgl_ops.graph_from_adj(sc.adj)
    return g, torch.from_numpy(sc.fvs).double() + 0.1 * torch.randn(sc.adj.shape[0], fdim, dtype=torch.float64,
                                                                   generator=torch.Generator().manual_seed(tree))


def _block(empty_dst):
    """A Block shaped like a sampled one (destinations = first source rows, fanout-limited in-edges in edge-list
    order grouped by destination); ``empty_dst``: destination 2 gets no in-edge."""
    src = [0, 5, 1, 6, 7, 3, 8, 4, 9, 2]
    dst = [0, 0, 1, 1, 1, 2, 3, 3, 4, 4]
    if empty_dst:
        keep = [i for i, d in enumerate(dst) if d != 2]
        src, dst = [src[i] for i in keep], [dst[i] for i in keep]
    b = dgl_ops.Block(torch.tensor(src), torch.tensor(dst), 10, 5)
    return b, torch.randn(10, 12, dtype=torch.float64, generator=torch.Generator().manual_seed(4))


def _cases():
    g, x = _tree_graph(3, 12)
    yield "tree", g, x, g.num_nodes
    b, xb = _block(False)
    yield "block", b, xb, b.num_dst
    b, xb = _block(True)
    yield "block_empty_dst", b, xb, b.num_dst


def _conv(agg, fin, fout, act=None):
    torch.manual_seed(0)
    conv = SAGEConv(fin, fout, aggregator_type=agg, activation=act).double()
    with torch.no_grad():
        conv.bias.normal_(0, 0.1)
    return conv


def _mean_sparse(g, x, n):
    """D^-1 A with torch.sparse.mm (rows = destinations)."""
    deg = torch.bincount(g.dst, minlength=n).double().clamp(min=1)
    a = torch.sparse_coo_tensor(torch.stack([g.dst, g.src]), 1.0 / deg[g.dst], (n, x.shape[0])).coalesce()
    return torch.sparse.mm(a, x)


def _gcn_scipy(g, x, n):
    """(A + I) / (deg + 1) as a scipy CSR (the self loops of the graph are counted again, DGL's rule)."""
    d, s = g.dst.numpy(), g.src.numpy()
    deg = np.bincount(d, minlength=n).astype(np.float64)
    a = sp.csr_matrix((np.ones(len(d)), (d, s)), shape=(n, x.shape[0]))
    a = a + sp.csr_matrix((np.ones(n), (np.arange(n), np.arange(n))), shape=(n, x.shape[0]))
    a = sp.diags(1.0 / (deg + 1)) @ a
    return torch.from_numpy(a @ x.detach().numpy())


def _lstm_loop(lstm, g, x, n):
    """One nn.LSTMCell step per message, destination by destination, messages in edge-list order."""
    cell = torch.nn.LSTMCell(lstm.input_size, lstm.hidden_size).double()
    with torch.no_grad():
        cell.weight_ih.copy_(lstm.weight_ih_l0)
        cell.weight_hh.copy_(lstm.weight_hh_l0)
        cell.bias_ih.copy_(lstm.bias_ih_l0)
        cell.bias_hh.copy_(lstm.bias_hh_l0)
    out = []
    for v in range(n):
        h = c = torch.zeros(1, lstm.hidden_size, dtype=torch.float64)
        for e in (g.dst == v).nonzero().flatten().tolist():
            h, c = cell(x[g.src[e]].view(1, -1), (h, c))
        out.append(h[0])
    return torch.stack(out)


def _independent(conv, g, x, n, agg):
    lin_before_mp = conv._in > conv._out
    x_dst = x[:n]
    if agg == "mean":
        if lin_before_mp:
            rst = x_dst @ conv.fc_self.weight.t() + _mean_sparse(g, x @ conv.fc_neigh.weight.t(), n)
        else:
            rst = x_dst @ conv.fc_self.weight.t() + _mean_sparse(g, x, n) @ conv.fc_neigh.weight.t()
    elif agg == "gcn":
        if lin_before_mp:
            rst = _gcn_scipy(g, x @ conv.fc_neigh.weight.t().detach(), n)
        else:
            rst = _gcn_scipy(g, x, n) @ conv.fc_neigh.weight.t().detach()
    else:
        rst = x_dst @ conv.fc_self.weight.t() + _lstm_loop(conv.lstm, g, x, n) @ conv.fc_neigh.weight.t()
    return rst + conv.bias


@pytest.mark.parametrize("agg", AGGS)
@pytest.mark.parametrize("fout", [5, 20])          # 12 -> 5 projects before the aggregation, 12 -> 20 after
def test_oracle_aggregators_against_independent_formulations(agg, fout):
    for name, g, x, n in _cases():
        conv = _conv(agg, x.shape[1], fout)
        with torch.no_grad():
            got = conv(g, x)
            ref = _independent(conv, g, x, n, agg)
        assert got.shape == (n, fout)
        assert torch.allclose(got, ref, rtol=1e-10, atol=1e-12), (agg, name, float((got - ref).abs().max()))


def test_zero_in_degree_rules():
    """Hand-made Block, destination 2 without in-edges: mean and lstm give a zero neighbour term, gcn gives x[v]."""
    b, x = _block(True)
    for agg in AGGS:
        conv = _conv(agg, 12, 20)
        with torch.no_grad():
            got = conv(b, x)[2]
            if agg == "gcn":
                ref = x[2] @ conv.fc_neigh.weight.t() + conv.bias
            else:
                ref = x[2] @ conv.fc_self.weight.t() + conv.bias
        assert torch.allclose(got, ref, rtol=1e-12, atol=1e-12), agg


def test_lstm_reducer_gradcheck():
    """fp64 gradcheck of the oracle's degree-bucketed LSTM reducer (input messages and all LSTM parameters)."""
    g, _ = _tree_graph(1, 4)
    conv = _conv("lstm", 3, 2)
    x = torch.randn(g.num_nodes, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(2),
                    requires_grad=True)
    names = [k for k, _ in conv.named_parameters() if k.startswith("lstm.")]
    params = [dict(conv.named_parameters())[k].detach().clone().requires_grad_() for k in names]

    def f(x, *ps):
        return torch.func.functional_call(conv, dict(zip(names, ps)), (g, x))

    assert torch.autograd.gradcheck(f, (x, *params), eps=1e-6, atol=1e-7)


def test_pool_equals_the_committed_oracle():
    """The extension computes 'pool' exactly as oracle.dgl_ops.SAGEConv does, with the same parameters."""
    g, x = _tree_graph(2, 12)
    torch.manual_seed(3)
    a = dgl_ops.SAGEConv(12, 5).double()
    torch.manual_seed(3)
    b = SAGEConv(12, 5).double()
    assert list(a.state_dict()) == list(b.state_dict())
    assert all(torch.equal(a.state_dict()[k], b.state_dict()[k]) for k in a.state_dict())
    with torch.no_grad():
        assert torch.equal(a(g, x), b(g, x))


def test_state_dict_of_nn_sageconv_equals_the_oracle():
    from spgnn_b200 import nn as snn
    for agg in ("pool",) + AGGS:
        a = snn.SAGEConv(24, 8, aggregator_type=agg).state_dict()
        b = SAGEConv(24, 8, aggregator_type=agg).state_dict()
        assert list(a) == list(b), agg
        assert all(a[k].shape == b[k].shape for k in a), agg
    assert "fc_self.weight" not in snn.SAGEConv(24, 8, aggregator_type="gcn").state_dict()


def test_unknown_aggregator_raises():
    from spgnn_b200 import nn as snn
    from spgnn_b200._lib import SpgnnError
    with pytest.raises(SpgnnError):
        snn.SAGEConv(8, 8, aggregator_type="max")


@pytest.mark.parametrize("agg,count", [("pool", 1_897_366), ("mean", 761_302), ("gcn", 392_662),
                                       ("lstm", 9_849_814)])
def test_sagenet_parameter_counts_at_st_sage_3_widths(agg, count):
    from helpers import FULL_MODELS
    from spgnn_b200 import models as sm
    _, cfg = FULL_MODELS["st_sage_3"]
    net = sm.SAGENet(**cfg, aggregator_type=agg)
    n = sum(p.numel() for p in net.sage.parameters()) + sum(p.numel() for p in net.gnn_out.parameters())
    assert n == count
    onet = gnn_net(dict(cfg, aggregator_type=agg))
    assert sum(p.numel() for p in onet.parameters()) == count
    assert list(net.state_dict()) == [k for k in net.state_dict() if k in onet.state_dict()]
    net.load_state_dict(onet.state_dict(), strict=True)
