"""CPU oracle for SAGEConv's mean / gcn / lstm aggregators (DGL 0.7.x, restated from its source; DESIGN.md §2).

TEST INFRASTRUCTURE, like ``oracle/``: the committed oracle restates the reference's shipped setting
(``aggregator_type='pool'``) and stays as it is; this module extends it, for the tests, with the three other
aggregators DGL 0.7 accepts.  ``SAGEConv`` subclasses ``oracle.dgl_ops.SAGEConv`` (so ``oracle.models``' stacks
reset it like any other conv) and computes pool exactly as the parent does; ``gnn_net`` is ``oracle.models.GNNNet``
for a SAGENet with a given aggregator.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import dgl_ops, kinks, models as om
from oracle.dgl_ops import Block, _seg_sum


class SAGEConv(dgl_ops.SAGEConv):
    """DGL 0.7.x SAGEConv with aggregator_type 'pool', 'mean', 'gcn' or 'lstm'.

    ``lin_before_mp = in_feats > out_feats`` decides whether mean / gcn project before or after the aggregation;
    'gcn' has no fc_self and computes (Σ_{u→v} x[u] + x[v]) / (in_deg(v) + 1) (v counted again when the graph already
    has self loops: DGL's rule); 'lstm' runs ``nn.LSTM(in, in, batch_first=True)`` from a zero state over each
    destination's mailbox (DGL's degree buckets), messages in edge-list order, and feeds the final hidden state to
    fc_neigh.  Zero in-degree: mean and lstm give a zero neighbour term, gcn gives x[v]."""

    def __init__(self, in_feats, out_feats, aggregator_type="pool", feat_drop=0.0, bias=True,
                 norm=None, activation=None):
        nn.Module.__init__(self)
        assert aggregator_type in ("pool", "mean", "gcn", "lstm")
        self._aggre_type = aggregator_type
        self._in, self._out = in_feats, out_feats
        self.feat_drop = nn.Dropout(feat_drop)
        self.norm, self.activation = norm, activation
        if aggregator_type == "pool":
            self.fc_pool = nn.Linear(in_feats, in_feats)
        if aggregator_type == "lstm":
            self.lstm = nn.LSTM(in_feats, in_feats, batch_first=True)
        per_linear = dgl_ops.VERSION_SWITCHES["sage_bias_layout"] == "per_linear"
        if aggregator_type != "gcn":
            self.fc_self = nn.Linear(in_feats, out_feats, bias=per_linear)
        self.fc_neigh = nn.Linear(in_feats, out_feats, bias=per_linear)
        if not per_linear and bias:
            self.bias = nn.Parameter(torch.zeros(out_feats))
        else:
            self.register_buffer("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        if self._aggre_type == "pool":
            nn.init.xavier_uniform_(self.fc_pool.weight, gain=gain)
        if self._aggre_type == "lstm":
            self.lstm.reset_parameters()
        if self._aggre_type != "gcn":
            nn.init.xavier_uniform_(self.fc_self.weight, gain=gain)
        nn.init.xavier_uniform_(self.fc_neigh.weight, gain=gain)

    def _lstm_reducer(self, m_edges, dst, n):
        """DGL's degree-bucketed mailbox: per in-degree d, the destinations of that degree each get their d messages
        in edge-list order, [B, d, D], and nn.LSTM from a zero state reduces them to h_d."""
        neigh = m_edges.new_zeros(n, m_edges.shape[1])
        order = torch.sort(dst, stable=True)[1]                    # edge positions grouped by destination
        deg = torch.bincount(dst, minlength=n)
        start = torch.cumsum(deg, 0) - deg
        for d in sorted(set(deg.tolist()) - {0}):
            nodes = (deg == d).nonzero().flatten()
            idx = order[start[nodes].view(-1, 1) + torch.arange(d).view(1, -1)]
            _, (h, _) = self.lstm(m_edges[idx])
            neigh[nodes] = h[0]
        return neigh

    def forward(self, g, feat):
        if self._aggre_type == "pool":
            return super().forward(g, feat)
        h = kinks.dropout(self.feat_drop, feat)
        n = g.num_dst if isinstance(g, Block) else g.num_nodes       # DGL: feat_dst = feat_src[:number_of_dst_nodes()]
        h_dst = h[:n]
        lin_before_mp = self._in > self._out
        agg = self._aggre_type
        if agg == "mean":
            x = self.fc_neigh(h) if lin_before_mp else h
            deg = torch.bincount(g.dst, minlength=n).to(x.dtype).clamp(min=1)
            neigh = _seg_sum(x[g.src], g.dst, n) / deg.view(-1, 1)
            rst = self.fc_self(h_dst) + (neigh if lin_before_mp else self.fc_neigh(neigh))
        elif agg == "gcn":
            x = self.fc_neigh(h) if lin_before_mp else h
            deg = torch.bincount(g.dst, minlength=n).to(x.dtype)
            neigh = (_seg_sum(x[g.src], g.dst, n) + x[:n]) / (deg.view(-1, 1) + 1)
            rst = neigh if lin_before_mp else self.fc_neigh(neigh)
        else:
            rst = self.fc_self(h_dst) + self.fc_neigh(self._lstm_reducer(h[g.src], g.dst, n))
        if self.bias is not None:
            rst = rst + self.bias
        if self.activation is not None:
            rst = self.activation(rst)
        if self.norm is not None:
            rst = self.norm(rst)
        return rst


def gnn_net(model):
    """``oracle.models.GNNNet("sage", model)`` with every SAGEConv built for ``model["aggregator_type"]``: the same
    layer widths, feat_drop and activations as ``oracle.models.SAGE`` (models.py:650-696)."""
    agg = model.get("aggregator_type", "pool")
    net = om.GNNNet("sage", dict(model, aggregator_type="pool"))
    m = model
    dims = [m["fv_dim"]] + list(m["num_hiddens"][:m["num_layers"]])
    layers = [SAGEConv(dims[i], dims[i + 1], aggregator_type=agg, feat_drop=0.0 if i == 0 else m["feat_drop"],
                       activation=F.elu) for i in range(m["num_layers"])]
    layers.append(SAGEConv(dims[-1], m["node_embed_dim"], aggregator_type=agg))
    net.sage.g_layers = nn.ModuleList(layers)
    return net
