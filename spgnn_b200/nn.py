"""Conv modules with DGL's constructor signatures and state-dict names, computed by this repo's CUDA kernels.

Replaces ``from dgl.nn.pytorch import GATConv, GraphConv, SAGEConv, GINConv`` (/root/reference/models.py:8).
Semantics are DGL 0.7.x (SURVEY.md §8a A1/A4); the version switches live in ``DGL_COMPAT``.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from ._lib import SpgnnError

DGL_COMPAT = {
    "gat_bias": True,                    # GATConv bias parameter (added in DGL 0.7)
    "gat_res_identity_rule": "in!=F",    # 0.7.x; ">=0.8" uses "in!=H*F"
    "sage_bias_layout": "single",        # 0.7.x: fc_self/fc_neigh bias-free + one bias
}


class Linear(nn.Linear):
    """nn.Linear whose forward/backward run on spgnn kernels (optionally with a fused activation)."""

    def __init__(self, in_features, out_features, bias=True, act=None, slope=0.01):
        super().__init__(in_features, out_features, bias=bias)
        self._act, self._slope = act, slope

    def forward(self, x):
        return ops.linear(x, self.weight, self.bias, self._act, self._slope)


class Dropout(nn.Module):
    def __init__(self, p=0.5):
        super().__init__()
        self.p = p

    def forward(self, x):
        return ops.concat_dropout(x, None, self.p, self.training)


class LeakyReLU(nn.Module):
    """``fused=True``: a placeholder that keeps the reference's ``nn.Sequential`` indices (state-dict keys) while the
    activation itself runs in the epilogue of the preceding :class:`Linear` (``act="leaky_relu"``)."""

    def __init__(self, negative_slope=0.01, fused=False):
        super().__init__()
        self.negative_slope, self.fused = negative_slope, fused

    def forward(self, x):
        return x if self.fused else ops.bias_act(x, None, "leaky_relu", self.negative_slope)


class GATConv(nn.Module):
    """``GATConv(in_feats, out_feats, num_heads, feat_drop, attn_drop, negative_slope, residual, activation)``.

    forward(g, feat, feat2=None): ``feat2`` is an optional second input block; ``[feat | feat2]`` is projected
    without materialising the concatenation (models.py:477,481).  Returns [N, H, F].
    ``forward_flat(..., mean_heads=True)`` fuses the ``.mean(1)`` of the output layer (models.py:326,482).
    """

    def __init__(self, in_feats, out_feats, num_heads, feat_drop=0.0, attn_drop=0.0, negative_slope=0.2,
                 residual=False, activation=None, allow_zero_in_degree=False, bias=None):
        super().__init__()
        self._in_feats, self._out_feats, self._num_heads = in_feats, out_feats, num_heads
        self.feat_drop_p, self.attn_drop_p = float(feat_drop), float(attn_drop)
        self.negative_slope = negative_slope
        self._allow_zero_in_degree = allow_zero_in_degree
        self.fc = nn.Linear(in_feats, out_feats * num_heads, bias=False)
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        if residual:
            rule = DGL_COMPAT["gat_res_identity_rule"]
            linear = (in_feats != out_feats) if rule == "in!=F" else (in_feats != out_feats * num_heads)
            self.res_fc = nn.Linear(in_feats, num_heads * out_feats, bias=False) if linear else nn.Identity()
        else:
            self.register_buffer("res_fc", None)
        if DGL_COMPAT["gat_bias"] if bias is None else bias:
            self.bias = nn.Parameter(torch.empty(num_heads * out_feats))
        else:
            self.register_buffer("bias", None)
        self.activation = activation
        self._act = ops.act_code(activation)
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        nn.init.xavier_normal_(self.fc.weight, gain=gain)
        nn.init.xavier_normal_(self.attn_l, gain=gain)
        nn.init.xavier_normal_(self.attn_r, gain=gain)
        if self.bias is not None:
            nn.init.constant_(self.bias, 0)
        if isinstance(self.res_fc, nn.Linear):
            nn.init.xavier_normal_(self.res_fc.weight, gain=gain)

    def _packed_weight(self):
        """[W_fc ; W_res ; W_fc^T·attn_l ; W_fc^T·attn_r] with rows padded to 16 bytes: one projection yields
        z, the residual and both attention logits (el = x·(W_fc^T attn_l) ≡ (x W_fc^T)·attn_l)."""
        w_res = self.res_fc.weight if isinstance(self.res_fc, nn.Linear) else None
        return ops.PackWeightFn.apply(self.fc.weight, w_res, self.attn_l, self.attn_r, self._num_heads,
                                      self._out_feats)

    def forward_flat(self, g, feat, feat2=None, mean_heads=False):
        if not self._allow_zero_in_degree:
            g.check_no_zero_in_degree()
        H, F = self._num_heads, self._out_feats
        k_in = feat.shape[1] + (feat2.shape[1] if feat2 is not None else 0)
        if k_in != self._in_feats:
            raise SpgnnError(f"GATConv expects {self._in_feats} input features, got {k_in}")
        drop = self.feat_drop_p if self.training else 0.0
        if drop > 0.0:
            feat, feat2 = ops.concat_dropout(feat, feat2, drop, True), None
        res_mode = 0 if self.res_fc is None else (1 if isinstance(self.res_fc, nn.Linear) else 2)
        xres = None
        if res_mode == 2:
            xres = feat if feat2 is None else ops.concat_dropout(feat, feat2, 0.0, False)
        y = ops.linear(feat, self._packed_weight(), x2=feat2)
        return ops.GatAggFn.apply(y, xres, self.bias, g, H, F, res_mode, self._act, self.negative_slope,
                                  bool(mean_heads), self.attn_drop_p if self.training else 0.0, ops.next_seed())

    def forward(self, g, feat, feat2=None):
        return self.forward_flat(g, feat, feat2).view(-1, self._num_heads, self._out_feats)


class GraphConv(nn.Module):
    """``GraphConv(in_feats, out_feats, activation=)`` with norm='both' (models.py:172-182)."""

    def __init__(self, in_feats, out_feats, norm="both", weight=True, bias=True, activation=None,
                 allow_zero_in_degree=False):
        super().__init__()
        if norm != "both" or not weight or not bias:
            raise SpgnnError("GraphConv: only norm='both', weight=True, bias=True (what the reference uses)")
        self._in_feats, self._out_feats = in_feats, out_feats
        self.weight = nn.Parameter(torch.empty(in_feats, out_feats))
        self.bias = nn.Parameter(torch.empty(out_feats))
        self._activation = activation
        self._act = ops.act_code(activation)
        self._allow_zero_in_degree = allow_zero_in_degree
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.weight)
        nn.init.zeros_(self.bias)

    def forward(self, g, feat):
        if not self._allow_zero_in_degree:
            g.check_no_zero_in_degree()
        out_s, in_s, _, _ = g.norms()
        wt = self.weight.t().contiguous()          # [out, in]
        if self._in_feats > self._out_feats:       # project first, aggregate the narrower rows
            x = ops.linear(feat, wt)
            return ops.SpmmFn.apply(x, None, self.bias, g, out_s, in_s, self._act, 0.0)
        x = ops.SpmmFn.apply(feat, None, None, g, out_s, in_s, 0, 0.0)
        return ops.linear(x, wt, self.bias, self._activation)


class _LSTMParams(nn.Module):
    """The parameters of ``nn.LSTM(D, D, batch_first=True)`` under its state-dict names, with its
    ``reset_parameters``; the LSTM itself runs in ``ops.LstmReduceFn``."""

    def __init__(self, D):
        super().__init__()
        self.hidden_size = D
        self.weight_ih_l0 = nn.Parameter(torch.empty(4 * D, D))
        self.weight_hh_l0 = nn.Parameter(torch.empty(4 * D, D))
        self.bias_ih_l0 = nn.Parameter(torch.empty(4 * D))
        self.bias_hh_l0 = nn.Parameter(torch.empty(4 * D))
        self.reset_parameters()

    def reset_parameters(self):
        stdv = 1.0 / self.hidden_size ** 0.5
        for w in self.parameters():
            nn.init.uniform_(w, -stdv, stdv)


class SAGEConv(nn.Module):
    """``SAGEConv(in, out, aggregator_type, feat_drop, activation, norm)`` (models.py:668-679) with DGL 0.7's four
    aggregators: 'pool', 'mean', 'gcn' and 'lstm' (DESIGN.md §2).  Parameters and ``reset_parameters`` are DGL's:
    'pool' has ``fc_pool``, 'lstm' has ``lstm`` (an ``nn.LSTM(in, in)``'s tensors), 'gcn' has no ``fc_self``."""

    AGGREGATORS = ("pool", "mean", "gcn", "lstm")

    def __init__(self, in_feats, out_feats, aggregator_type="pool", feat_drop=0.0, bias=True, norm=None,
                 activation=None):
        super().__init__()
        if aggregator_type not in self.AGGREGATORS:
            raise SpgnnError(f"SAGEConv: aggregator_type must be one of {self.AGGREGATORS}, got {aggregator_type!r}")
        self._aggre_type = aggregator_type
        self._in_feats, self._out_feats = in_feats, out_feats
        self.feat_drop_p = float(feat_drop)
        self.norm, self.activation = norm, activation
        per_linear = DGL_COMPAT["sage_bias_layout"] == "per_linear"
        if aggregator_type == "pool":
            self.fc_pool = nn.Linear(in_feats, in_feats)
        if aggregator_type == "lstm":
            self.lstm = _LSTMParams(in_feats)
        if aggregator_type != "gcn":
            self.fc_self = nn.Linear(in_feats, out_feats, bias=per_linear)
        else:
            self.fc_self = None
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

    def _bias(self):
        b = self.bias
        if b is None and self.fc_neigh.bias is not None:
            b = self.fc_neigh.bias + (self.fc_self.bias if self.fc_self is not None else 0)
        return b

    def forward(self, g, feat):
        """``g``: a batched Graph, or a sampled ``sampling.Block`` (``feat`` then has one row per SOURCE node and the
        output one row per destination node: DGL's ``feat_dst = feat_src[:number_of_dst_nodes]``)."""
        is_block = getattr(g, "is_block", False)
        if is_block and feat.shape[0] != g.num_src_nodes:
            raise SpgnnError(f"SAGEConv: block has {g.num_src_nodes} source nodes, features have {feat.shape[0]} rows")
        h = ops.concat_dropout(feat, None, self.feat_drop_p, self.training)
        h_dst = h[:g.num_dst_nodes] if is_block else h
        b = self._bias()
        lin_before_mp = self._in_feats > self._out_feats
        agg = self._aggre_type
        if agg == "mean" and lin_before_mp:
            # mean_{u→v} fc_neigh(h)[u] + fc_self(h_dst) + bias, activation: self block and bias in the epilogue
            x = ops.linear(h, self.fc_neigh.weight)
            rst = ops.SpmmFn.apply(x, None, b, g, None, ops.inv_degree(g, 0), ops.act_code(self.activation), 0.0,
                                   ops.linear(h_dst, self.fc_self.weight))
        elif agg == "gcn":
            # (Σ_{u→v} x[u] + x[v]) / (in_deg(v) + 1), x = fc_neigh(h) before or after the aggregation
            if lin_before_mp:
                rst = ops.SpmmFn.apply(ops.linear(h, self.fc_neigh.weight), None, b, g, None, ops.inv_degree(g, 1),
                                       ops.act_code(self.activation), 0.0, None, True)
            else:
                neigh = ops.SpmmFn.apply(h, None, None, g, None, ops.inv_degree(g, 1), 0, 0.0, None, True)
                rst = ops.linear(neigh, self.fc_neigh.weight, b, self.activation)
        else:
            if agg == "pool":
                m = ops.linear(h, self.fc_pool.weight, self.fc_pool.bias, "relu")
                neigh = ops.MaxPoolFn.apply(m, g)
            elif agg == "mean":
                neigh = ops.SpmmFn.apply(h, None, None, g, None, ops.inv_degree(g, 0), 0, 0.0)
            else:
                lp = self.lstm
                P = ops.linear(h, lp.weight_ih_l0, lp.bias_ih_l0 + lp.bias_hh_l0)
                neigh = ops.LstmReduceFn.apply(P, lp.weight_hh_l0, g)
            # fc_self(h_dst) + fc_neigh(neigh) as ONE two-source projection
            w = torch.cat([self.fc_self.weight, self.fc_neigh.weight], 1)
            rst = ops.linear(h_dst, w, b, self.activation, x2=neigh)
        return self.norm(rst) if self.norm is not None else rst


class GINConv(nn.Module):
    """``GINConv(apply_func, 'mean', learn_eps=True)`` (models.py:358-383)."""

    def __init__(self, apply_func, aggregator_type, init_eps=0, learn_eps=False):
        super().__init__()
        if aggregator_type != "mean":
            raise SpgnnError("GINConv: only aggregator_type='mean' (the reference's setting) is implemented")
        self.apply_func = apply_func
        if learn_eps:
            self.eps = nn.Parameter(torch.FloatTensor([init_eps]))
        else:
            self.register_buffer("eps", torch.FloatTensor([init_eps]))

    def forward(self, g, feat):
        _, _, in_inv, _ = g.norms()
        rst = ops.SpmmFn.apply(feat, self.eps, None, g, None, in_inv, 0, 0.0)
        mlp = self.apply_func
        if mlp is None:
            return rst
        if _is_gin_mlp(mlp) and rst.is_cuda:
            # the reference's MLP in one Function: no dropout pass in either direction (ops.MlpDropFn)
            return ops.mlp_drop(rst, mlp[0].weight, mlp[0].bias, mlp[3].weight, mlp[3].bias, "leaky_relu",
                                mlp[0]._slope, mlp[1].p if mlp[1].training else 0.0)
        return mlp(rst)


def _is_gin_mlp(mlp):
    """Linear(leaky) → Dropout → [fused LeakyReLU] → Linear(leaky) → [fused LeakyReLU], as models.GIN builds it."""
    return (isinstance(mlp, nn.Sequential) and len(mlp) == 5 and isinstance(mlp[0], Linear) and
            isinstance(mlp[1], Dropout) and isinstance(mlp[2], LeakyReLU) and mlp[2].fused and
            isinstance(mlp[3], Linear) and isinstance(mlp[4], LeakyReLU) and mlp[4].fused and
            mlp[0]._act == "leaky_relu" and mlp[3]._act == "leaky_relu" and mlp[0]._slope == mlp[3]._slope)
