"""autograd.Function wrappers over the C ABI (include/spgnn_b200.h).  PyTorch here is plumbing: it owns the
device memory and the autograd tape; every arithmetic step below is one of this repo's CUDA kernels.

No fallbacks: CPU tensors raise.
"""
from __future__ import annotations

import torch
from torch.autograd import Function

from ._lib import SpgnnError, lib, ptr, require_cuda, stream

ACT = {None: 0, "none": 0, "elu": 1, "tanh": 2, "relu": 3, "leaky_relu": 4}

# The one projection arithmetic: the planes + TMA-fed tcgen05 GEMMs of csrc/gemm_tma.cu, behind ``linear``, the GIN
# MLP, the LSTM reducer and the GAT stacks alike.  bench.py sets GEMM_MODE from --gemm-mode and writes it into its JSON
# line; stack.planes_linear refuses any value but 2, so no run is reported under a mode it did not use.
GEMM_MODE = 2

# Test hook (oracle/kinks.py replays it): when a list, every non-smooth decision the path takes is appended in call
# order — ("sign", bool mask: pre-activation of a LeakyReLU / ReLU > 0), ("argmax", source node of every max-pooled
# element), ("drop", dropout mask already scaled by 1/(1-p)) — so a checker can take the same branches and compare
# gradients exactly, in train mode too.  None (production): no extra work.
KINK_TRACE = None


def tracing():
    return KINK_TRACE is not None


def trace(kind, value):
    KINK_TRACE.append((kind, value.detach()))


def drop_mask(rows, cols, p, seed, device):
    """The mask ``concat_dropout`` / attention dropout applies for (p, seed): u01(seed, row*cols + col) >= p."""
    ones = torch.ones(rows, cols, dtype=torch.float32, device=device)
    return ConcatDropoutFn.apply(ones, None, float(p), seed)[:, :cols].contiguous()


def trace_gat(graph, el, er, attn_p, attn_seed):
    """GATConv's decisions: LeakyReLU branch of every attention logit and the attention-dropout mask, in DGL edge
    order ([E, H, 1], the shape of DGL's edge data)."""
    trace("sign", ((el[graph.src] + er[graph.dst]) > 0).unsqueeze(-1))
    if attn_p > 0.0:
        H = el.shape[1]
        slot_mask = drop_mask(graph.num_edges, H, attn_p, attn_seed, el.device)      # in-CSC slot order
        edge_mask = torch.empty_like(slot_mask)
        edge_mask[graph.in_eid.long()] = slot_mask
        trace("drop", edge_mask.unsqueeze(-1))


_seed_state = {"seed": 0x5350474E, "counter": 0}


def manual_seed(seed: int):
    """Seed of the dropout / node-sampling masks (counter-hash based, regenerated in backward)."""
    _seed_state["seed"] = int(seed) & 0xFFFFFFFFFFFFFFFF
    _seed_state["counter"] = 0


def next_seed() -> int:
    _seed_state["counter"] += 1
    return (_seed_state["seed"] * 0x9E3779B97F4A7C15 + _seed_state["counter"] * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF


def act_code(act):
    """Map an activation given as a name, None or a torch callable (F.elu, torch.tanh, ...) to the ABI code."""
    if act is None or isinstance(act, str):
        return ACT[act]
    name = getattr(act, "__name__", "")
    if name in ("elu", "tanh", "relu", "leaky_relu"):
        return ACT[name]
    raise SpgnnError(f"unsupported activation {act!r} (supported: elu, tanh, relu, leaky_relu, None)")


def _pad4(n):
    return (n + 3) // 4 * 4


def _rows(t):
    """Row-major 2-D view requirements: unit inner stride."""
    if t.dim() != 2 or t.stride(1) != 1:
        t = t.contiguous()
    return t


def empty_padded(rows, cols, device):
    """[rows, cols] fp32 view of a buffer whose leading dimension is padded to a multiple of 4 (16-byte rows)."""
    return torch.empty(rows, _pad4(cols), dtype=torch.float32, device=device)[:, :cols]


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def colsum(x):
    x = _rows(x)
    M, N = x.shape
    out = torch.empty(N, dtype=torch.float32, device=x.device)
    ws = torch.empty(int(lib().colsum_ws(N)), dtype=torch.uint8, device=x.device)
    lib().colsum(ptr(x), x.stride(0), M, N, ptr(out), ptr(ws), stream())
    return out


def _planes_of(x):
    """Planes of an fp32 activation, converted once per tensor: a tensor feeding several projections (SAGEConv's
    ``h`` goes to fc_pool and fc_self) is split a single time.  The planes ride on the tensor object and are
    dropped with it; an in-place update (version counter) invalidates them."""
    from . import stack
    c = getattr(x, "_spgnn_planes", None)
    if c is not None and c[0] == x._version and c[1].buf.device == x.device:
        return c[1]
    P = stack.split_planes(x)
    try:
        x._spgnn_planes = (x._version, P)
    except Exception:
        pass
    return P


class PlanesLinearFn(Function):
    """y = act([x1 | x2] @ W^T + bias) through the planes pipeline: the inputs are converted to
    split-bf16 planes once (``spgnn_split_planes``), the projection and both of its gradients are the TMA-fed
    tcgen05 GEMMs of csrc/gemm_tma.cu, and the backward keeps the input PLANES (same bytes as the fp32 input)."""

    @staticmethod
    def forward(ctx, x1, x2, W, bias, act, slope):
        from . import stack
        require_cuda(x1, x2, W, bias)
        W = _rows(W)
        K1 = x1.shape[1]
        K2 = x2.shape[1] if x2 is not None else 0
        if W.shape[1] != K1 + K2:
            raise SpgnnError(f"linear: weight has {W.shape[1]} columns, input has {K1}+{K2}")
        P1 = _planes_of(x1)
        P2 = _planes_of(x2) if x2 is not None else None
        b = bias.contiguous() if bias is not None else None
        y = stack.planes_linear(P1, W, b, act, float(slope), A2=P2)
        need = ctx.needs_input_grad
        ctx.planes = (P1, P2) if need[2] else None          # only the weight gradient reads the inputs again
        ctx.save_for_backward(W, y if act else None)
        ctx.cfg = (act, float(slope), bias is not None, K1, K2)
        return y

    @staticmethod
    def backward(ctx, g):
        from . import stack
        W, y = ctx.saved_tensors
        act, slope, has_bias, K1, K2 = ctx.cfg
        g = _rows(g)
        M, N = g.shape
        dx1 = dx2 = dW = db = None
        want_db = has_bias and ctx.needs_input_grad[3]
        n4 = _pad4(N)
        if (g.stride(0) % 4 == 0 and g.stride(0) >= n4 and g.data_ptr() % 16 == 0 and
                (not act or (y.stride(0) % 4 == 0 and y.stride(0) >= n4 and y.data_ptr() % 16 == 0))):
            # one pass: d = g * act'(y) -> planes (+ bias gradient)
            L = lib()
            gp = stack.Planes(M, N, g.device)
            db = torch.empty(N, dtype=torch.float32, device=g.device) if want_db else None
            ws = _ws(L.act_bwd_planes_ws(N), g.device) if want_db else None
            L.act_bwd_planes(ptr(g), g.stride(0), ptr(y) if act else None, y.stride(0) if act else 0, act, slope,
                             0.0, 0, gp.ptr(), gp.ld, gp.ps, M, N, ptr(db), ptr(ws), stream(),
                             _key=("bytes", (12.0 if act else 8.0) * M * N))
            want_db = False
        else:
            if act:
                d = empty_padded(M, N, g.device)
                lib().act_bwd(ptr(g), g.stride(0), ptr(y), y.stride(0), act, slope, ptr(d), d.stride(0), M, N, stream())
                g = d
            gp = stack.split_planes(g)
        if ctx.needs_input_grad[0]:
            dx1 = stack.planes_linear_bwd_input(gp, W, K1, 0)
        if K2 and ctx.needs_input_grad[1]:
            dx2 = stack.planes_linear_bwd_input(gp, W, K2, K1)
        if ctx.needs_input_grad[2]:
            P1, P2 = ctx.planes
            dW = stack.planes_linear_bwd_weight(gp, P1, P2)
            ctx.planes = None
        if want_db:
            db = colsum(g)
        return dx1, dx2, dW, db, None, None


class MlpDropFn(Function):
    """y = act(W3 · dropout(act(W0·x + b0), p) + b3) — the MLP of the reference's GINConv layers (Linear → Dropout(0.1)
    → LeakyReLU → Linear → LeakyReLU, models.py:358-383, with the activation moved in front of the dropout: the two
    commute) — without a dropout pass in either direction: the mask is applied where the hidden activation is converted
    to planes for the second projection (``spgnn_split_planes(p, seed)``) and, in the backward, where the gradient of
    the dropped tensor is read by the fused ``spgnn_act_bwd_planes`` pass (same (seed, chunk) hash)."""

    @staticmethod
    def forward(ctx, x, W0, b0, W3, b3, act, slope, p, seed):
        from . import stack
        require_cuda(x, W0, b0, W3, b3)
        W0, W3 = _rows(W0), _rows(W3)
        if W0.shape[1] != x.shape[1] or W3.shape[1] != W0.shape[0]:
            raise SpgnnError(f"mlp: shapes {tuple(x.shape)} -> {tuple(W0.shape)} -> {tuple(W3.shape)} do not chain")
        P0 = _planes_of(x)
        y1 = stack.planes_linear(P0, W0, b0.contiguous() if b0 is not None else None, act, float(slope))
        P1 = stack.split_planes(y1, float(p), seed)
        y2 = stack.planes_linear(P1, W3, b3.contiguous() if b3 is not None else None, act, float(slope))
        if tracing():
            if p > 0.0:
                trace("drop", (stack.split_planes(torch.ones_like(y1), float(p), seed).float() > 0).float() * (1.0 / (1.0 - p)))
            trace("sign", y1 > 0)
            trace("sign", y2 > 0)
        ctx.planes = (P0, P1)
        ctx.save_for_backward(W0, W3, y1, y2)
        ctx.cfg = (act, float(slope), float(p), seed, b0 is not None, b3 is not None)
        return y2

    @staticmethod
    def backward(ctx, g):
        from . import stack
        W0, W3, y1, y2 = ctx.saved_tensors
        act, slope, p, seed, has_b0, has_b3 = ctx.cfg
        P0, P1 = ctx.planes
        ctx.planes = None
        L = lib()
        dev = g.device
        M = y1.shape[0]
        need = ctx.needs_input_grad

        def glue(gr, y, drop_p, drop_seed, want_db):
            """planes of mask(gr) * act'(y) and (optionally) their column sums"""
            gr = stack._grad_rows(gr)
            n = y.shape[1]
            gp = stack.Planes(M, n, dev)
            db = torch.empty(n, dtype=torch.float32, device=dev) if want_db else None
            ws = _ws(L.act_bwd_planes_ws(n), dev) if want_db else None
            L.act_bwd_planes(ptr(gr), gr.stride(0), ptr(y) if act else None, y.stride(0) if act else 0, act, slope,
                             drop_p, drop_seed, gp.ptr(), gp.ld, gp.ps, M, n, ptr(db), ptr(ws), stream(),
                             _key=("bytes", (12.0 if act else 8.0) * M * n))
            return gp, db

        gp2, db3 = glue(g, y2, 0.0, 0, has_b3 and need[4])
        dW3 = stack.planes_linear_bwd_weight(gp2, P1) if need[3] else None
        dy1 = stack.planes_linear_bwd_input(gp2, W3, W3.shape[1])          # gradient of the DROPPED hidden tensor
        del gp2
        gp1, db0 = glue(dy1, y1, p, seed, has_b0 and need[2])
        dW0 = stack.planes_linear_bwd_weight(gp1, P0) if need[1] else None
        dx = stack.planes_linear_bwd_input(gp1, W0, W0.shape[1]) if need[0] else None
        return dx, dW0, db0, dW3, db3, None, None, None, None


def mlp_drop(x, W0, b0, W3, b3, act="leaky_relu", slope=0.01, p=0.0):
    return MlpDropFn.apply(x, W0, b0, W3, b3, act_code(act), slope, float(p), next_seed() if p > 0.0 else 0)


def linear(x1, W, bias=None, act=None, slope=0.0, x2=None):
    code = act_code(act)
    out = PlanesLinearFn.apply(x1, x2, W, bias, code, slope)
    if tracing() and code in (ACT["relu"], ACT["leaky_relu"]):
        trace("sign", out > 0)          # the activation is fused; sign(out) == sign(pre-activation)
    return out


class ConcatDropoutFn(Function):
    """out = dropout(cat([x1, x2], 1), p) with a hash mask regenerated in backward (GATConv feat_drop)."""

    @staticmethod
    def forward(ctx, x1, x2, p, seed):
        require_cuda(x1, x2)
        x1 = _rows(x1)
        x2 = _rows(x2) if x2 is not None else None
        M, K1 = x1.shape
        K2 = x2.shape[1] if x2 is not None else 0
        out = empty_padded(M, K1 + K2, x1.device)
        lib().concat_dropout(ptr(x1), x1.stride(0), K1, ptr(x2), x2.stride(0) if x2 is not None else 0, K2, float(p),
                             seed, ptr(out), out.stride(0), M, stream())
        ctx.cfg = (K1, K2, float(p), seed)
        return out

    @staticmethod
    def backward(ctx, g):
        K1, K2, p, seed = ctx.cfg
        g = _rows(g)
        M = g.shape[0]
        d1 = empty_padded(M, K1, g.device) if ctx.needs_input_grad[0] else None
        d2 = empty_padded(M, K2, g.device) if (K2 and ctx.needs_input_grad[1]) else None
        lib().concat_dropout_bwd(ptr(g), g.stride(0), K1, K2, p, seed, ptr(d1), d1.stride(0) if d1 is not None else 0,
                                 ptr(d2), d2.stride(0) if d2 is not None else 0, M, stream())
        return d1, d2, None, None


def concat_dropout(x1, x2, p, training):
    p = float(p) if training else 0.0
    if p == 0.0 and x2 is None:
        return x1
    seed = next_seed()
    if tracing() and p > 0.0:
        trace("drop", drop_mask(x1.shape[0], x1.shape[1] + (x2.shape[1] if x2 is not None else 0), p, seed, x1.device))
    return ConcatDropoutFn.apply(x1, x2, p, seed)


class BiasActFn(Function):
    @staticmethod
    def forward(ctx, x, bias, act, slope):
        require_cuda(x, bias)
        x = _rows(x)
        M, N = x.shape
        y = empty_padded(M, N, x.device)
        lib().bias_act(ptr(x), x.stride(0), ptr(bias), act, float(slope), ptr(y), y.stride(0), M, N, stream())
        ctx.save_for_backward(y)
        ctx.cfg = (act, float(slope), bias is not None)
        return y

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        act, slope, has_bias = ctx.cfg
        g = _rows(g)
        M, N = g.shape
        d = empty_padded(M, N, g.device)
        lib().act_bwd(ptr(g), g.stride(0), ptr(y), y.stride(0), act, slope, ptr(d), d.stride(0), M, N, stream())
        return d, (colsum(d) if has_bias and ctx.needs_input_grad[1] else None), None, None


def bias_act(x, bias=None, act=None, slope=0.0):
    return BiasActFn.apply(x, bias, act_code(act), slope)


class PackWeightFn(Function):
    """[W_fc ; W_res ; W_fc^T·attn_l ; W_fc^T·attn_r] of a GATConv in one kernel each way (include/spgnn_b200.h,
    spgnn_gat_pack_weight).  Returns [rows, K] with 16-byte aligned rows."""

    @staticmethod
    def forward(ctx, w_fc, w_res, attn_l, attn_r, H, F):
        require_cuda(w_fc, w_res, attn_l, attn_r)
        w_fc = _rows(w_fc)
        w_res = _rows(w_res) if w_res is not None else None
        al, ar = attn_l.contiguous(), attn_r.contiguous()
        K = w_fc.shape[1]
        rows = H * F * (2 if w_res is not None else 1) + 2 * H
        out = torch.empty(rows, _pad4(K), dtype=torch.float32, device=w_fc.device)
        lib().gat_pack_weight(ptr(w_fc), w_fc.stride(0), ptr(w_res), w_res.stride(0) if w_res is not None else 0,
                              ptr(al), ptr(ar), H, F, K, ptr(out), out.stride(0), stream())
        ctx.save_for_backward(w_fc, al, ar)
        ctx.cfg = (H, F, K, w_res is not None)
        return out[:, :K]

    @staticmethod
    def backward(ctx, g):
        w_fc, al, ar = ctx.saved_tensors
        H, F, K, has_res = ctx.cfg
        g = _rows(g)
        need = ctx.needs_input_grad
        dev = g.device
        dW = torch.empty(H * F, K, dtype=torch.float32, device=dev) if need[0] else None
        dR = torch.empty(H * F, K, dtype=torch.float32, device=dev) if (has_res and need[1]) else None
        dal = torch.empty(al.shape, dtype=torch.float32, device=dev) if need[2] else None
        dar = torch.empty(ar.shape, dtype=torch.float32, device=dev) if need[3] else None
        lib().gat_pack_weight_bwd(ptr(g), g.stride(0), ptr(w_fc), w_fc.stride(0), ptr(al), ptr(ar), H, F, K,
                                  int(has_res), ptr(dW), K, ptr(dR), K, ptr(dal), ptr(dar), stream())
        return dW, dR, dal, dar, None, None


class GatAggFn(Function):
    """Fused edge-softmax + aggregation + residual + bias + activation (+ head mean) over the projection output Y."""

    @staticmethod
    def forward(ctx, Y, xres, bias, graph, H, F, res_mode, act, neg_slope, mean_heads, drop_p, seed):
        require_cuda(Y, xres, bias)
        Y = _rows(Y)
        N = Y.shape[0]
        HF = H * F
        res_off = HF
        el_off = 2 * HF if res_mode == 1 else HF
        er_off = el_off + H
        if Y.shape[1] != er_off + H:
            raise SpgnnError(f"gat_agg: projection has {Y.shape[1]} columns, expected {er_off + H}")
        xr = _rows(xres) if res_mode == 2 else None
        out = empty_padded(N, F if mean_heads else HF, Y.device)
        att = torch.empty(graph.num_edges, H, dtype=torch.float32, device=Y.device)
        b = bias.contiguous() if bias is not None else None
        lib().gat_agg_fwd(ptr(Y), Y.stride(0), res_off, el_off, er_off, res_mode, ptr(xr),
                          xr.stride(0) if xr is not None else 0, xr.shape[1] if xr is not None else 0, ptr(b), act,
                          float(neg_slope), int(mean_heads), float(drop_p), seed, ptr(graph.in_ptr), ptr(graph.in_src),
                          N, H, F, ptr(out), out.stride(0), ptr(att), stream(),
                          _key=("bytes", 4.0 * N * (HF + (HF if res_mode == 1 else 0) + 2 * H + (F if mean_heads else HF))
                                + 4.0 * (N + 1) + 4.0 * graph.num_edges))
        if tracing():
            trace_gat(graph, Y[:, el_off:el_off + H], Y[:, er_off:er_off + H], float(drop_p), seed)
        ctx.save_for_backward(Y, xr, b, out if not mean_heads else None, att)
        ctx.graph = graph
        ctx.cfg = (H, F, res_mode, act, float(neg_slope), int(mean_heads), float(drop_p), seed, res_off, el_off, er_off)
        return out

    @staticmethod
    def backward(ctx, g):
        Y, xr, b, out, att = ctx.saved_tensors
        H, F, res_mode, act, neg_slope, mean_heads, drop_p, seed, res_off, el_off, er_off = ctx.cfg
        gr = ctx.graph
        g = _rows(g)
        N, HF = Y.shape[0], H * F
        dY = torch.empty(N, Y.stride(0), dtype=torch.float32, device=Y.device)[:, :Y.shape[1]]
        g_ws = torch.empty(N, HF, dtype=torch.float32, device=Y.device) if res_mode != 1 else None
        dxres = torch.empty(N, xr.stride(0), dtype=torch.float32, device=Y.device)[:, :xr.shape[1]] \
            if res_mode == 2 else None
        ds = torch.empty(gr.num_edges * H, dtype=torch.float32, device=Y.device)
        lib().gat_agg_bwd(ptr(g), g.stride(0), ptr(out), out.stride(0) if out is not None else 0, ptr(Y), Y.stride(0),
                          res_off, el_off, er_off, res_mode, ptr(xr), xr.stride(0) if xr is not None else 0,
                          xr.shape[1] if xr is not None else 0, ptr(b), act, neg_slope, mean_heads, drop_p, seed,
                          ptr(att), ptr(gr.in_ptr), ptr(gr.in_src), ptr(gr.out_ptr), ptr(gr.out_dst), ptr(gr.out_slot),
                          N, H, F, ptr(dY), ptr(dxres), ptr(g_ws), ptr(ds), stream(),
                          _key=("bytes", 4.0 * N * ((F if mean_heads else 2 * HF) + 2 * (Y.shape[1]))
                                + 8.0 * (N + 1) + 12.0 * gr.num_edges))
        db = None
        if b is not None and ctx.needs_input_grad[2]:
            db = colsum(dY[:, res_off:res_off + HF] if res_mode == 1 else g_ws)
        return dY, dxres, db, None, None, None, None, None, None, None, None, None


class SpmmFn(Function):
    """out = act(post ⊙ (Σ_{u→v} pre[u]·x[u] + [self_in] pre[v]·x[v]) + (1+eps)·x[v]·[eps given] + add[v] + bias)
    — GraphConv / GINConv-mean / SAGEConv mean and gcn.  ``graph`` is a batched Graph (output rows = nodes) or a
    sampled ``sampling.Block`` (rows of ``x`` = source nodes, output rows = destination nodes; the self terms read
    x[v] for the destinations, which are the first source rows)."""

    @staticmethod
    def forward(ctx, x, eps, bias, graph, pre, post, act, slope, add=None, self_in=False):
        require_cuda(x, eps, bias, add)
        x = _rows(x)
        n_src, F = x.shape
        N = _n_dst(graph)
        out = empty_padded(N, F, x.device)
        b = bias.contiguous() if bias is not None else None
        a = _rows(add) if add is not None else None
        lib().spmm(ptr(x), x.stride(0), ptr(graph.in_ptr), ptr(graph.in_src), ptr(pre), ptr(post), ptr(eps),
                   int(self_in), N, ptr(a), a.stride(0) if a is not None else 0, ptr(b), act, float(slope), ptr(out),
                   out.stride(0), N, F, stream(),
                   _key=("bytes", 4.0 * (n_src + N * (2 if a is not None else 1)) * F + 4.0 * (N + 1) + 4.0 * graph.num_edges))
        ctx.save_for_backward(x if eps is not None else None, eps, out if act else None)
        ctx.graph, ctx.pre, ctx.post = graph, pre, post
        ctx.cfg = (act, float(slope), b is not None, bool(self_in), n_src)
        return out

    @staticmethod
    def backward(ctx, g):
        x, eps, out = ctx.saved_tensors
        act, slope, has_bias, self_in, n_src = ctx.cfg
        gr = ctx.graph
        L = lib()
        g = _rows(g)
        N, F = g.shape
        if act:
            d = empty_padded(N, F, g.device)
            L.act_bwd(ptr(g), g.stride(0), ptr(out), out.stride(0), act, slope, ptr(d), d.stride(0), N, F, stream())
            g = d
        dx = deps = db = None
        if ctx.needs_input_grad[0]:
            dx = empty_padded(n_src, F, g.device)
            # transpose graph: out-edges into the source rows, with the roles of the two norms swapped; the self terms
            # exist for the first N (destination) rows only
            L.spmm(ptr(g), g.stride(0), ptr(gr.out_ptr), ptr(gr.out_dst), ptr(ctx.post), ptr(ctx.pre), ptr(eps),
                   int(self_in), N, None, 0, None, 0, 0.0, ptr(dx), dx.stride(0), n_src, F, stream(),
                   _key=("bytes", 4.0 * (n_src + N) * F + 4.0 * (n_src + 1) + 4.0 * gr.num_edges))
        if eps is not None and ctx.needs_input_grad[1]:
            deps = (g * x[:N]).sum().reshape(1)
        if has_bias and ctx.needs_input_grad[2]:
            db = colsum(g)
        need = ctx.needs_input_grad
        dadd = g if len(need) > 8 and need[8] else None
        return (dx, deps, db, None, None, None, None, None, dadd, None)[:len(need)]


def _n_dst(graph):
    return int(graph.num_dst_nodes) if getattr(graph, "is_block", False) else int(graph.num_nodes)


def inv_degree(graph, add):
    """1 / max(in_degree + add, 1) per destination node (SAGEConv mean: add 0, gcn: add 1), cached on the graph."""
    cache = graph.__dict__.setdefault("_inv_degree", {})
    hit = cache.get(add)
    if hit is None:
        n = _n_dst(graph)
        hit = torch.empty(n, dtype=torch.float32, device=graph.in_ptr.device)
        lib().inv_degree(ptr(graph.in_ptr), n, float(add), ptr(hit), stream())
        cache[add] = hit
    return hit


class LstmOrder:
    """Destinations sorted by in-degree, descending and stable (a device counting sort): ``perm[row]`` = destination,
    ``rank[destination]`` = row; ``steps[t]`` = n_t = destinations with in-degree > t, so LSTM step t runs over rows
    [0, n_t); ``off[t]`` = Σ_{s<t} n_s is where step t's rows start in the per-step buffers (int64, host and device).
    Built once per graph (two small device→host reads) and cached on it, like ``Graph.norms()``."""

    def __init__(self, graph):
        L = lib()
        dev = graph.in_ptr.device
        n = _n_dst(graph)
        self.n = n
        deg = graph.in_ptr[1:n + 1] - graph.in_ptr[:n]
        max_deg = int(deg.max().item()) if n > 0 else 0
        chunks = (n + 255) // 256
        counts = torch.empty((max_deg + 1) * chunks, dtype=torch.int64, device=dev)
        L.lstm_order_count(ptr(graph.in_ptr), n, max_deg, ptr(counts), stream())
        from .graph import device_scan
        offs = device_scan(counts)
        self.perm = torch.empty(n, dtype=torch.int32, device=dev)
        self.rank = torch.empty(n, dtype=torch.int32, device=dev)
        L.lstm_order_scatter(ptr(graph.in_ptr), n, max_deg, ptr(offs), ptr(self.perm), ptr(self.rank), stream())
        # bucket of degree d starts at offs[(max_deg - d) * chunks]: the rows before it have degree > d
        self.steps = offs[torch.arange(max_deg, 0, -1, device=dev) * chunks].tolist()     # d = 0 .. max_deg - 1
        self.off = [0]
        for k in self.steps:
            self.off.append(self.off[-1] + k)
        self.off_dev = torch.tensor(self.off, dtype=torch.int64, device=dev)


def lstm_order(graph):
    o = graph.__dict__.get("_lstm_order")
    if o is None:
        o = graph.__dict__["_lstm_order"] = LstmOrder(graph)
    return o


class LstmReduceFn(Function):
    """neigh[v] = h_T(v) of DGL 0.7's ``_lstm_reducer``: an LSTM (zero initial state, gates i, f, g, o) over the
    messages of v's in-edges in in-CSC order.  ``P`` = X·W_ihᵀ + b_ih + b_hh [n_src, 4D] is the input projection
    (``linear``: autograd takes its gradients), ``W_hh`` [4D, D].  Returns [n_dst, D]; zero for in-degree 0.

    Step t runs over the first n_t rows of ``LstmOrder`` (destinations by descending in-degree); step 0 needs no
    GEMM (h_0 = 0), step t ≥ 1 adds R_t = H_{t-1}[:n_t]·W_hhᵀ from the planes GEMMs.
    Per-step buffers hold step t at rows [off_t, off_t + n_t): the gate activations (as the 16-bit halves of the
    planes the backward overwrites with the gate gradients), c, and h as planes at the rows of the step that reads
    it, so dW_hh is ONE GEMM over all steps."""

    @staticmethod
    def forward(ctx, P, W_hh, graph):
        from . import stack
        require_cuda(P, W_hh)
        P, W = _rows(P), _rows(W_hh)
        D = W.shape[1]
        if W.shape[0] != 4 * D or P.shape[1] != 4 * D:
            raise SpgnnError(f"lstm reducer: W_hh {tuple(W.shape)} and P {tuple(P.shape)} do not match an LSTM")
        if D % 4:
            raise SpgnnError(f"lstm reducer: the feature width must be a multiple of 4, got {D}")
        if P.stride(0) % 4 or P.data_ptr() % 16:
            P = empty_padded(P.shape[0], 4 * D, P.device).copy_(P)
        o = lstm_order(graph)
        dev = P.device
        out = torch.zeros(o.n, _pad4(D), dtype=torch.float32, device=dev)[:, :D]
        ctx.graph, ctx.order, ctx.n_src, ctx.rec = graph, o, P.shape[0], None
        ctx.save_for_backward(W)
        T = len(o.steps)
        if T == 0:
            return out
        E, n0 = o.off[-1], o.steps[0]
        G = stack.Planes(E, 4 * D, dev)
        C = torch.empty(E, D, dtype=torch.float32, device=dev)
        Hn = stack.Planes(E - n0, D, dev) if T > 1 else None
        R = torch.empty(o.steps[1], 4 * D, dtype=torch.float32, device=dev) if T > 1 else None
        L = lib()
        for t in range(T):
            n_t, n_next = o.steps[t], (o.steps[t + 1] if t + 1 < T else 0)
            Rt = None
            if t > 0:
                Rt = stack.planes_linear(stack.PlanesView(Hn, 0, D, o.off[t] - n0, n_t), W, out=R[:n_t])
            hn = Hn.ptr() + 2 * (o.off[t + 1] - n0) * Hn.ld if n_next else None
            L.lstm_cell_fwd(t, n_t, n_next, ptr(o.perm), ptr(graph.in_ptr), ptr(graph.in_src), ptr(P), P.stride(0),
                            ptr(Rt), R.stride(0) if Rt is not None else 0, G.ptr() + 2 * o.off[t] * G.ld, G.ld, G.ps,
                            ptr(C[o.off[t - 1]:]) if t > 0 else None, ptr(C[o.off[t]:]), hn,
                            Hn.ld if Hn is not None else 0, Hn.ps if Hn is not None else 0, ptr(out), out.stride(0), D,
                            stream(), _name="lstm_cell_fwd",
                            _key=("bytes", n_t * (40.0 * D + (20.0 * D if t > 0 else 0.0) + 12.0)))
        ctx.rec = (G, C, Hn)
        return out

    @staticmethod
    def backward(ctx, g):
        from . import stack
        (W,) = ctx.saved_tensors
        o, graph, n_src = ctx.order, ctx.graph, ctx.n_src
        D = W.shape[1]
        dev = W.device
        dP = empty_padded(n_src, 4 * D, dev)
        T = len(o.steps)
        if T == 0:
            return dP.zero_(), torch.zeros_like(W), None
        G, C, Hn = ctx.rec
        ctx.rec = None
        g = _rows(g)
        if g.stride(0) % 4 or g.data_ptr() % 16:
            g = empty_padded(g.shape[0], D, dev).copy_(g)
        E, n0 = o.off[-1], o.steps[0]
        dH = torch.empty(o.steps[1], D, dtype=torch.float32, device=dev) if T > 1 else None
        dc = torch.empty(o.steps[1], D, dtype=torch.float32, device=dev) if T > 1 else None
        L = lib()
        for t in reversed(range(T)):
            n_t, n_next = o.steps[t], (o.steps[t + 1] if t + 1 < T else 0)
            L.lstm_cell_bwd(t, n_t, n_next, ptr(o.perm), ptr(g), g.stride(0), ptr(dH) if n_next else None, D,
                            ptr(dc) if (t > 0 or n_next) else None, G.ptr() + 2 * o.off[t] * G.ld, G.ld, G.ps,
                            ptr(C[o.off[t - 1]:]) if t > 0 else None, ptr(C[o.off[t]:]), D, stream(),
                            _name="lstm_cell_bwd",
                            _key=("bytes", n_t * (40.0 * D + (8.0 * D if t > 0 else 0.0) + (4.0 * D if n_next else 0.0))))
            if t > 0:
                stack.planes_linear_bwd_input(stack.PlanesView(G, 0, 4 * D, o.off[t], n_t), W, D, out=dH[:n_t])
        dW = (stack.planes_linear_bwd_weight(stack.PlanesView(G, 0, 4 * D, n0, E - n0), Hn) if T > 1
              else torch.zeros_like(W))
        L.lstm_dp(G.ptr(), G.ld, G.ps, ptr(o.off_dev), ptr(o.rank), ptr(graph.in_ptr), ptr(graph.out_ptr),
                  ptr(graph.out_dst), ptr(graph.out_slot), ptr(dP), dP.stride(0), n_src, D, stream(),
                  _key=("bytes", 16.0 * D * (E + n_src) + 16.0 * E))
        return dP, dW, None


class MaxPoolFn(Function):
    """neigh[v] = max over in-neighbours (SAGEConv 'pool'), arg-slot saved for the backward scatter.  ``graph`` is a
    batched Graph (square: rows of ``m`` = nodes) or a sampled ``sampling.Block`` (rows of ``m`` = source nodes,
    output rows = destination nodes)."""

    @staticmethod
    def forward(ctx, m, graph):
        require_cuda(m)
        m = _rows(m)
        n_src, F = m.shape
        n_dst = int(getattr(graph, "num_dst_nodes", n_src))
        out = empty_padded(n_dst, F, m.device)
        arg = torch.empty(n_dst, F, dtype=torch.int32, device=m.device)
        lib().sage_maxpool_fwd(ptr(m), m.stride(0), ptr(graph.in_ptr), ptr(graph.in_src), ptr(out), out.stride(0),
                               ptr(arg), n_dst, F, stream(),
                               _key=("bytes", 4.0 * F * (n_src + 2 * n_dst) + 4.0 * (n_dst + 1) + 4.0 * graph.num_edges))
        if tracing():
            trace("argmax", torch.where(arg >= 0, graph.in_src.long()[arg.clamp(min=0).long()], arg.long()))
        ctx.save_for_backward(arg)
        ctx.graph, ctx.n_src = graph, n_src
        return out

    @staticmethod
    def backward(ctx, g):
        (arg,) = ctx.saved_tensors
        gr = ctx.graph
        g = _rows(g)
        n_dst, F = g.shape
        dm = empty_padded(ctx.n_src, F, g.device)
        lib().sage_maxpool_bwd(ptr(g), g.stride(0), ptr(arg), ptr(gr.out_ptr), ptr(gr.out_dst), ptr(gr.out_slot),
                               ptr(dm), dm.stride(0), ctx.n_src, F, stream(),
                               _key=("bytes", 4.0 * F * (ctx.n_src + 2 * n_dst) + 8.0 * (ctx.n_src + 1) + 8.0 * gr.num_edges))
        return dm, None


class MaskedCEFn(Function):
    """F.cross_entropy(logits[mask], y[mask], weight) with the node mask either given or drawn on device
    (keep = y != 0 or u < rate), job_runner.py:1885-1900.  ``extra`` (sum of class weights from other ranks) lets
    data-parallel training normalise by the global Σw."""

    @staticmethod
    def forward(ctx, logits, y, mask, rate, seed, class_w, reduce_fn):
        require_cuda(logits, y, mask, class_w)
        logits = _rows(logits)
        N, C = logits.shape
        sums = torch.empty(2, dtype=torch.float64, device=logits.device)
        m = mask.to(torch.uint8).contiguous() if mask is not None else None
        lib().masked_ce_fwd(ptr(logits), logits.stride(0), C, ptr(y), ptr(m), float(rate), seed, ptr(class_w), N,
                            ptr(sums), stream())
        if reduce_fn is not None:
            sums = reduce_fn(sums)          # all-reduce (Σ w·nll, Σ w) across ranks
        ctx.save_for_backward(logits, y, m, class_w, sums)
        ctx.cfg = (float(rate), seed)
        return (sums[0] / sums[1]).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        logits, y, m, class_w, sums = ctx.saved_tensors
        rate, seed = ctx.cfg
        N, C = logits.shape
        d = empty_padded(N, C, logits.device)
        lib().masked_ce_bwd(ptr(logits), logits.stride(0), C, ptr(y), ptr(m), rate, seed, ptr(class_w), ptr(sums),
                            1.0, N, ptr(d), d.stride(0), stream())
        return d * g, None, None, None, None, None, None


def masked_cross_entropy(logits, y, class_w, mask=None, rate=1.0, seed=None, reduce_fn=None):
    return MaskedCEFn.apply(logits, y, mask, rate, next_seed() if seed is None else seed, class_w, reduce_fn)


def segmented_argmax(logits, graph):
    """job_runner.py:158-165: per tree and class 1..C-1 the node (global id) with the highest softmax probability."""
    require_cuda(logits)
    logits = _rows(logits)
    C = logits.shape[1]
    out = torch.empty(graph.batch_size, C - 1, dtype=torch.int64, device=logits.device)
    lib().segmented_argmax(ptr(logits), logits.stride(0), C, ptr(graph.node_off), graph.batch_size, ptr(out), stream())
    return out
