"""Planes pipeline for whole GAT stacks (GAT, GATPSPGNN, GATPSPGNNNL of /root/reference/models.py:283-540).

One autograd.Function runs a whole stack with an explicit tape instead of one Function per op:

  * every activation lives in HBM as split-bf16 *planes* (x = hi + lo, see include/spgnn_b200.h), written by the
    kernel that produces it — the layer kernel's epilogue, or ``spgnn_split_planes`` for the raw inputs — already
    carrying the feat_drop mask of the GATConv that will consume it; ``torch.cat([h_s, h_p])`` is two TMA sources;
  * the projections are TMA-fed tcgen05 GEMMs (``spgnn_planes_linear_*``), fp32 output Y = [z | res | el | er];
  * the backward of a layer reads the masked ``dX`` of its consumers directly (no gradient accumulation pass, no
    dropout-backward pass), writes ``dY`` as planes for the dX / dW projections and emits the bias gradient.

Semantics are those of ``nn.GATConv`` (DGL 0.7.x, SURVEY.md §8a A1) — the per-layer path in ``nn.py``/``ops.py``
stays as the general fallback (identity residuals, exotic shapes, inputs that need gradients).
PyTorch is plumbing here: memory, streams, the autograd hook-up of the parameters.
"""
from __future__ import annotations

import ctypes

import torch
from torch.autograd import Function

from . import ops
from ._lib import SpgnnError, lib, ptr, stream


class _Sink(ctypes.Structure):
    _fields_ = [("hi", ctypes.c_void_p), ("ld", ctypes.c_int64), ("plane_stride", ctypes.c_int64),
                ("concat_chunks", ctypes.c_int64), ("chunk_off", ctypes.c_int64),
                ("drop_p", ctypes.c_float), ("reserved", ctypes.c_uint32), ("seed", ctypes.c_uint64)]


class _GSrc(ctypes.Structure):
    _fields_ = [("g", ctypes.c_void_p), ("ld", ctypes.c_int64), ("concat_chunks", ctypes.c_int64),
                ("chunk_off", ctypes.c_int64), ("drop_p", ctypes.c_float), ("reserved", ctypes.c_uint32),
                ("seed", ctypes.c_uint64)]


class _Layer(ctypes.Structure):
    _fields_ = [("in_ptr", ctypes.c_void_p), ("in_src", ctypes.c_void_p), ("out_ptr", ctypes.c_void_p),
                ("out_dst", ctypes.c_void_p), ("out_slot", ctypes.c_void_p),
                ("N", ctypes.c_int64), ("H", ctypes.c_int32), ("F", ctypes.c_int32),
                ("Y", ctypes.c_void_p), ("ldy", ctypes.c_int64), ("res_off", ctypes.c_int64),
                ("el_off", ctypes.c_int64), ("er_off", ctypes.c_int64),
                ("res_mode", ctypes.c_int32), ("act", ctypes.c_int32), ("negative_slope", ctypes.c_float),
                ("mean_heads", ctypes.c_int32),
                ("bias", ctypes.c_void_p), ("attn_drop_p", ctypes.c_float), ("reserved0", ctypes.c_uint32),
                ("attn_seed", ctypes.c_uint64),
                ("att", ctypes.c_void_p),
                ("out", ctypes.c_void_p), ("ldo", ctypes.c_int64), ("n_sinks", ctypes.c_int32),
                ("reserved1", ctypes.c_int32), ("sinks", _Sink * 2),
                ("n_gsrc", ctypes.c_int32), ("reserved2", ctypes.c_int32), ("gsrc", _GSrc * 3),
                ("dY_hi", ctypes.c_void_p), ("dY_ld", ctypes.c_int64), ("dY_ps", ctypes.c_int64),
                ("g_ws", ctypes.c_void_p), ("ds_ws", ctypes.c_void_p), ("dbias", ctypes.c_void_p),
                ("dbias_ws", ctypes.c_void_p),
                ("node_off", ctypes.c_void_p), ("B", ctypes.c_int64), ("max_nodes", ctypes.c_int64),
                ("max_degree", ctypes.c_int64)]


class _Wide(ctypes.Structure):
    _fields_ = [("in_ptr", ctypes.c_void_p), ("in_src", ctypes.c_void_p), ("out_ptr", ctypes.c_void_p),
                ("out_dst", ctypes.c_void_p), ("out_slot", ctypes.c_void_p),
                ("N", ctypes.c_int64), ("H", ctypes.c_int32), ("has_res", ctypes.c_int32),
                ("X1", ctypes.c_void_p), ("ldx1", ctypes.c_int64), ("psx1", ctypes.c_int64),
                ("X2", ctypes.c_void_p), ("ldx2", ctypes.c_int64), ("psx2", ctypes.c_int64),
                ("K1", ctypes.c_int32), ("K2", ctypes.c_int32),
                ("eler", ctypes.c_void_p), ("ld_eler", ctypes.c_int64),
                ("negative_slope", ctypes.c_float), ("attn_drop_p", ctypes.c_float), ("attn_seed", ctypes.c_uint64),
                ("att", ctypes.c_void_p),
                ("XA", ctypes.c_void_p), ("ldxa", ctypes.c_int64), ("psxa", ctypes.c_int64), ("kp", ctypes.c_int64),
                ("dXA", ctypes.c_void_p), ("ld_dxa", ctypes.c_int64), ("head_stride", ctypes.c_int64),
                ("w_eler", ctypes.c_void_p), ("ld_w", ctypes.c_int64),
                ("ds_ws", ctypes.c_void_p),
                ("d_eler", ctypes.c_void_p), ("ld_de", ctypes.c_int64),
                ("d_eler_planes", ctypes.c_void_p), ("ld_dep", ctypes.c_int64), ("ps_dep", ctypes.c_int64),
                ("dX", ctypes.c_void_p), ("ld_dx", ctypes.c_int64)]


# Aggregate-first evaluation of head-averaged output layers (include/spgnn_b200.h, spgnn_gat_wide).  Switch off to
# run every layer through the projection-first kernels (tests compare the two).
WIDE_OUTPUT_LAYER = True
# Training an aggregate-first output layer that feeds the head (train mode, tape kept): the forward keeps act'(pre) of
# every head and the backward builds the pre-activation gradient from the head's output gradient in one memory-bound
# pass (spgnn_wide_dpre) instead of the head's dX GEMM plus a recompute of the wide GEMM (spgnn_wide_linear mode 1).
# Costs H*F*4 bytes per node from the forward to the backward.  Off: mode 1 (tests compare the two).
WIDE_SAVED_DACT = True
# One CTA per graph with the graph's rows staged in shared memory (spgnn_gat_layer.node_off).  Off: chunk kernels.
TREE_KERNELS = True

_checked = False


def _check_abi():
    global _checked
    if not _checked:
        n = int(lib().gat_layer_sizeof())
        if n != ctypes.sizeof(_Layer):
            raise SpgnnError(f"spgnn_gat_layer layout mismatch: library {n} bytes, binding {ctypes.sizeof(_Layer)}")
        n = int(lib().gat_wide_sizeof())
        if n != ctypes.sizeof(_Wide):
            raise SpgnnError(f"spgnn_gat_wide layout mismatch: library {n} bytes, binding {ctypes.sizeof(_Wide)}")
        _checked = True


class Planes:
    """[rows, cols] fp32-valued matrix as two bf16 planes (buf[0] = hi, buf[1] = lo), rows padded to 64 columns."""

    __slots__ = ("buf", "rows", "cols", "ld")

    def __init__(self, rows, cols, device):
        self.rows, self.cols = int(rows), int(cols)
        self.ld = (self.cols + 63) // 64 * 64
        self.buf = torch.empty(2, self.rows, self.ld, dtype=torch.bfloat16, device=device)

    @property
    def ps(self):
        return self.rows * self.ld

    def ptr(self, col=0):
        return self.buf.data_ptr() + 2 * col

    def float(self):
        return (self.buf[0].float() + self.buf[1].float())[:, :self.cols]


class PlanesView:
    """Columns [col0, col0 + cols) and rows [row0, row0 + rows) of a Planes (same ld and plane stride)."""

    __slots__ = ("buf", "rows", "cols", "ld", "ps", "_p")

    def __init__(self, base, col0, cols, row0=0, rows=None):
        self.buf, self.cols, self.ld, self.ps = base.buf, int(cols), base.ld, base.ps
        self.rows = base.rows - int(row0) if rows is None else int(rows)
        self._p = base.ptr(int(col0)) + 2 * int(row0) * base.ld

    def ptr(self, col=0):
        return self._p + 2 * col


def split_planes(x, p=0.0, seed=0, concat_chunks=0, chunk_off=0, x2=None):
    """fp32 [M, K] (optionally [x | x2]) → Planes, with the consumer's feat_drop applied when p > 0."""
    x = ops._rows(x)
    M, K1 = x.shape
    K2 = 0
    if x2 is not None:
        x2 = ops._rows(x2)
        K2 = x2.shape[1]
    out = Planes(M, K1 + K2, x.device)
    lib().split_planes(ptr(x), x.stride(0), K1, ptr(x2), x2.stride(0) if x2 is not None else 0, K2, float(p), seed,
                       int(concat_chunks), int(chunk_off), out.ptr(), out.ld, out.ps, M, stream(),
                       _key=("bytes", 8.0 * M * (K1 + K2)))
    return out


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def planes_linear(A1: Planes, W, bias=None, act=0, slope=0.0, A2: Planes | None = None, out=None):
    """fp32 [M, N] = [A1 | A2] @ W^T (+bias)(act); W fp32 [N, K1+K2] with unit inner stride.  ``out``: an [M, N]
    destination with 16-byte aligned rows (a buffer reused across calls)."""
    if ops.GEMM_MODE != 2:
        raise SpgnnError(f"ops.GEMM_MODE = {ops.GEMM_MODE!r}: the planes GEMMs (2) are the only projection path")
    W = ops._rows(W)
    M, N = A1.rows, W.shape[0]
    K1, K2 = A1.cols, (A2.cols if A2 is not None else 0)
    if W.shape[1] != K1 + K2:
        raise SpgnnError(f"planes_linear: weight has {W.shape[1]} columns, input has {K1}+{K2}")
    # rows padded to 128 bytes once they are wide enough to be sliced by the per-tree layer kernels (TMA boxes of 32
    # columns then start on cache-line boundaries)
    if out is not None:
        C = out
    else:
        C = ops.empty_padded(M, N, W.device) if N < 64 else torch.empty(
            M, (N + 31) // 32 * 32, dtype=torch.float32, device=W.device)[:, :N]
    L = lib()
    ws = _ws(L.planes_linear_fwd_ws(N, K1, K2), W.device)
    L.planes_linear_fwd(A1.ptr(), A1.ld, A1.ps, K1, A2.ptr() if A2 is not None else None,
                        A2.ld if A2 is not None else 0, A2.ps if A2 is not None else 0, K2, ptr(W), W.stride(0),
                        ptr(bias), act, float(slope), ptr(C), C.stride(0), M, N, ptr(ws), ws.numel(), stream(),
                        _key=("flops", 2.0 * M * N * (K1 + K2)))
    return C


def planes_linear_bwd_input(dC: Planes, W, K, k_off=0, out=None, drop_p=0.0, seed=0, concat_chunks=0):
    """fp32 [M, K] = dC @ W[:, k_off:k_off+K]; ``drop_p`` > 0: times the feat_drop mask (and 1 / (1 - p)) of the layer
    whose dropped input this is the gradient of — the mask every plane producer derives from (seed, row, column
    chunk), applied here in the GEMM epilogue so the producing layer's backward reads a finished gradient."""
    W = ops._rows(W)
    M, N = dC.rows, dC.cols
    dA = ops.empty_padded(M, K, W.device) if out is None else out
    L = lib()
    ws = _ws(L.planes_linear_bwd_input_ws(N, K), W.device)
    if drop_p > 0.0:
        L.planes_linear_bwd_input_masked(dC.ptr(), dC.ld, dC.ps, ptr(W), W.stride(0), k_off, ptr(dA), dA.stride(0), M,
                                         N, K, float(drop_p), int(seed), int(concat_chunks), ptr(ws), ws.numel(),
                                         stream(), _key=("flops", 2.0 * M * N * K), _name="planes_linear_bwd_input")
    else:
        L.planes_linear_bwd_input(dC.ptr(), dC.ld, dC.ps, ptr(W), W.stride(0), k_off, ptr(dA), dA.stride(0), M, N, K,
                                  ptr(ws), ws.numel(), stream(), _key=("flops", 2.0 * M * N * K))
    return dA


def planes_linear_bwd_weight(dC: Planes, X1: Planes, X2: Planes | None = None):
    """fp32 [N, K1+K2] = dC^T @ [X1 | X2]"""
    M, N = dC.rows, dC.cols
    K1, K2 = X1.cols, (X2.cols if X2 is not None else 0)
    dW = torch.empty(N, K1 + K2, dtype=torch.float32, device=dC.buf.device)
    L = lib()
    ws = _ws(L.planes_linear_bwd_weight_ws(M, N, K1, K2), dW.device)
    L.planes_linear_bwd_weight(dC.ptr(), dC.ld, dC.ps, X1.ptr(), X1.ld, X1.ps, K1, X2.ptr() if X2 is not None else None,
                               X2.ld if X2 is not None else 0, X2.ps if X2 is not None else 0, K2, ptr(dW),
                               dW.stride(0), M, N, ptr(ws), ws.numel(), stream(),
                               _key=("flops", 2.0 * M * N * (K1 + K2)))
    return dW


# ----------------------------------------------------------------------------------------------------- the plan
class LayerPlan:
    """One GATConv in a stack: which tensors it reads ([a] or [a | b], concatenation order) and which it writes."""

    def __init__(self, conv, inputs, output, mean_heads=False):
        self.conv, self.inputs, self.output, self.mean_heads = conv, list(inputs), output, bool(mean_heads)
        self.H, self.F = conv._num_heads, conv._out_feats
        self.res_mode = 0 if conv.res_fc is None else (1 if isinstance(conv.res_fc, torch.nn.Linear) else 2)
        self.width = self.F if mean_heads else self.H * self.F
        hf = self.H * self.F
        self.res_off = hf
        self.el_off = 2 * hf if self.res_mode == 1 else hf
        self.er_off = self.el_off + self.H
        self.ycols = self.er_off + self.H
        self.wide = False            # set by StackPlan once the input widths are known


class StackPlan:
    def __init__(self, layers, ext_widths, outputs):
        self.layers, self.ext_widths, self.outputs = layers, dict(ext_widths), list(outputs)
        self.widths = dict(ext_widths)
        self.producer = {}
        for i, L in enumerate(layers):
            self.widths[L.output] = L.width
            self.producer[L.output] = i
        self.consumers = {}          # tensor -> [(layer index, column offset inside the layer's concatenated input)]
        for i, L in enumerate(layers):
            off = 0
            for t in L.inputs:
                self.consumers.setdefault(t, []).append((i, off))
                off += self.widths[t]
            L.k_in = off
            L.in_offs = [sum(self.widths[t] for t in L.inputs[:j]) for j in range(len(L.inputs))]
            k1 = self.widths[L.inputs[0]]
            L.wide = (L.mean_heads and L.res_mode in (0, 1) and L.H in (1, 2, 4) and L.F % 32 == 0
                      and L.H * L.F <= 8192 and len(L.inputs) <= 2 and k1 % 64 == 0 and L.H * L.F >= 4 * L.k_in)

    def supported(self):
        for L in self.layers:
            if L.res_mode == 2 or L.H > 8 or L.F % 4 or len(L.inputs) > 2 or any(o % 4 for o in L.in_offs):
                return False
            if L.conv.fc.weight.shape[1] != L.k_in:
                return False
        return True


def _drop_p(conv, training):
    return conv.feat_drop_p if training else 0.0


class _Tape:
    pass


def _forward(plan: StackPlan, graph, ext, packed, biases, head, training, keep):
    """Runs the stack.  ext: {name: fp32 tensor}; packed[i]: [ycols, k_in] fp32; head: (W, b) or None.
    Returns (logits or None, {output name: fp32}, tape or None)."""
    _check_abi()
    L_ = lib()
    dev = graph.in_ptr.device
    N, E = graph.num_nodes, graph.num_edges
    nL = len(plan.layers)
    fseed = [ops.next_seed() for _ in range(nL)]
    aseed = [ops.next_seed() for _ in range(nL)]
    pdrop = [_drop_p(L.conv, training) for L in plan.layers]
    vkey = [i if pdrop[i] > 0.0 else -1 for i in range(nL)]
    variants = {}
    tape = _Tape() if keep else None
    if keep:
        tape.layers = [None] * nL
        tape.fseed, tape.aseed, tape.pdrop = fseed, aseed, pdrop
    outs = {}
    emb_planes = None
    for i, L in enumerate(plan.layers):
        conv = L.conv
        nch = (L.k_in + 3) // 4
        if ops.tracing() and pdrop[i] > 0.0:          # this layer's feat_drop mask over its concatenated input
            kept = split_planes(torch.ones(N, L.k_in, device=dev), pdrop[i], fseed[i], nch, 0).float() > 0
            ops.trace("drop", kept.float() * (1.0 / (1.0 - pdrop[i])))
        ins = []
        for t, off in zip(L.inputs, L.in_offs):
            key = (t, vkey[i])
            if key not in variants:
                if t not in ext:
                    raise SpgnnError(f"stack: tensor {t!r} consumed before it is produced")
                variants[key] = split_planes(ext[t], pdrop[i], fseed[i], nch, off // 4)
            ins.append(variants[key])
        # one planes copy of the output per distinct consumer mask (consumers without dropout share one)
        cons = plan.consumers.get(L.output, [])
        keys = []
        for ci, _ in cons:
            if vkey[ci] not in keys:
                keys.append(vkey[ci])
        is_out = L.output in plan.outputs
        want_head = head is not None and L.output == plan.outputs[0]
        if want_head and -1 not in keys:
            keys.append(-1)
        if len(keys) > 2:
            raise SpgnnError("stack: more than two dropout variants of one tensor are not supported")
        if L.wide and WIDE_OUTPUT_LAYER and all(k < 0 for k in keys):
            save_dact = keep and training and want_head and WIDE_SAVED_DACT and not ops.tracing()
            out32, P, rec = _wide_forward(L, graph, ins, packed[i], biases[i], conv, training, aseed[i], is_out,
                                          bool(keys), save_dact)
            if P is not None:
                variants[(L.output, -1)] = P
            if is_out:
                outs[L.output] = out32
            if want_head:
                emb_planes = P
            if keep:
                tape.layers[i] = rec
            for t in L.inputs:
                if all(ci <= i for ci, _ in plan.consumers[t]):
                    for k in [k for k in variants if k[0] == t]:
                        del variants[k]
            continue
        Y = planes_linear(ins[0], packed[i], A2=ins[1] if len(ins) > 1 else None)
        d = _Layer()
        d.in_ptr, d.in_src = ptr(graph.in_ptr), ptr(graph.in_src)
        d.N, d.H, d.F = N, L.H, L.F
        if TREE_KERNELS:
            d.node_off, d.B, d.max_nodes = ptr(graph.node_off), graph.batch_size, graph.max_nodes
            d.max_degree = graph.max_degree()
        d.Y, d.ldy, d.res_off, d.el_off, d.er_off = ptr(Y), Y.stride(0), L.res_off, L.el_off, L.er_off
        d.res_mode, d.act, d.negative_slope, d.mean_heads = L.res_mode, conv._act, conv.negative_slope, int(L.mean_heads)
        b = biases[i]
        d.bias = ptr(b)
        d.attn_drop_p = conv.attn_drop_p if training else 0.0
        d.attn_seed = aseed[i]
        if ops.tracing():
            ops.trace_gat(graph, Y[:, L.el_off:L.el_off + L.H], Y[:, L.er_off:L.er_off + L.H], d.attn_drop_p, aseed[i])
        att = torch.empty(E, L.H, dtype=torch.float32, device=dev)
        d.att = ptr(att)
        out32 = ops.empty_padded(N, L.width, dev) if is_out else None
        d.out, d.ldo = ptr(out32), (out32.stride(0) if out32 is not None else 0)
        d.n_sinks = len(keys)
        for s, k in enumerate(keys):
            P = Planes(N, L.width, dev)
            variants[(L.output, k)] = P
            sk = d.sinks[s]
            sk.hi, sk.ld, sk.plane_stride = P.ptr(), P.ld, P.ps
            if k >= 0:
                coff = [o for ci, o in cons if ci == k][0]
                sk.concat_chunks, sk.chunk_off = (plan.layers[k].k_in + 3) // 4, coff // 4
                sk.drop_p, sk.seed = pdrop[k], fseed[k]
            else:
                sk.concat_chunks, sk.chunk_off, sk.drop_p, sk.seed = 1, 0, 0.0, 0
        hf = L.H * L.F
        # SURVEY 8d: the kernel's ALGORITHMIC bytes read z, res, el, er once and write the output ONCE; every further
        # copy of the output (fp32 + one planes sink per distinct consumer mask) is implementation traffic
        n_writes = len(keys) + (1 if is_out else 0)
        algo = 4.0 * N * (hf * (2 if L.res_mode == 1 else 1) + 2 * L.H) + 4.0 * N * L.width + 4.0 * (N + 1) + 4.0 * E
        L_.gat_layer_fwd(ctypes.byref(d), stream(),
                         _key=("bytes", algo, algo + 4.0 * N * L.width * max(n_writes - 1, 0)))
        if is_out:
            outs[L.output] = out32
        if want_head:
            emb_planes = variants[(L.output, -1)]
        if keep:
            tape.layers[i] = (ins, Y, att, b)
        # inputs whose last consumer this was can go
        for t in L.inputs:
            if all(ci <= i for ci, _ in plan.consumers[t]):
                for k in [k for k in variants if k[0] == t]:
                    del variants[k]
    logits = None
    if head is not None:
        logits = planes_linear(emb_planes, head[0], head[1])
        if keep:
            tape.emb_planes = emb_planes
    return logits, outs, tape


class _WideRec:
    """Tape record of a layer evaluated aggregate-first."""
    __slots__ = ("XA", "att", "eler", "bias", "aseed", "kp", "dact")


def _wide_desc(L, graph, conv, training, aseed, XA, kp, eler, att):
    d = _Wide()
    d.in_ptr, d.in_src = ptr(graph.in_ptr), ptr(graph.in_src)
    d.out_ptr, d.out_dst, d.out_slot = ptr(graph.out_ptr), ptr(graph.out_dst), ptr(graph.out_slot)
    d.N, d.H, d.has_res = graph.num_nodes, L.H, int(L.res_mode == 1)
    d.eler, d.ld_eler = ptr(eler), eler.stride(0)
    d.negative_slope = conv.negative_slope
    d.attn_drop_p = conv.attn_drop_p if training else 0.0
    d.attn_seed = aseed
    d.att = ptr(att)
    d.XA, d.ldxa, d.psxa, d.kp = XA.ptr(), XA.ld, XA.ps, kp
    return d


def _wide_forward(L, graph, ins, W, bias, conv, training, aseed, want_out, want_planes, save_dact=False):
    """Head-averaged output layer, aggregate-first (spgnn_gat_aggx_fwd + spgnn_wide_linear mode 0).  save_dact: also
    keep act'(pre) of every head [N, H*F] on the tape for spgnn_wide_dpre."""
    L_ = lib()
    dev = graph.in_ptr.device
    N, E, H, F = graph.num_nodes, graph.num_edges, L.H, L.F
    hf, k_in = H * F, L.k_in
    has_res = int(L.res_mode == 1)
    kp = (k_in + 63) // 64 * 64
    rows0 = hf * (1 + has_res)
    eler = planes_linear(ins[0], W[rows0:rows0 + 2 * H], A2=ins[1] if len(ins) > 1 else None)
    XA = Planes(N, (H + 1) * kp, dev)
    att = torch.empty(E, H, dtype=torch.float32, device=dev)
    d = _wide_desc(L, graph, conv, training, aseed, XA, kp, eler, att)
    if ops.tracing():
        ops.trace_gat(graph, eler[:, :H], eler[:, H:2 * H], d.attn_drop_p, aseed)
    d.X1, d.ldx1, d.psx1, d.K1 = ins[0].ptr(), ins[0].ld, ins[0].ps, ins[0].cols
    if len(ins) > 1:
        d.X2, d.ldx2, d.psx2, d.K2 = ins[1].ptr(), ins[1].ld, ins[1].ps, ins[1].cols
    L_.gat_aggx_fwd(ctypes.byref(d), stream(),
                    _key=("bytes", 4.0 * N * (k_in + 2 * H) + 4.0 * N * (H + 1) * kp + 4.0 * (N + 1) + 4.0 * E))
    out32 = ops.empty_padded(N, F, dev) if want_out else None
    P = Planes(N, F, dev) if want_planes else None
    ws = _ws(L_.wide_linear_ws(H, F, kp, has_res), dev)
    outs = (ptr(out32), out32.stride(0) if out32 is not None else 0,
            P.ptr() if P is not None else None, P.ld if P is not None else 0, P.ps if P is not None else 0)
    flops = ("flops", 2.0 * N * hf * k_in * (1 + has_res))
    dact = None
    if save_dact:
        dact = torch.empty(N, hf, dtype=torch.float32, device=dev)
        L_.wide_linear_fwd_dact(XA.ptr(), XA.ld, XA.ps, kp, k_in, N, H, F, has_res, ptr(W), W.stride(0), ptr(bias),
                                conv._act, *outs, ptr(dact), dact.stride(0), ptr(ws), ws.numel(), stream(),
                                _key=flops, _name="wide_linear")
    else:
        L_.wide_linear(XA.ptr(), XA.ld, XA.ps, kp, k_in, N, H, F, has_res, ptr(W), W.stride(0), ptr(bias), conv._act,
                       0, *outs, None, 0, None, 0, None, 0, None, 0, 0, None, ptr(ws), ws.numel(), stream(), _key=flops)
    rec = _WideRec()
    rec.XA, rec.att, rec.eler, rec.bias, rec.aseed, rec.kp = XA, att, eler, bias, aseed, kp
    rec.dact = dact
    return out32, P, rec


def _wide_backward(L, graph, rec, W, gsrcs, training, need_bias, head_grad=None):
    """Returns (d packed weight [ycols, k_in], d bias or None, dX fp32 [N, k_in]).  head_grad: (planes of the head's
    output gradient, head weight) when the layer output feeds the head and rec.dact was saved; the head's dX is then
    the last gradient source, formed inside spgnn_wide_dpre."""
    L_ = lib()
    dev = graph.in_ptr.device
    N, E, H, F = graph.num_nodes, graph.num_edges, L.H, L.F
    hf, k_in, kp = H * F, L.k_in, rec.kp
    k4 = (k_in + 3) // 4 * 4
    has_res = int(L.res_mode == 1)
    conv = L.conv
    if not 1 <= len(gsrcs) + (head_grad is not None) <= 3:
        raise SpgnnError("stack: 1..3 gradient contributions to the output layer are supported")
    XA = rec.XA
    dpre = Planes(N, hf, dev)
    db = torch.empty(hf, dtype=torch.float32, device=dev) if rec.bias is not None and need_bias else None
    gp = [(ptr(g), g.stride(0)) for g in gsrcs] + [(None, 0)] * (3 - len(gsrcs))
    if head_grad is not None:
        glp, Wh = head_grad
        Wh = ops._rows(Wh)
        ws = _ws(L_.wide_dpre_ws(H, F), dev)
        L_.wide_dpre(glp.ptr(), glp.ld, glp.ps, glp.cols, N, H, F, ptr(Wh), Wh.stride(0), ptr(rec.dact),
                     rec.dact.stride(0), gp[0][0], gp[0][1], gp[1][0], gp[1][1], dpre.ptr(), dpre.ld, dpre.ps, ptr(db),
                     ptr(ws), ws.numel(), stream(),
                     _key=("bytes", 4.0 * N * hf * (2 + len(gsrcs) / H) + 4.0 * N * glp.cols))
        rec.dact = None
    else:
        ws = _ws(L_.wide_linear_ws(H, F, kp, has_res), dev)
        L_.wide_linear(XA.ptr(), XA.ld, XA.ps, kp, k_in, N, H, F, has_res, ptr(W), W.stride(0), ptr(rec.bias),
                       conv._act, 1, None, 0, None, 0, 0, gp[0][0], gp[0][1], gp[1][0], gp[1][1], gp[2][0], gp[2][1],
                       dpre.ptr(), dpre.ld, dpre.ps, ptr(db), ptr(ws), ws.numel(), stream(),
                       _key=("flops", 2.0 * N * hf * k_in * (1 + has_res)))
    ldx = (1 + has_res) * k4
    dXA = torch.empty(H, N, ldx, dtype=torch.float32, device=dev)
    x_view = PlanesView(XA, H * kp, k_in)
    dWz, dWres = [], []
    pad = k4 - k_in
    for h in range(H):
        dpre_h = PlanesView(dpre, h * F, F)
        dW_h = planes_linear_bwd_weight(dpre_h, PlanesView(XA, h * kp, k_in), x_view if has_res else None)
        dWz.append(dW_h[:, :k_in])
        blocks = [W[h * F:(h + 1) * F]] + ([W[hf + h * F:hf + (h + 1) * F]] if has_res else [])
        if pad:
            blocks = [torch.nn.functional.pad(b_, (0, pad)) for b_ in blocks]
        Wcat = torch.cat(blocks, 1) if len(blocks) > 1 else blocks[0].contiguous()
        planes_linear_bwd_input(dpre_h, Wcat, ldx, out=dXA[h])
        if has_res:
            dWres.append(dW_h[:, k_in:])
    del dpre
    rows0 = hf * (1 + has_res)
    w_eler = ops._rows(W[rows0:rows0 + 2 * H])
    if w_eler.stride(0) < k4:
        w_eler = torch.nn.functional.pad(w_eler, (0, k4 - k_in))
    d_eler = torch.empty(N, 2 * H, dtype=torch.float32, device=dev)
    dep = Planes(N, 2 * H, dev)
    ds = torch.empty(E * H, dtype=torch.float32, device=dev)
    dX = ops.empty_padded(N, k_in, dev)
    d = _wide_desc(L, graph, conv, training, rec.aseed, XA, kp, rec.eler, rec.att)
    # the backward kernels read x from XA; X1/X2 only have to pass the descriptor checks
    d.X1, d.ldx1, d.psx1 = XA.ptr(), XA.ld, XA.ps
    d.X2, d.ldx2, d.psx2 = XA.ptr(), XA.ld, XA.ps
    d.K1, d.K2 = _wide_k_split(L, k_in)
    d.dXA, d.ld_dxa, d.head_stride = ptr(dXA), ldx, N * ldx
    d.w_eler, d.ld_w = ptr(w_eler), w_eler.stride(0)
    d.ds_ws = ptr(ds)
    d.d_eler, d.ld_de = ptr(d_eler), d_eler.stride(0)
    d.d_eler_planes, d.ld_dep, d.ps_dep = dep.ptr(), dep.ld, dep.ps
    d.dX, d.ld_dx = ptr(dX), dX.stride(0)
    L_.gat_aggx_bwd(ctypes.byref(d), stream(),
                    _key=("bytes", 4.0 * N * (H * ldx + 2 * k_in + 4 * H) + 4.0 * N * H * k4 + 8.0 * (N + 1) + 12.0 * E))
    dW_eler = planes_linear_bwd_weight(dep, x_view)
    d_packed = torch.cat(dWz + dWres + [dW_eler], 0)
    return d_packed, db, dX


def _wide_k_split(L, k_in):
    """(K1, K2) of the layer's concatenated input as the aggx descriptor wants them (K1 % 64 == 0)."""
    k1 = L.in_offs[1] if len(L.in_offs) > 1 else k_in
    return k1, k_in - k1


def _grad_rows(g):
    """fp32 gradient tensor usable as a gradient source: unit inner stride, 16-byte aligned rows."""
    g = ops._rows(g)
    if g.stride(0) % 4 or g.data_ptr() % 16:
        p = ops.empty_padded(g.shape[0], g.shape[1], g.device)
        p.copy_(g)
        g = p
    return g


def _backward(plan: StackPlan, graph, tape, packed, head, g_logits, g_outs, need_bias):
    """Returns (d packed[i], d bias[i], d head W, d head b)."""
    L_ = lib()
    dev = graph.in_ptr.device
    N, E = graph.num_nodes, graph.num_edges
    nL = len(plan.layers)
    d_packed, d_bias = [None] * nL, [None] * nL
    d_hw = d_hb = None
    extra = {}          # tensor -> [fp32 gradient tensors without a mask]
    head_grad = {}      # tensor -> (head output-gradient planes, head weight): dX of the head formed by its consumer
    for name, g in g_outs.items():
        if g is not None:
            extra.setdefault(name, []).append(_grad_rows(g))
    if head is not None and g_logits is not None:
        gl = _grad_rows(g_logits)
        glp = split_planes(gl)
        d_hw = planes_linear_bwd_weight(glp, tape.emb_planes)
        d_hb = ops.colsum(gl)
        rec = tape.layers[plan.producer[plan.outputs[0]]] if plan.outputs[0] in plan.producer else None
        if isinstance(rec, _WideRec) and rec.dact is not None and head[0].shape[0] <= 64:    # one k-block of classes
            head_grad[plan.outputs[0]] = (glp, head[0])
        else:
            extra.setdefault(plan.outputs[0], []).append(planes_linear_bwd_input(glp, head[0], head[0].shape[1]))
        tape.emb_planes = None
    dX = {}             # layer index -> fp32 [N, k] gradient of its concatenated (dropped) input
    # layers whose dX already includes their own feat_drop mask: the mask is applied in the dX GEMM epilogue
    # (tensor-bound, idle issue slots) rather than in the producing layer's aggregation backward (issue-bound: the
    # mask hash was a quarter of its destination-side instructions).  The aggregate-first backward's dX is unmasked.
    masked = set()
    for i in range(nL - 1, -1, -1):
        L = plan.layers[i]
        conv = L.conv
        srcs = []
        for ci, off in plan.consumers.get(L.output, []):
            if ci in dX and dX[ci] is not None and off < dX[ci].shape[1]:
                pm = 0.0 if ci in masked else tape.pdrop[ci]
                srcs.append((dX[ci], off, pm, tape.fseed[ci], (plan.layers[ci].k_in + 3) // 4))
        for g in extra.get(L.output, []):
            srcs.append((g, 0, 0.0, 0, 1))
        hg = head_grad.pop(L.output, None)
        if not srcs and hg is None:
            dX[i] = None          # nothing flows into this layer: its parameters get no gradient
            tape.layers[i] = None
            continue
        if len(srcs) + (hg is not None) > 3:
            raise SpgnnError("stack: more than three gradient contributions to one tensor are not supported")
        hf = L.H * L.F
        if isinstance(tape.layers[i], _WideRec):
            rec = tape.layers[i]
            tape.layers[i] = None
            # every consumer of an aggregate-first layer has no feat_drop (see _forward), so no source is masked
            if any(off for _, off, *_ in srcs):
                raise SpgnnError("stack: a head-averaged output layer cannot take a gradient at a column offset")
            d_packed[i], d_bias[i], dX[i] = _wide_backward(L, graph, rec, packed[i], [g for g, *_ in srcs],
                                                           tape.training, need_bias[i], hg)
            continue
        ins, Y, att, b = tape.layers[i]
        tape.layers[i] = None
        dY = Planes(N, L.ycols, dev)
        d = _Layer()
        d.in_ptr, d.in_src = ptr(graph.in_ptr), ptr(graph.in_src)
        d.out_ptr, d.out_dst, d.out_slot = ptr(graph.out_ptr), ptr(graph.out_dst), ptr(graph.out_slot)
        d.N, d.H, d.F = N, L.H, L.F
        if TREE_KERNELS:
            d.node_off, d.B, d.max_nodes = ptr(graph.node_off), graph.batch_size, graph.max_nodes
            d.max_degree = graph.max_degree()
        d.Y, d.ldy, d.res_off, d.el_off, d.er_off = ptr(Y), Y.stride(0), L.res_off, L.el_off, L.er_off
        d.res_mode, d.act, d.negative_slope, d.mean_heads = L.res_mode, conv._act, conv.negative_slope, int(L.mean_heads)
        d.bias = ptr(b)
        d.attn_drop_p = conv.attn_drop_p if tape.training else 0.0
        d.attn_seed = tape.aseed[i]
        d.att = ptr(att)
        d.n_gsrc = len(srcs)
        for s, (g, off, p, seed, nch) in enumerate(srcs):
            gs = d.gsrc[s]
            gs.g, gs.ld = g.data_ptr() + 4 * off, g.stride(0)
            gs.concat_chunks, gs.chunk_off, gs.drop_p, gs.seed = nch, off // 4, p, seed
        d.dY_hi, d.dY_ld, d.dY_ps = dY.ptr(), dY.ld, dY.ps
        g_ws = torch.empty(N, hf, dtype=torch.float32, device=dev) if L.res_mode != 1 else None
        ds = torch.empty(E * L.H, dtype=torch.float32, device=dev)
        d.g_ws, d.ds_ws = ptr(g_ws), ptr(ds)
        db = dbw = None
        if b is not None and need_bias[i]:
            db = torch.empty(hf, dtype=torch.float32, device=dev)
            dbw = _ws(L_.gat_layer_dbias_ws(N, L.H, L.F), dev)
        d.dbias, d.dbias_ws = ptr(db), ptr(dbw)
        # algorithmic (SURVEY 8d): ONE gradient of the layer output, z (+ residual projection), el/er read once; dY
        # written once (4 bytes per column: dz | G as the residual part | d el, d er) + indices and edge scalars.
        # Implementation: every further gradient source (one per consumer) and the G workspace without a residual.
        algo = 4.0 * N * (L.width + hf * (2 if L.res_mode == 1 else 1) + 2 * L.H) + 4.0 * N * L.ycols \
            + 8.0 * (N + 1) + 12.0 * E + 8.0 * E * L.H
        impl = algo + 4.0 * N * L.width * (len(srcs) - 1) + (0.0 if L.res_mode == 1 else 4.0 * N * hf)
        L_.gat_layer_bwd(ctypes.byref(d), stream(), _key=("bytes", algo, impl))
        d_bias[i] = db
        d_packed[i] = planes_linear_bwd_weight(dY, ins[0], ins[1] if len(ins) > 1 else None)
        # dX only over the leading inputs that are produced inside the stack
        k_need = 0
        for t, off in zip(L.inputs, L.in_offs):
            if t in plan.producer:
                k_need = off + plan.widths[t]
        dX[i] = planes_linear_bwd_input(dY, packed[i], k_need, drop_p=tape.pdrop[i], seed=tape.fseed[i],
                                        concat_chunks=(L.k_in + 3) // 4) if k_need else None
        masked.add(i)
        del dY, Y, att, ins
    return d_packed, d_bias, d_hw, d_hb


class StackFn(Function):
    """(logits | None, *outputs) = stack(ext inputs; packed weights, biases, head) with a hand-written backward."""

    @staticmethod
    def forward(ctx, plan, graph, training, ext_names, n_layers, has_head, grad_enabled, *tensors):
        ext = dict(zip(ext_names, tensors[:len(ext_names)]))
        o = len(ext_names)
        packed = list(tensors[o:o + n_layers])
        biases = list(tensors[o + n_layers:o + 2 * n_layers])
        head = (tensors[o + 2 * n_layers], tensors[o + 2 * n_layers + 1]) if has_head else None
        # no tape when the caller runs without autograd (forward() itself always runs with grad mode off)
        keep = grad_enabled and any(t is not None and t.requires_grad for t in tensors[o:])
        logits, outs, tape = _forward(plan, graph, ext, packed, biases, head, training, keep)
        ctx.plan, ctx.graph, ctx.tape, ctx.n_ext, ctx.n_layers, ctx.has_head = plan, graph, tape, o, n_layers, has_head
        if tape is not None:
            tape.training = training
            tape.packed, tape.head = packed, head
        ctx.set_materialize_grads(False)
        res = tuple(outs[n] for n in plan.outputs)
        return ((logits,) + res) if has_head else res

    @staticmethod
    def backward(ctx, *grads):
        plan, tape, nL = ctx.plan, ctx.tape, ctx.n_layers
        if tape is None or tape.layers is None:
            raise SpgnnError("stack backward called twice (the tape is released after the first backward)")
        if ctx.has_head:
            g_logits, g_outs = grads[0], dict(zip(plan.outputs, grads[1:]))
        else:
            g_logits, g_outs = None, dict(zip(plan.outputs, grads))
        o = ctx.n_ext
        need = ctx.needs_input_grad[7:]
        need_bias = [need[o + nL + i] for i in range(nL)]
        d_packed, d_bias, d_hw, d_hb = _backward(plan, ctx.graph, tape, tape.packed, tape.head, g_logits, g_outs, need_bias)
        tape.layers = None
        out = [None] * 7 + [None] * o + d_packed + d_bias
        if ctx.has_head:
            out += [d_hw, d_hb]
        return tuple(out)


def run_stack(plan: StackPlan, graph, ext, training, head=None):
    """ext: {name: fp32 [N, width]}.  Returns (logits or None, [outputs in plan.outputs order])."""
    for t in ext.values():
        if t.requires_grad:
            raise SpgnnError("stack: gradients with respect to the stack inputs are not supported (use the layer API)")
    names = list(ext)
    packed = [L.conv._packed_weight() for L in plan.layers]
    biases = [L.conv.bias for L in plan.layers]
    args = [ext[n] for n in names] + packed + biases
    if head is not None:
        args += [head.weight, head.bias]
    res = StackFn.apply(plan, graph, bool(training), tuple(names), len(plan.layers), head is not None,
                        torch.is_grad_enabled(), *args)
    if head is not None:
        return res[0], list(res[1:])
    return None, list(res)
