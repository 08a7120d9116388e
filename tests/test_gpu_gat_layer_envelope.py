"""The GAT aggregation kernels of every hidden layer over everything their entry points accept, not just the H = 2,
F in {64, 128, 256}, ELU / tanh, ~300-node trees of the shipped presets.

* spgnn_gat_layer_fwd / _bwd, called directly with a stack._Layer descriptor built as stack._forward / _backward do.
  The entry point picks the per-tree kernels (csrc/gat_tree.cu: one CTA per tree, z slices staged by TMA, one or two
  shared-memory stages, slices or heads of a tree split across CTAs for small batches) or the chunk kernels
  (csrc/gat_layer.cu).  Every case states the regime it is meant to reach; the test checks that claim against the
  shared-memory arithmetic of gat_tree.cu restated below, and the profiler trace shows the exact launch.
* spgnn_gat_agg_fwd / _bwd (csrc/gat.cu), the per-layer path behind nn.GATConv.forward_flat: the fast H <= 2 kernel
  next to the general one, every backward column bucket, identity residuals, head means and the F > 1024 refusal.
* nn.GATConv with the activations that take the kernels' runtime branch (leaky_relu, relu) against the DGL oracle,
  on the per-layer path and as an aggregate-first output layer.

References are plain fp64 formulas on the CPU.  Every output buffer starts as NaN, so an entry a kernel does not write
fails the comparison."""
import copy
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import assert_grads_match, rel_err, replay, traced
from test_gpu_parity import GRAD_TOL, TRAIN_GRAD_TOL, _random_tree_adj

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NONE, ELU, TANH, RELU, LEAKY = 0, 1, 2, 3, 4         # SPGNN_ACT_*
LEAKY_SLOPE = 0.01         # F.leaky_relu's default negative_slope: what GATConv(activation=F.leaky_relu) computes
NEG_SLOPE = 0.2            # LeakyReLU slope of the attention logits
# fp32 kernels vs fp64, relative to each output's largest entry.  The planes outputs (sinks, dY) are hi + lo bf16
# planes, exact to ~2^-17 relative; the remaining error is fp32 rounding of the <= 4-term (generic: <= 8-term) sums and
# of the fast exponentials, well below this bound.
TOL = 3e-5
NAN = float("nan")


def _load_mods():
    from oracle import dgl_ops
    from spgnn_b200 import graph as sg, nn as snn, ops, stack
    from spgnn_b200._lib import SpgnnError, lib, ptr, stream
    return dict(dgl_ops=dgl_ops, sg=sg, snn=snn, ops=ops, stack=stack, SpgnnError=SpgnnError, lib=lib, ptr=ptr,
                stream=stream)


@pytest.fixture(scope="module")
def mods():
    return _load_mods()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ gat_tree.cu restated
# fwd_smem_bytes (gat_tree.cu:125), bwd_smem_bytes (:309), kSmemLimit, applicable() and the launch shapes of
# launch_fwd_act / launch_bwd_act.  nstages is a runtime value, so the regime of a case is computed here.
SMEM_LIMIT = 232448
TREE_MAX_NODES = 384


def fwd_smem_bytes(nmax, H, nstages):
    return 128 + nmax * (4 + 8 + H * 16) + 128 + nstages * nmax * 32 * 4 + 128


def bwd_smem_bytes(nmax, H, HF, nstages, nwarps):
    return (128 + nmax * (12 + 24 + 5 * H * 16) + nwarps * 32 * 4 + HF * 4 + 128 + (nstages + 1) * nmax * 32 * 4
            + 128)


def fwd_shape(n, variant=0):
    """(threads, rounds per slice); SPGNN_TREE_FWD=1 selects variant 1"""
    if variant == 1:
        return (896, 3) if n <= 3 * 112 else (896, 4)
    return (512, 5) if n <= 5 * 64 else (512, 6)


def bwd_shape(n, variant=3):
    """(threads, rounds per slice, prefetch depth); SPGNN_TREE_BWD = 0 / 1 / 9 select the alternatives"""
    if variant == 0:
        return (512, 5, 5) if n <= 5 * 64 else (512, 6, 6)
    if variant == 1:
        return (896, 3, 2) if n <= 3 * 112 else (896, 4, 2)
    if variant == 9:
        return (640, 4, 2) if n <= 4 * 80 else (640, 5, 2)
    return (640, 4, 3) if n <= 4 * 80 else (640, 5, 2)


def tree_plan(H, F, mean, max_nodes, max_degree, B, n_g, tree, sms, fvar=0, bvar=3):
    """(forward launch or None, backward launch or None) of the per-tree kernels; None: the chunk kernels run."""
    fwd = bwd = None
    if not (tree and B > 0 and 0 < max_nodes <= TREE_MAX_NODES and 0 < max_degree <= 4 and not mean and F % 64 == 0
            and H <= 8):
        return fwd, bwd
    nmax = -(-max_nodes // 32) * 32
    nslices = H * F // 32
    T, K = fwd_shape(max_nodes, fvar)
    st = 2 if fwd_smem_bytes(nmax, H, 2) <= SMEM_LIMIT else 1
    if fwd_smem_bytes(nmax, H, st) <= SMEM_LIMIT:
        fwd = dict(threads=T, kper=K, stages=st, split=min(sms // B, nslices) if B < sms else 1, nslices=nslices)
    if 1 <= n_g <= 2:
        T, K, PF = bwd_shape(max_nodes, bvar)
        st = 2 if bwd_smem_bytes(nmax, H, H * F, 2, T // 32) <= SMEM_LIMIT else 1
        if bwd_smem_bytes(nmax, H, H * F, st, T // 32) <= SMEM_LIMIT:
            bwd = dict(threads=T, kper=K, pf=PF, stages=st, split=H if H > 1 and B * H <= sms else 1,
                       headroom=SMEM_LIMIT - bwd_smem_bytes(nmax, H, H * F, st, T // 32))
    return fwd, bwd


def _profiled(run):
    """Short names of the GAT kernels run() launches.  A throwaway kernel opens the session: the profiler has been
    seen to drop the first launch of a session."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        run()
        torch.cuda.synchronize()
    return _kernels(prof)


def _kernels(prof):
    """Short names of the GAT kernels a profiler trace holds, template arguments included: 'gat_tree_fwd_kernel<1,512,5>'"""
    names = set()
    for e in prof.events():
        m = re.search(r"(\w+_kernel)\s*(<[\d,\s]*>)?\s*\(", e.name)
        if m and ("gat" in m.group(1) or "dbias" in m.group(1)):
            names.add(m.group(1) + re.sub(r"\s+", "", m.group(2) or ""))
    return names


# ------------------------------------------------------------------------------------------------ graphs
def _with_degree5(adj):
    """One more leaf under a non-root node that already has two children: that node gets in-degree 5."""
    n = adj.shape[0]
    deg = adj.sum(1)
    v = int(next(i for i in range(1, n) if deg[i] == 4))
    out = np.zeros((n + 1, n + 1), dtype=np.uint8)
    out[:n, :n] = adj
    out[n, n] = out[n, v] = out[v, n] = 1
    return out


def _with_holes(adj):
    """Three isolated nodes appended.  Returns the adjacency and the local ids whose self loops _drop_self_loops
    removes: three leaves (in-degree 1) and the isolated nodes (in-degree 0)."""
    n = adj.shape[0]
    out = np.zeros((n + 3, n + 3), dtype=np.uint8)
    out[:n, :n] = adj
    for i in range(n, n + 3):
        out[i, i] = 1
    leaves = [i for i in range(1, n) if adj[i].sum() == 2][:3]
    return out, leaves + [n, n + 1, n + 2]


def _drop_self_loops(sg, g, nodes):
    """The batch g without the self loops of ``nodes`` (global ids): the batch builder gives every node a self loop,
    so in-degree 0 only exists at the descriptor level."""
    drop = torch.zeros(g.num_nodes, dtype=torch.bool, device=g.src.device)
    drop[torch.tensor(nodes, device=g.src.device)] = True
    keep = ~((g.src == g.dst) & drop[g.src])
    gid = torch.repeat_interleave(torch.arange(g.batch_size, device=g.src.device), g.batch_num_edges())
    n_edges = torch.bincount(gid[keep], minlength=g.batch_size)
    return sg.Graph.from_edge_lists(g.batch_num_nodes(), n_edges, g.src_local[keep], g.dst_local[keep],
                                    max_nodes=g.max_nodes)


def build_graph(sg, sizes, max_children=2, holes=False, deg5=False, seed=0):
    rng = np.random.default_rng(seed)
    sizes = list(sizes)
    if (sum(sizes) + 3 * holes + deg5) % 32 == 0:
        # N must not be a multiple of 32 (the TMA boxes of the last tree then run past N): grow a tree that is not
        # the largest, so the regime stays the same
        i = next(i for i, n in enumerate(sizes[:-1]) if n < max(sizes) - 1)
        sizes[i] += 1
    adjs = [_random_tree_adj(int(n), max_children, rng) for n in sizes]
    if deg5:
        adjs[0] = _with_degree5(adjs[0])
    loops = []
    if holes:
        adjs[-1], loops = _with_holes(adjs[-1])
    g = sg.batch_from_adjs(adjs)
    if holes:
        off = g.num_nodes - adjs[-1].shape[0]
        g = _drop_self_loops(sg, g, [off + i for i in loops])
        assert int((g.in_degrees() == 0).sum()) == 3
    return g, adjs


def _csc_dst(g):
    in_ptr = g.in_ptr.long().cpu()
    return torch.repeat_interleave(torch.arange(g.num_nodes), in_ptr[1:] - in_ptr[:-1])


# ------------------------------------------------------------------------------------------------ fp64 reference
def act64(x, act, branch):
    if act == NONE:
        return x
    if act == ELU:
        return torch.where(x > 0, x, torch.expm1(x))
    if act == TANH:
        return torch.tanh(x)
    return torch.where(branch, x, (0.0 if act == RELU else LEAKY_SLOPE) * x)


def gat_ref64(g, Y, H, F, res_mode, el_off, er_off, bias, act, mean, keep, gsum, branch, xres=None):
    """out = act(sum_u att * keep * z[u] + res + b) (mean over heads), att = softmax over the in-edges of
    LeakyReLU(el[u] + er[v]); gradients of sum(out * gsum) by fp64 autograd.  The LeakyReLU branch of every logit is
    taken from the fp32 sum the kernels compute, the ReLU / LeakyReLU branch of every pre-activation from ``branch``
    (the sign of the device's fp32 output)."""
    N, HF = Y.shape[0], H * F
    src, dst = g.in_src.long().cpu(), _csc_dst(g)
    Y64 = Y.double()
    z = Y64[:, :HF].clone().requires_grad_()
    el = Y64[:, el_off:el_off + H].clone().requires_grad_()
    er = Y64[:, er_off:er_off + H].clone().requires_grad_()
    res = xr = None
    if res_mode == 1:
        res = Y64[:, HF:2 * HF].clone().requires_grad_()
        res_full = res
    elif res_mode == 2:
        xr = xres.double().clone().requires_grad_()
        res_full = xr.repeat(1, HF // xr.shape[1])          # column hc reads xres[:, hc % xres_cols]
    b = bias.double().clone().requires_grad_() if bias is not None else None
    pos = (Y[:, el_off:el_off + H][src] + Y[:, er_off:er_off + H][dst]) > 0
    raw = el[src] + er[dst]
    e = torch.where(pos, raw, NEG_SLOPE * raw)
    m = torch.full((N, H), -torch.inf, dtype=torch.float64).scatter_reduce(0, dst[:, None].expand(-1, H), e.detach(),
                                                                          "amax")
    p = torch.exp(e - m[dst])
    a = p / torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, p)[dst]
    w = a * keep if keep is not None else a
    pre = torch.zeros(N, H, F, dtype=torch.float64).index_add(0, dst, w[:, :, None] * z.view(N, H, F)[src])
    pre = pre + (res_full.view(N, H, F) if res_mode else 0) + (b.view(H, F) if b is not None else 0)
    pre.retain_grad()
    y = act64(pre, act, branch)
    out = y.mean(1) if mean else y.reshape(N, HF)
    (out * gsum).sum().backward()
    return dict(att=a.detach(), out=out.detach(), dz=z.grad, G=pre.grad.reshape(N, HF), del_=el.grad, der=er.grad,
                db=b.grad if b is not None else None, dxres=xr.grad if xr is not None else None)


def _random_y(N, H, F, res_mode, seed):
    """Y [N, ldy] with the stack's column layout z | res (res_mode 1) | el | er, ldy padded to 32 columns as
    planes_linear pads it, exactly N rows."""
    HF = H * F
    el_off = 2 * HF if res_mode == 1 else HF
    er_off = el_off + H
    ldy = (er_off + H + 31) // 32 * 32
    gen = torch.Generator().manual_seed(seed)
    Y = torch.randn(N, ldy, generator=gen)
    if res_mode == 1:
        Y[:, HF:2 * HF] *= 0.5
    return Y, el_off, er_off


# ------------------------------------------------------------------------------------------------ spgnn_gat_layer
def run_layer_case(mods, c, fvar=0, bvar=3):
    """One forward + backward of spgnn_gat_layer on case ``c`` under the profiler, checked against fp64.  Returns the
    short names of the kernels that ran."""
    sg, stack, ops, lib, ptr, stream = (mods[k] for k in ("sg", "stack", "ops", "lib", "ptr", "stream"))
    sms = _sms()
    H, F, res, act, mean = c["H"], c["F"], c.get("res", 1), c.get("act", ELU), c.get("mean", False)
    sizes = c["sizes"](sms) if callable(c["sizes"]) else c["sizes"]
    g, _ = build_graph(sg, sizes, c.get("max_children", 2), c.get("holes", False), c.get("deg5", False),
                       seed=H * 1000 + F)
    N, E, HF = g.num_nodes, g.num_edges, H * F
    W = F if mean else HF
    tree = c.get("tree", True)
    max_degree = c.get("max_degree", g.max_degree())
    gsrc, sinks, attn_p = c.get("gsrc", (0.0,)), c.get("sinks", ()), c.get("attn_p", 0.0)
    want_out, want_bias, want_db = c.get("out", True), c.get("bias", True), c.get("dbias", True)
    assert N % 32 and g.max_nodes and int(g.batch_num_nodes()[-1]) % 32, "the last tree's boxes must run past N"

    # the regime the case claims, from the restated shared-memory arithmetic
    fwd, bwd = tree_plan(H, F, mean, g.max_nodes, max_degree, g.batch_size, len(gsrc), tree, sms, fvar, bvar)
    claim_f, claim_b = c["regime"]
    assert (fwd is None) == (claim_f == "chunk"), (fwd, claim_f)
    if claim_f != "chunk" and claim_f != "tree":
        assert claim_f == f"tree{fwd['kper']}", (fwd, claim_f)
    assert (bwd is None) == (claim_b == "chunk"), (bwd, claim_b)
    if bwd is not None:
        assert claim_b == f"tree{bwd['stages']}", (bwd, claim_b)
    if "fsplit" in c:
        assert fwd["split"] > 1 and (fwd["nslices"] % fwd["split"] != 0) == (c["fsplit"] == "uneven"), fwd
    if "bsplit" in c:
        assert (bwd["split"] > 1) == c["bsplit"], bwd
    if c.get("grid_stride"):
        assert g.batch_size > sms
    if "headroom" in c:
        assert 0 <= bwd["headroom"] <= c["headroom"], bwd

    Y, el_off, er_off = _random_y(N, H, F, res, seed=N + HF)
    Yd = Y.cuda()
    gen = torch.Generator().manual_seed(HF + len(gsrc))
    bias = (0.3 * torch.randn(HF, generator=gen)) if want_bias else None
    bias_d = bias.cuda() if bias is not None else None
    att = torch.full((E, H), NAN, device="cuda")
    out = torch.full((N, W), NAN, device="cuda") if want_out else None
    aseed = 77 + H
    d = stack._Layer()
    d.in_ptr, d.in_src = ptr(g.in_ptr), ptr(g.in_src)
    d.out_ptr, d.out_dst, d.out_slot = ptr(g.out_ptr), ptr(g.out_dst), ptr(g.out_slot)
    d.N, d.H, d.F = N, H, F
    if tree:
        d.node_off, d.B, d.max_nodes, d.max_degree = ptr(g.node_off), g.batch_size, g.max_nodes, max_degree
    d.Y, d.ldy, d.res_off, d.el_off, d.er_off = ptr(Yd), Yd.stride(0), HF, el_off, er_off
    d.res_mode, d.act, d.negative_slope, d.mean_heads = res, act, NEG_SLOPE, int(mean)
    d.bias = ptr(bias_d)
    d.attn_drop_p, d.attn_seed = attn_p, aseed
    d.att = ptr(att)
    d.out, d.ldo = ptr(out), (W if out is not None else 0)
    # sinks: a masked one sits at column 8 of a consumer input 12 columns wider than this layer's output
    planes, sink_masks = [], []
    d.n_sinks = len(sinks)
    for s, p in enumerate(sinks):
        P = stack.Planes(N, W, "cuda")
        P.buf.fill_(NAN)
        sk = d.sinks[s]
        sk.hi, sk.ld, sk.plane_stride = P.ptr(), P.ld, P.ps
        nch, off = ((W + 12) // 4, 2) if p > 0 else (1, 0)
        sk.concat_chunks, sk.chunk_off, sk.drop_p, sk.seed = nch, off, p, 500 + s
        planes.append(P)
        sink_masks.append(stack.split_planes(torch.ones(N, W, device="cuda"), p, 500 + s, nch, off).float().cpu()
                          if p > 0 else None)
    # gradient sources: column 8 of a [N, W + 12] consumer dX; masked ones with the consumer's feat_drop convention
    gbufs, gsum = [], torch.zeros(N, W, dtype=torch.float64)
    d.n_gsrc = len(gsrc)
    for q, p in enumerate(gsrc):
        buf = torch.randn(N, W + 12, generator=gen)
        gv = buf[:, 8:8 + W].double()
        nch, off = ((W + 12) // 4, 2) if p > 0 else (1, 0)
        if p > 0:
            gv = gv * stack.split_planes(torch.ones(N, W, device="cuda"), p, 900 + q, nch, off).float().cpu().double()
        gsum += gv
        buf = buf.cuda()
        gbufs.append(buf)
        gs = d.gsrc[q]
        gs.g, gs.ld = buf.data_ptr() + 4 * 8, buf.stride(0)
        gs.concat_chunks, gs.chunk_off, gs.drop_p, gs.seed = nch, off, p, 900 + q
    dY = stack.Planes(N, er_off + H, "cuda")
    dY.buf.fill_(NAN)
    d.dY_hi, d.dY_ld, d.dY_ps = dY.ptr(), dY.ld, dY.ps
    g_ws = torch.full((N, HF), NAN, device="cuda") if res != 1 else None
    ds = torch.full((E * H,), NAN, device="cuda")
    d.g_ws, d.ds_ws = ptr(g_ws), ptr(ds)
    db = dbw = None
    if want_db and bias is not None:
        db = torch.full((HF,), NAN, device="cuda")
        dbw = torch.full((int(lib().gat_layer_dbias_ws(N, H, F)) // 4,), NAN, device="cuda")
    d.dbias, d.dbias_ws = ptr(db), ptr(dbw)
    torch.cuda.synchronize()

    def run():
        lib().gat_layer_fwd(ctypes.byref(d), stream())
        lib().gat_layer_bwd(ctypes.byref(d), stream())

    names = _profiled(run)

    # the launches the regime implies, and nothing else
    A = act if act in (ELU, TANH) else 0
    want = set()
    if fwd is not None:
        want.add(f"gat_tree_fwd_kernel<{A},{fwd['threads']},{fwd['kper']}>")
    else:
        want.add("gat_layer_fwd_kernel")
    if bwd is not None:
        want.add(f"gat_tree_bwd_kernel<{len(gsrc)},{A},{bwd['threads']},{bwd['kper']},{bwd['pf']}>")
        if db is not None:
            want.add("tree_dbias_reduce_kernel")
    else:
        want |= {"gat_layer_bwd_dst_kernel", "gat_layer_bwd_src_kernel"} | ({"dbias_reduce_kernel"} if db is not None
                                                                          else set())
    assert names == want, (sorted(names), sorted(want))

    # fp64 reference
    keep = ops.drop_mask(E, H, attn_p, aseed, "cuda").cpu().double() if attn_p > 0 else None
    branch = None
    if act in (RELU, LEAKY):
        assert not mean, "the pre-activation branch is read from the device output"
        src = out.cpu() if out is not None else planes[sinks.index(0.0)].float().cpu()
        branch = (src > 0).view(N, H, F)
    ref = gat_ref64(g, Y, H, F, res, el_off, er_off, bias, act, mean, keep, gsum, branch)
    assert rel_err(att.cpu(), ref["att"]) < TOL, "att"
    if out is not None:
        assert rel_err(out.cpu(), ref["out"]) < TOL, "out"
    for s, P in enumerate(planes):
        r = ref["out"] * sink_masks[s].double() if sink_masks[s] is not None else ref["out"]
        assert rel_err(P.float().cpu(), r) < TOL, f"sink {s}"
    dYf = dY.float().cpu()
    assert rel_err(dYf[:, :HF], ref["dz"]) < TOL, "dz"
    if res == 1:
        assert rel_err(dYf[:, HF:2 * HF], ref["G"]) < TOL, "G (residual part of dY)"
    assert rel_err(dYf[:, el_off:el_off + H], ref["del_"]) < TOL, "d el"
    assert rel_err(dYf[:, er_off:er_off + H], ref["der"]) < TOL, "d er"
    if db is not None:
        assert rel_err(db.cpu(), ref["db"]) < TOL, "dbias"
    return names


def _case(name, H, F, sizes, regime, **kw):
    return pytest.param(dict(H=H, F=F, sizes=sizes, regime=regime, **kw), id=name)


def _uneven_batch(sms, nslices=64):
    """The smallest B >= 2 with #SMs % B != 0 and #SMs / B < nslices: the forward splits every tree unevenly."""
    B = next(b for b in range(2, sms) if sms % b and sms // b < nslices and nslices % (sms // b))
    return [200 - 7 * i for i in range(B)]


# regime = (forward, backward): forward "tree5" / "tree6" (<ACT, 512, 5|6>) or "chunk"; backward "tree2" / "tree1"
# (shared-memory stages of <NG, ACT, 640, 4|5, 3|2>) or "chunk".  Every axis takes every value at least once:
# H {1,2,3,4,8}; F {64,128,192,256,512} per tree, {4,36,96} chunk only; res_mode {0,1}; bias / dbias; 0-2 sinks with
# and without feat_drop; out or not; 1-3 gradient sources, masked and not; attention dropout; all five activations.
LAYER_CASES = [
    _case("headline_h2_f256_2stages", 2, 256, [301] * 6 + [297], ("tree5", "tree2"), act=ELU, sinks=(0.0, 0.1),
          gsrc=(0.1, 0.0), attn_p=0.1, holes=True),
    _case("h2_f512_384_2stages_2.6kb_headroom", 2, 512, [384, 200, 157], ("tree6", "tree2"), act=TANH, res=0,
          bias=False, gsrc=(0.1,), headroom=2700),
    _case("h4_f64_301_1stage", 4, 64, [301, 301, 301, 250], ("tree5", "tree1"), act=RELU, sinks=(0.1,),
          gsrc=(0.0, 0.2)),
    _case("h3_f64_384_1stage", 3, 64, [384, 77], ("tree6", "tree1"), act=LEAKY, res=0, sinks=(0.0,), out=False,
          attn_p=0.2, holes=True),
    _case("h8_f64_224_1stage", 8, 64, [224, 100], ("tree5", "tree1"), act=NONE, dbias=False, gsrc=(0.2,)),
    _case("h4_f64_384_bwd_smem_fallback", 4, 64, [384, 130], ("tree6", "chunk"), act=ELU, gsrc=(0.0, 0.1),
          sinks=(0.1, 0.0)),
    _case("max_nodes_321", 2, 128, [321, 50], ("tree6", "tree2"), act=TANH, attn_p=0.1),
    _case("max_nodes_352", 1, 192, [352, 351, 10], ("tree6", "tree2"), act=ELU, res=0, gsrc=(0.1, 0.1)),
    _case("385_nodes", 2, 64, [385, 40], ("chunk", "chunk"), act=ELU),
    _case("degree_5", 2, 128, [120, 61], ("chunk", "chunk"), act=LEAKY, deg5=True, gsrc=(0.0, 0.1)),
    _case("f96", 2, 96, [301, 45], ("chunk", "chunk"), act=TANH, sinks=(0.1, 0.2), out=False),
    _case("mean_heads", 3, 64, [301, 45], ("chunk", "chunk"), act=ELU, mean=True, sinks=(0.1,), gsrc=(0.1, 0.0),
          attn_p=0.1, holes=True),
    _case("three_gradient_sources", 2, 64, [301, 45], ("tree5", "chunk"), act=ELU, gsrc=(0.1, 0.0, 0.2)),
    _case("max_degree_unknown", 2, 64, [200, 45], ("chunk", "chunk"), act=NONE, max_degree=0),
    _case("f4_no_tree_descriptor", 1, 4, [90, 45], ("chunk", "chunk"), act=RELU, tree=False, gsrc=(0.1, 0.0, 0.0)),
    _case("f36_h8_mean", 8, 36, [90, 45], ("chunk", "chunk"), act=NONE, res=0, mean=True, tree=False, bias=False,
          gsrc=(0.0, 0.0, 0.1)),
    _case("b1_h8_f512_slice_split", 8, 512, [301], ("tree5", "chunk"), act=ELU, gsrc=(0.1,), fsplit="even"),
    _case("b1_h2_f64_head_split", 2, 64, [301], ("tree5", "tree2"), act=LEAKY, fsplit="even", bsplit=True),
    _case("uneven_slice_split", 4, 512, _uneven_batch, ("tree5", "tree2"), act=ELU, fsplit="uneven", bsplit=True,
          attn_p=0.1, sinks=(0.0,)),
    # B * H = #SMs (on 148 SMs) and the next batch up: one CTA per (tree, head), then one CTA per tree
    _case("per_head_split_on", 4, 64, lambda sms: [100 + i % 7 for i in range(sms // 4)], ("tree5", "tree2"),
          act=TANH, bsplit=True, gsrc=(0.1, 0.0)),
    _case("per_head_split_off", 4, 64, lambda sms: [100 + i % 7 for i in range(sms // 4 + 1)], ("tree5", "tree2"),
          act=TANH, bsplit=False, gsrc=(0.1, 0.0)),
    _case("grid_stride_sms_plus_1", 2, 64, lambda sms: [90 + i % 5 for i in range(sms + 1)], ("tree5", "tree2"),
          act=ELU, grid_stride=True, sinks=(0.1,)),
    _case("1000_small_trees", 1, 64, lambda sms: [1 + (i * 37) % 40 for i in range(1001)], ("tree5", "tree2"),
          act=RELU, grid_stride=True, attn_p=0.1),
    _case("tiny_trees", 2, 128, [1, 2, 31, 32, 33], ("tree5", "tree2"), act=LEAKY, gsrc=(0.1, 0.0), sinks=(0.2, 0.0)),
]


@pytest.mark.parametrize("c", LAYER_CASES)
def test_gat_layer_against_fp64(mods, c):
    """spgnn_gat_layer_fwd + _bwd on one case: att, out, the sinks (with their feat_drop masks), dY = [dz | G | d el |
    d er] and dbias against fp64, after checking the case is in the regime it claims and that exactly the launches of
    that regime ran."""
    run_layer_case(mods, c)


_VARIANT_SCRIPT = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import test_gpu_gat_layer_envelope as t
m = t._load_mods()
names = [sorted(t.run_layer_case(m, c, fvar=int(sys.argv[2]), bvar=int(sys.argv[3]))) for c in t.VARIANT_CASES]
print("KERNELS " + json.dumps(names))
"""

VARIANT_CASES = [
    dict(H=2, F=128, sizes=[301, 120], regime=("tree", "tree2"), act=ELU, gsrc=(0.1, 0.0), attn_p=0.1),
    dict(H=2, F=64, sizes=[384, 33], regime=("tree", "tree2"), act=TANH, sinks=(0.1,)),
]


@pytest.mark.parametrize("fwd_env,bwd_env", [("1", "1"), (None, "0"), (None, "9")])
def test_alternate_tree_launch_shapes_against_fp64(fwd_env, bwd_env):
    """SPGNN_TREE_FWD / SPGNN_TREE_BWD are read once per process, hence a subprocess per setting.  Two shapes, one with
    max_nodes <= 320 and one above, must match fp64 and run the 512- / 896-thread instantiations."""
    env = dict(os.environ, SPGNN_TREE_BWD=bwd_env)
    env.pop("SPGNN_TREE_FWD", None)
    if fwd_env:
        env["SPGNN_TREE_FWD"] = fwd_env
    fvar, bvar = int(fwd_env or 0), int(bwd_env)
    r = subprocess.run([sys.executable, "-c", _VARIANT_SCRIPT, ROOT, str(fvar), str(bvar)], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("KERNELS ")][-1]
    names = json.loads(line[len("KERNELS "):])
    threads = {"0": 512, "1": 896, "9": 640}[bwd_env]
    for case_names in names:
        assert any(n.startswith("gat_tree_bwd_kernel<") and f",{threads}," in n for n in case_names), case_names
        ft = 896 if fwd_env == "1" else 512
        assert any(n.startswith("gat_tree_fwd_kernel<") and f",{ft}," in n for n in case_names), case_names


# ------------------------------------------------------------------------------------------------ spgnn_gat_agg (gat.cu)
def run_agg_case(mods, H, F, res, xres_cols, mean, act, attn_p, bias):
    sg, ops, lib, ptr, stream = (mods[k] for k in ("sg", "ops", "lib", "ptr", "stream"))
    # trees of in-degree <= 4 (the fast kernel for H <= 2), one with up to 7 children (the general kernel) and nodes of
    # in-degree 0
    rng = np.random.default_rng(H * 100 + F)
    adjs = [_random_tree_adj(n, 2, rng) for n in (150, 61)] + [_random_tree_adj(40, 7, rng)]
    adjs[1], loops = _with_holes(adjs[1])
    g = _drop_self_loops(sg, sg.batch_from_adjs(adjs), [adjs[0].shape[0] + i for i in loops])
    N, E, HF = g.num_nodes, g.num_edges, H * F
    deg = g.in_degrees().cpu()
    assert int(deg.max()) >= 6 and int((deg == 0).sum()) == 3
    W = F if mean else HF
    Y, el_off, er_off = _random_y(N, H, F, res, seed=N + HF + res)
    Yd = Y.cuda()
    gen = torch.Generator().manual_seed(F + H)
    xres = torch.randn(N, xres_cols, generator=gen) if res == 2 else None
    xres_d = xres.cuda() if xres is not None else None
    b = (0.3 * torch.randn(HF, generator=gen)) if bias else None
    b_d = b.cuda() if b is not None else None
    out = torch.full((N, W), NAN, device="cuda")
    att = torch.full((E, H), NAN, device="cuda")
    seed = 31 + F
    res_args = (res, ptr(xres_d), xres_cols if res == 2 else 0, xres_cols if res == 2 else 0)
    gout = torch.randn(N, W, generator=gen)
    gout_d = gout.cuda()
    dY = torch.full((N, Yd.stride(0)), NAN, device="cuda")
    dxres = torch.full((N, xres_cols), NAN, device="cuda") if res == 2 else None
    g_ws = torch.full((N, HF), NAN, device="cuda") if res != 1 else None
    ds = torch.full((E * H,), NAN, device="cuda")
    torch.cuda.synchronize()

    def run():
        lib().gat_agg_fwd(ptr(Yd), Yd.stride(0), HF, el_off, er_off, res_args[0], res_args[1], res_args[2],
                          res_args[3], ptr(b_d), act, NEG_SLOPE, int(mean), attn_p, seed, ptr(g.in_ptr), ptr(g.in_src),
                          N, H, F, ptr(out), W, ptr(att), stream())
        lib().gat_agg_bwd(ptr(gout_d), W, ptr(out), W, ptr(Yd), Yd.stride(0), HF, el_off, er_off, res_args[0],
                          res_args[1], res_args[2], res_args[3], ptr(b_d), act, NEG_SLOPE, int(mean), attn_p, seed,
                          ptr(att), ptr(g.in_ptr), ptr(g.in_src), ptr(g.out_ptr), ptr(g.out_dst), ptr(g.out_slot), N, H,
                          F, ptr(dY), ptr(dxres), ptr(g_ws), ptr(ds), stream())

    names = _profiled(run)
    nch = 1 if F <= 128 else 2 if F <= 256 else 4 if F <= 512 else 8
    want = {"gat_agg_fwd_kernel", f"gat_agg_bwd_dst_kernel<{nch}>", "gat_agg_bwd_src_kernel"}
    if H <= 2:
        want |= {f"gat_fast_kernel<{H},{w}>" for w in range(3)}
    assert names == want, (sorted(names), sorted(want))

    keep = ops.drop_mask(E, H, attn_p, seed, "cuda").cpu().double() if attn_p > 0 else None
    branch = (out.cpu() > 0).view(N, H, F) if act in (RELU, LEAKY) else None
    ref = gat_ref64(g, Y, H, F, res, el_off, er_off, b, act, mean, keep, gout.double(), branch, xres)
    assert rel_err(att.cpu(), ref["att"]) < TOL, "att"
    assert rel_err(out.cpu(), ref["out"]) < TOL, "out"
    dYc = dY.cpu()
    assert rel_err(dYc[:, :HF], ref["dz"]) < TOL, "dz"
    if res == 1:
        assert rel_err(dYc[:, HF:2 * HF], ref["G"]) < TOL, "G (residual part of dY)"
    else:
        assert rel_err(g_ws.cpu(), ref["G"]) < TOL, "G (g_ws)"
    assert rel_err(dYc[:, el_off:el_off + H], ref["del_"]) < TOL, "d el"
    assert rel_err(dYc[:, er_off:er_off + H], ref["der"]) < TOL, "d er"
    if res == 2:
        assert rel_err(dxres.cpu(), ref["dxres"]) < TOL, "dxres"
    return names


# (H, F, res_mode, xres_cols, mean_heads, act, attn_p, bias): F covers every backward bucket (<= 128 / 256 / 512 /
# 1024) and both sides of each boundary; identity residuals with F columns (broadcast over the heads, DGL 0.7) and
# with H*F columns
AGG_CASES = [
    (1, 4, 0, 0, False, ELU, 0.0, True),
    (2, 128, 1, 0, False, LEAKY, 0.1, True),
    (2, 132, 2, 132, True, TANH, 0.0, True),
    (3, 256, 2, 768, False, RELU, 0.1, True),
    (8, 260, 0, 0, True, NONE, 0.2, False),
    (1, 512, 2, 512, False, LEAKY, 0.0, True),
    (2, 516, 1, 0, False, ELU, 0.1, False),
    (3, 1024, 2, 1024, True, ELU, 0.0, True),
    (8, 128, 2, 1024, False, TANH, 0.1, True),
    (1, 1024, 0, 0, False, RELU, 0.2, True),
    (2, 64, 2, 128, True, NONE, 0.1, True),
]


@pytest.mark.parametrize("H,F,res,xres_cols,mean,act,attn_p,bias", AGG_CASES)
def test_gat_agg_against_fp64(mods, H, F, res, xres_cols, mean, act, attn_p, bias):
    """spgnn_gat_agg_fwd + _bwd: att, out, dY = [dz | G | d el | d er], G and dxres against fp64, with the fast
    kernel (H <= 2, in-degree 1-4) next to the general kernel and the backward bucket F implies."""
    run_agg_case(mods, H, F, res, xres_cols, mean, act, attn_p, bias)


def test_gat_agg_backward_refuses_f_above_1024_before_any_launch(mods):
    """F = 1028 runs forward; the backward raises SpgnnError and writes nothing."""
    sg, lib, ptr, stream = (mods[k] for k in ("sg", "lib", "ptr", "stream"))
    H, F = 1, 1028
    g = sg.batch_from_adjs([_random_tree_adj(40, 2, np.random.default_rng(0))])
    N, E = g.num_nodes, g.num_edges
    Y, el_off, er_off = _random_y(N, H, F, 0, seed=1)
    Yd = Y.cuda()
    out = torch.full((N, F), NAN, device="cuda")
    att = torch.full((E, H), NAN, device="cuda")
    lib().gat_agg_fwd(ptr(Yd), Yd.stride(0), F, el_off, er_off, 0, None, 0, 0, None, ELU, NEG_SLOPE, 0, 0.0, 0,
                      ptr(g.in_ptr), ptr(g.in_src), N, H, F, ptr(out), F, ptr(att), stream())
    torch.cuda.synchronize()
    assert not torch.isnan(out).any()
    gout = torch.randn(N, F, device="cuda")
    dY = torch.full((N, Yd.stride(0)), NAN, device="cuda")
    g_ws = torch.full((N, F), NAN, device="cuda")
    ds = torch.full((E,), NAN, device="cuda")
    with pytest.raises(mods["SpgnnError"], match="exceeds"):
        lib().gat_agg_bwd(ptr(gout), F, ptr(out), F, ptr(Yd), Yd.stride(0), F, el_off, er_off, 0, None, 0, 0, None,
                          ELU, NEG_SLOPE, 0, 0.0, 0, ptr(att), ptr(g.in_ptr), ptr(g.in_src), ptr(g.out_ptr),
                          ptr(g.out_dst), ptr(g.out_slot), N, H, F, ptr(dY), None, ptr(g_ws), ptr(ds), stream())
    torch.cuda.synchronize()
    assert torch.isnan(dY).all() and torch.isnan(g_ws).all() and torch.isnan(ds).all()


# ------------------------------------------------------------------------------------------------ nn.GATConv
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("act", ["leaky_relu", "relu"])
@pytest.mark.parametrize("path", ["per_layer", "aggregate_first"])
def test_gatconv_runtime_activations_vs_oracle(mods, path, act, train):
    """nn.GATConv(activation=F.leaky_relu or torch.relu) against oracle.dgl_ops.GATConv in fp64: forward and every
    parameter gradient, on the per-layer path (forward_flat) and as the aggregate-first output layer of a hand-wired
    StackPlan.  The loss weights are 0 at the few outputs whose fp64 pre-activation lies within 1e-4 of the kink, so
    the fp32 / fp64 branch choice there does not matter; the attention logits' branches and the dropout masks are
    replayed from the device."""
    ops, stack, snn, dgl, sg = (mods[k] for k in ("ops", "stack", "snn", "dgl_ops", "sg"))
    fn = {"leaky_relu": torch.nn.functional.leaky_relu, "relu": torch.relu}[act]
    rng = np.random.default_rng(3)
    adjs = [_random_tree_adj(n, 2, rng) for n in (140, 77, 301)]
    g = sg.batch_from_adjs(adjs)
    og = dgl.batch([dgl.graph_from_adj(a) for a in adjs])
    N = g.num_nodes
    k_in, H, F = (64, 2, 128) if path == "aggregate_first" else (48, 2, 64)
    torch.manual_seed(0)
    oconv = dgl.GATConv(k_in, F, H, feat_drop=0.1, attn_drop=0.2, negative_slope=0.2, residual=True, activation=fn)
    with torch.no_grad():
        oconv.bias.normal_(0, 0.3)
    conv = snn.GATConv(k_in, F, H, 0.1, 0.2, 0.2, residual=True, activation=fn).cuda()
    conv.load_state_dict(oconv.state_dict())
    conv.train(train)
    oconv.train(train)
    x = torch.randn(N, k_in)
    ops.manual_seed(11)
    if path == "per_layer":
        out, rec = traced(ops, lambda: conv(g, x.cuda()).reshape(N, H * F))
    else:
        L = stack.LayerPlan(conv, ["x"], "emb", mean_heads=True)
        plan = stack.StackPlan([L], {"x": k_in}, ["emb"])
        assert L.wide, "the layer should be planned aggregate-first"
        out, rec = traced(ops, lambda: stack.run_stack(plan, g, {"x": x.cuda()}, train)[1][0])
    o64 = copy.deepcopy(oconv).double()
    o64.train(train)
    x64 = x.double()
    o64.activation = None
    pre, _ = replay(rec, lambda: o64(og, x64))
    pre = pre.detach()
    o64.activation = fn
    near = pre.abs() < 1e-4 * pre.abs().max()
    gw = torch.randn(out.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(5))
    gw[near.reshape(N, H * F) if path == "per_layer" else near.any(1)] = 0.0
    ref_fwd = fn(pre)
    ref_fwd = ref_fwd.reshape(N, H * F) if path == "per_layer" else ref_fwd.mean(1)
    assert rel_err(out.detach().cpu(), ref_fwd) < 1e-4, "forward"
    (out * gw.float().cuda()).sum().backward()
    y64, _ = replay(rec, lambda: o64(og, x64))
    y64 = y64.reshape(N, H * F) if path == "per_layer" else y64.mean(1)
    (y64 * gw).sum().backward()
    assert_grads_match(conv, o64, TRAIN_GRAD_TOL if train else GRAD_TOL, (path, act, train))
