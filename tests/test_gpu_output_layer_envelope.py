"""The aggregate-first output layer (spgnn_gat_aggx_fwd / _bwd + spgnn_wide_linear) over everything its entry points
accept, not just the H = 2, F = 1024, k_in in {128, 192} of the shipped presets: H in {1, 2, 4}, F % 32 == 0 up to
H*F = 8192 (ragged last n-tile), k_in < kp (padding inside every 64-column block of XA), a ragged second source,
activation NONE / ELU / the generic branch, 1..3 gradient sources, either output alone and no bias.  References are
fp64 on the CPU: the wide GEMM against its formula, aggx_fwd against an fp64 edge softmax, and whole nets against the
fp64 oracle with the device's kinks replayed."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import assert_grads_match, oracle_fp64, rel_err, replay, traced
from test_gpu_parity import (GRAD_TOL, NET_CLS, TOL, TRAIN_GRAD_TOL, _device_batch, _oracle_batch, _random_tree_adj,
                             _scans_on)

pytestmark = pytest.mark.gpu

SMS = 148
ACT_NONE, ACT_ELU, ACT_TANH = 0, 1, 2          # tanh takes the generic wide_act<-1> branch of the epilogue
GEMM_TOL = 4e-5                                # split-bf16 planes GEMMs vs fp64 (test_linear_fwd_bwd_against_fp64)


@pytest.fixture(scope="module")
def mods():
    from oracle import dgl_ops, models as om, pe as ope
    from spgnn_b200 import graph as sg, models as sm, ops, stack
    return dict(dgl_ops=dgl_ops, om=om, ope=ope, sg=sg, sm=sm, ops=ops, stack=stack)


def _act64(x, act):
    return {ACT_NONE: x, ACT_ELU: torch.nn.functional.elu(x), ACT_TANH: torch.tanh(x)}[act]


def _act_grad64(x, act):
    if act == ACT_NONE:
        return torch.ones_like(x)
    if act == ACT_ELU:
        return torch.where(x > 0, torch.ones_like(x), torch.exp(x))
    return 1.0 - torch.tanh(x) ** 2


def _pad4(n):
    return (n + 3) // 4 * 4


def wide_operands(stack, M, H, F, k_in, has_res, seed):
    """XA planes [M, (H+1)*kp] built from fp32 data with zero padding columns (the aggx_fwd contract), the packed
    weight [(1+has_res)*H*F, k_in] (16-byte aligned rows) and a bias [H*F]."""
    kp = (k_in + 63) // 64 * 64
    gen = torch.Generator().manual_seed(seed)
    xa = torch.zeros(M, (H + 1) * kp)
    for h in range(H + 1):
        xa[:, h * kp:h * kp + k_in] = torch.randn(M, k_in, generator=gen)
    XA = stack.split_planes(xa.cuda())
    rows = (1 + has_res) * H * F
    W = torch.empty(rows, _pad4(k_in), device="cuda")[:, :k_in]
    W.copy_(torch.randn(rows, k_in, generator=gen) / (k_in * (1 + has_res)) ** 0.5)
    b = (0.3 * torch.randn(H * F, generator=gen)).cuda()
    return XA, kp, W, b


def wide_pre64(XA, kp, W, b, M, H, F, k_in, has_res):
    """fp64 pre-activations [H, M, F] from exactly the values the kernel reads (the planes' hi + lo)."""
    xa = XA.float().double().cpu()
    W64 = W.double().cpu()
    x = xa[:, H * kp:H * kp + k_in]
    pre = []
    for h in range(H):
        p = xa[:, h * kp:h * kp + k_in] @ W64[h * F:(h + 1) * F].t()
        if has_res:
            p += x @ W64[H * F + h * F:H * F + (h + 1) * F].t()
        if b is not None:
            p += b[h * F:(h + 1) * F].double().cpu()
        pre.append(p)
    return torch.stack(pre)


def run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, mode, out_fp32=True, out_planes=True, grads=()):
    """One spgnn_wide_linear call; returns (out fp32 or None, out planes or None) in mode 0, (dpre planes, dbias or
    None) in mode 1."""
    from spgnn_b200._lib import lib, ptr, stream
    L = lib()
    ws = torch.empty(int(L.wide_linear_ws(H, F, kp, has_res)), dtype=torch.uint8, device="cuda")
    if mode == 0:
        out = torch.full((M, F), float("nan"), device="cuda") if out_fp32 else None
        P = stack.Planes(M, F, "cuda") if out_planes else None
        L.wide_linear(XA.ptr(), XA.ld, XA.ps, kp, k_in, M, H, F, has_res, ptr(W), W.stride(0), ptr(b), act, 0,
                      ptr(out), F if out is not None else 0, P.ptr() if P is not None else None,
                      P.ld if P is not None else 0, P.ps if P is not None else 0,
                      None, 0, None, 0, None, 0, None, 0, 0, None, ptr(ws), ws.numel(), stream())
        return out, P
    gp = [(ptr(g), g.stride(0)) for g in grads] + [(None, 0)] * (3 - len(grads))
    dpre = stack.Planes(M, H * F, "cuda")
    db = torch.full((H * F,), float("nan"), device="cuda") if b is not None else None
    L.wide_linear(XA.ptr(), XA.ld, XA.ps, kp, k_in, M, H, F, has_res, ptr(W), W.stride(0), ptr(b), act, 1,
                  None, 0, None, 0, 0, gp[0][0], gp[0][1], gp[1][0], gp[1][1], gp[2][0], gp[2][1],
                  dpre.ptr(), dpre.ld, dpre.ps, ptr(db), ptr(ws), ws.numel(), stream())
    return dpre, db


# (H, F, k_in, has_res, act, M, outputs of mode 0, gradient sources of mode 1, bias): every value of every axis at
# least once; F = 288 leaves a ragged last n-tile at every H (BN = 256 / H), M = 40 001 gives more tiles than CTAs
WIDE_CASES = [
    (1, 32, 64, 0, ACT_ELU, 1, "both", 1, True),
    (2, 288, 100, 1, ACT_NONE, 127, "fp32", 2, True),
    (4, 96, 232, 1, ACT_TANH, 129, "planes", 3, False),
    (1, 1024, 192, 1, ACT_TANH, 40001, "both", 3, True),
    (2, 1024, 232, 0, ACT_ELU, 40001, "fp32", 1, False),
    (4, 2048, 64, 1, ACT_ELU, 129, "both", 2, True),           # H*F = 8192
    (2, 4096, 100, 0, ACT_NONE, 127, "planes", 1, True),       # H*F = 8192
    (1, 8192, 232, 1, ACT_ELU, 1, "fp32", 3, True),            # H*F = 8192
    (4, 288, 192, 0, ACT_ELU, 40001, "both", 2, True),
    (2, 96, 64, 1, ACT_TANH, 40001, "planes", 1, False),
    (4, 32, 100, 0, ACT_NONE, 1, "both", 3, False),
    (1, 288, 64, 1, ACT_NONE, 40001, "fp32", 2, True),
]


@pytest.mark.parametrize("H,F,k_in,has_res,act,M,outs,n_g,bias", WIDE_CASES)
def test_wide_linear_against_fp64(mods, H, F, k_in, has_res, act, M, outs, n_g, bias):
    """Mode 0: out = mean_h act(A_h W_fc,h^T + [x W_res,h^T] + b_h) into the fp32 output, the planes output or both.
    Mode 1: dpre_h = (sum_s g_s / H) * act'(pre_h) as planes and dbias = column sums of dpre.  Both against fp64."""
    stack = mods["stack"]
    XA, kp, W, b = wide_operands(stack, M, H, F, k_in, has_res, seed=M * 7 + H * F + k_in)
    b = b if bias else None
    BN = min(256 // H, F)
    tiles = -(-M // 128) * -(-F // BN)
    if M > 40000:
        assert tiles > SMS, "both TMEM accumulator buffers should wrap"
    if F == 288:
        assert F % BN != 0, "the last n-tile should be ragged"
    pre = wide_pre64(XA, kp, W, b, M, H, F, k_in, has_res)
    ref = _act64(pre, act).mean(0)

    out, P = run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, 0, out_fp32=outs != "planes",
                      out_planes=outs != "fp32")
    assert (out is None) == (outs == "planes") and (P is None) == (outs == "fp32")
    if out is not None:
        assert rel_err(out.cpu(), ref) < GEMM_TOL, "mode 0, fp32 output"
    if P is not None:
        assert rel_err(P.float().cpu(), ref) < GEMM_TOL, "mode 0, planes output"

    gen = torch.Generator().manual_seed(M + n_g)
    grads = [torch.randn(M, F, generator=gen) for _ in range(n_g)]
    dpre, db = run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, 1, grads=[g.cuda() for g in grads])
    gsum = torch.stack(grads).double().sum(0) / H
    dref = torch.cat([gsum * _act_grad64(pre[h], act) for h in range(H)], 1)
    assert rel_err(dpre.float().cpu(), dref) < GEMM_TOL, "mode 1, dpre"
    if b is not None:
        assert rel_err(db.cpu(), dref.sum(0)) < GEMM_TOL, "mode 1, dbias"


# ------------------------------------------------------------------------------------------------ aggx_fwd
def _wide_graph(sg, rng, n_trees):
    """Trees with up to six children (in-degree up to 8 with the self loop: both the <= 4 and the general branch of
    the aggregation kernels) as one batch."""
    adjs = [_random_tree_adj(int(n), 6, rng) for n in rng.integers(40, 300, n_trees)]
    return sg.batch_from_adjs(adjs)


@pytest.mark.parametrize("H,K1,K2", [(1, 64, 20), (2, 128, 39), (4, 64, 0), (4, 192, 40)])
def test_aggx_forward_pads_xa_with_zeros_and_aggregates_in_fp64(mods, H, K1, K2):
    """spgnn_gat_aggx_fwd into an XA buffer filled with NaN: every padding column [k_in, kp) of every block is exactly
    0 in both planes (spgnn_wide_linear relies on it), block H is x, and every A_h = sum_u a[u->v, h] x[u] with a the
    fp64 edge softmax of LeakyReLU(el[u] + er[v]).  el / er are drawn at least 0.7 away from the kink."""
    from spgnn_b200._lib import lib, ptr, stream
    stack, sg = mods["stack"], mods["sg"]
    rng = np.random.default_rng(H * 100 + K1 + K2)
    g = _wide_graph(sg, rng, 12)
    N, E = g.num_nodes, g.num_edges
    assert g.max_degree() > 4
    k_in = K1 + K2
    kp = (k_in + 63) // 64 * 64
    gen = torch.Generator().manual_seed(K1 + K2)
    X1 = stack.split_planes(torch.randn(N, K1, generator=gen).cuda())
    X2 = stack.split_planes(torch.randn(N, K2, generator=gen).cuda()) if K2 else None
    sign = torch.where(torch.rand(N, H, generator=gen) < 0.5, -1.0, 1.0)
    el = sign * (1.0 + torch.rand(N, H, generator=gen))
    er = 0.6 * torch.rand(N, H, generator=gen) - 0.3
    eler = torch.cat([el, er], 1).cuda()
    XA = stack.Planes(N, (H + 1) * kp, "cuda")
    XA.buf.fill_(float("nan"))
    att = torch.empty(E, H, device="cuda")
    d = stack._Wide()
    d.in_ptr, d.in_src = ptr(g.in_ptr), ptr(g.in_src)
    d.out_ptr, d.out_dst, d.out_slot = ptr(g.out_ptr), ptr(g.out_dst), ptr(g.out_slot)
    d.N, d.H, d.has_res = N, H, 1
    d.X1, d.ldx1, d.psx1, d.K1 = X1.ptr(), X1.ld, X1.ps, K1
    if X2 is not None:
        d.X2, d.ldx2, d.psx2, d.K2 = X2.ptr(), X2.ld, X2.ps, K2
    d.eler, d.ld_eler = ptr(eler), eler.stride(0)
    d.negative_slope, d.attn_drop_p, d.attn_seed = 0.2, 0.0, 0
    d.att = ptr(att)
    d.XA, d.ldxa, d.psxa, d.kp = XA.ptr(), XA.ld, XA.ps, kp
    lib().gat_aggx_fwd(ctypes.byref(d), stream())
    torch.cuda.synchronize()

    buf = XA.buf.cpu()
    for h in range(H + 1):
        pad = buf[:, :, h * kp + k_in:(h + 1) * kp]
        assert torch.equal(pad, torch.zeros_like(pad)), f"padding of block {h} is not zero"
    xa = XA.float().cpu()
    assert not torch.isnan(xa).any()
    x = torch.cat([X1.float()] + ([X2.float()] if X2 is not None else []), 1).double().cpu()
    assert rel_err(xa[:, H * kp:H * kp + k_in], x) < 1e-6
    # fp64 edge softmax over the in-CSC
    in_ptr, in_src = g.in_ptr.long().cpu(), g.in_src.long().cpu()
    dst = torch.repeat_interleave(torch.arange(N), in_ptr[1:] - in_ptr[:-1])
    e = torch.nn.functional.leaky_relu(el.double()[in_src] + er.double()[dst], 0.2)
    m = torch.full((N, H), -torch.inf, dtype=torch.float64).scatter_reduce(0, dst[:, None].expand(-1, H), e, "amax")
    p = torch.exp(e - m[dst])
    a = p / torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, p)[dst]
    assert rel_err(att.cpu(), a) < 1e-5
    for h in range(H):
        A = torch.zeros(N, k_in, dtype=torch.float64).index_add(0, dst, a[:, h:h + 1] * x[in_src])
        assert rel_err(xa[:, h * kp:h * kp + k_in], A) < 2e-5, h


# ------------------------------------------------------------------------------------------------ whole nets
NETS = {
    # GAT, one output head, residual projection: k_in = 64, H*F = 256
    "gat_h1_res": ("gat", dict(out_ch=22, fv_dim=128, num_gat_layers=3, num_heads=2, num_out_heads=1, feat_drop=0.1,
                               attn_drop=0.1, negative_slope=0.2, num_hiddens=[64, 48, 32], node_embed_dim=256)),
    # GAT, four output heads, no residual: k_in = 64, H*F = 512
    "gat_h4_nores": ("gat", dict(out_ch=22, fv_dim=128, num_gat_layers=3, num_heads=2, num_out_heads=4, feat_drop=0.1,
                                 attn_drop=0.1, negative_slope=0.2, num_hiddens=[64, 48, 32], node_embed_dim=128,
                                 res=False)),
    # SPGNN, four output heads, ragged second source: k_in = 64 + 20 = 84, kp = 128, H*F = 384
    "spgnn_h4_ragged": ("spgnn", dict(out_ch=22, fv_dim=128, num_gat_layers=3, num_heads=2, num_out_heads=4,
                                      feat_drop=0.1, attn_drop=0.1, negative_slope=0.2, num_hiddens=[64, 48, 32],
                                      pos_hiddens=[32, 24, 20], num_pos_heads=1, pos_enc_dim=39, node_embed_dim=96)),
    # SPGNN, one output head, no residual, ragged second source: k_in = 84, H*F = 352
    "spgnn_h1_ragged_nores": ("spgnn", dict(out_ch=22, fv_dim=128, num_gat_layers=3, num_heads=2, num_out_heads=1,
                                            feat_drop=0.1, attn_drop=0.1, negative_slope=0.2, num_hiddens=[64, 48, 32],
                                            pos_hiddens=[32, 24, 20], num_pos_heads=1, pos_enc_dim=39,
                                            node_embed_dim=352, res=False)),
    # st_gat_3 with eight hidden heads and four output heads: k_in = 512, H*F = 4096 (the backward's logit-weight
    # stage is 52 KB, above the 48 KB a launch gets without opting in)
    "st_gat_3_h8_out4": ("gat", dict(out_ch=22, fv_dim=1024, num_gat_layers=3, num_heads=8, num_out_heads=4,
                                     feat_drop=0.1, attn_drop=0.1, negative_slope=0.2, num_hiddens=[256, 128, 64],
                                     node_embed_dim=1024)),
}


def _net_pair(mods, kind, cfg, train):
    torch.manual_seed(0)
    onet = mods["om"].GNNNet(kind, cfg)
    onet.init_like_reference()
    with torch.no_grad():
        for k, p in onet.named_parameters():
            if k.endswith("bias"):
                p.normal_(0, 0.05)
    net = getattr(mods["sm"], NET_CLS[kind])(**cfg).cuda()
    net.load_state_dict(onet.state_dict(), strict=True)
    onet.train(train)
    net.train(train)
    if train:               # the output layer has no attention dropout of its own in these nets: give it some
        dict(net.named_modules())["gat.gat_layers.3"].attn_drop_p = 0.2
        dict(onet.named_modules())["gat.gat_layers.3"].attn_drop.p = 0.2
    return onet, net


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("name", sorted(NETS))
def test_aggregate_first_nets_outside_the_shipped_widths_vs_oracle(mods, name, train, monkeypatch):
    """Forward, loss and every parameter gradient of nets whose output layer is aggregate-first at widths no preset
    uses, against the fp64 oracle with the device's LeakyReLU branches and dropout masks replayed, and against the
    same net with the output layer projection-first (same seeds: same masks)."""
    ops, stack = mods["ops"], mods["stack"]
    kind, cfg = NETS[name]
    rng = np.random.default_rng(23)
    adjs = [_random_tree_adj(int(n), 3, rng) for n in (140, 60, 95, 33)]
    scans = _scans_on(adjs, rng)
    if cfg["fv_dim"] != 1024:
        for s in scans:
            s["fvs"] = np.ascontiguousarray(s["fvs"][:, :cfg["fv_dim"]])
    onet, net = _net_pair(mods, kind, cfg, train)
    plan = net.gat._stack_plan()
    out_layer = plan.layers[-1]
    assert out_layer.wide, f"{name}: the output layer should be planned aggregate-first"
    assert out_layer.H == cfg["num_out_heads"] and out_layer.res_mode == (1 if cfg.get("res", True) else 0)
    pos = None
    if kind == "spgnn":
        pos = [mods["ope"].dist_pos_enc(s["adj"], mods["ope"].anchors_39(s["fvs_out"], s["adj"]))[0] for s in scans]
        assert out_layer.k_in == 84 and len(out_layer.inputs) == 2
    og = _oracle_batch(mods, scans, pos)
    g = _device_batch(mods, scans, np.concatenate(pos) if pos is not None else None)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]))
    cw = torch.tensor([0.2] + [0.8] * 21)
    mask = torch.ones(y.numel(), dtype=torch.bool)

    ops.manual_seed(5)
    out, rec = traced(ops, lambda: net(g))
    loss = ops.masked_cross_entropy(out[0], y.cuda(), cw.cuda(), mask=mask.cuda())
    loss.backward()
    ref, tape = replay(rec, lambda: onet(og))
    loss_ref = mods["om"].cross_entropy_masked(ref[0], y, mask, cw)
    onet64, og64 = oracle_fp64(onet, og)
    ref64, _ = replay(rec, lambda: onet64(og64))
    mods["om"].cross_entropy_masked(ref64[0], y, mask, cw.double()).backward()
    if train:
        assert sum(k == "drop" for k, _ in rec) >= 3
    for j in range(len(ref)):
        assert rel_err(out[j].detach().cpu(), ref[j].detach()) < TOL, (name, j)
    assert abs(loss.item() - loss_ref.item()) < TOL * abs(loss_ref.item())
    assert_grads_match(net, onet64, TRAIN_GRAD_TOL if train else GRAD_TOL,
                       (name, f"{tape.flips} of {tape.decisions} decisions pinned"))

    wide_grads = {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None}
    monkeypatch.setattr(stack, "WIDE_OUTPUT_LAYER", False)
    net.zero_grad(set_to_none=True)
    ops.manual_seed(5)
    out2 = net(g)
    ops.masked_cross_entropy(out2[0], y.cuda(), cw.cuda(), mask=mask.cuda()).backward()
    for a, b in zip(out, out2):
        assert rel_err(a.detach().cpu(), b.detach().cpu()) < 2e-5, name
    gmax = max(float(v.abs().max()) for v in wide_grads.values())
    for k, p in net.named_parameters():
        if p.grad is None:
            assert k not in wide_grads, k
            continue
        err = float((wide_grads[k].double() - p.grad.double()).abs().max())
        assert err <= 5e-5 * float(p.grad.abs().max()) or err <= 1e-6 * gmax, (name, k, err)

