"""The output layer's saved derivative: spgnn_wide_linear_fwd_dact (mode 0 that also keeps act'(pre) of every head)
and spgnn_wide_dpre (the pre-activation gradient built from the head's output gradient and that saved derivative,
without recomputing the wide GEMM).  Kernel level: the forward's outputs equal plain mode 0 bit for bit, dact equals
the act' mode 1 recomputes bit for bit, and dpre / dbias equal mode 1 fed the head's fp32 dX and an fp64 reference.
Net level: train-step gradients with stack.WIDE_SAVED_DACT on and off agree, and nothing extra is kept in eval."""
import numpy as np
import pytest
import torch

from helpers import FULL_MODELS, rel_err
from test_gpu_output_layer_envelope import (ACT_ELU, ACT_NONE, ACT_TANH, GEMM_TOL, _act64, _act_grad64, run_wide,
                                            wide_operands, wide_pre64)
from test_gpu_parity import NET_CLS, _device_batch, _scan_dicts

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    from oracle import pe as ope
    from spgnn_b200 import graph as sg, models as sm, ops, stack, synth
    return dict(ope=ope, sg=sg, sm=sm, ops=ops, stack=stack, synth=synth)


def run_fwd_dact(stack, XA, kp, k_in, M, H, F, has_res, W, b, act):
    from spgnn_b200._lib import lib, ptr, stream
    L = lib()
    ws = torch.empty(int(L.wide_linear_ws(H, F, kp, has_res)), dtype=torch.uint8, device="cuda")
    out = torch.full((M, F), float("nan"), device="cuda")
    P = stack.Planes(M, F, "cuda")
    dact = torch.full((M, H * F), float("nan"), device="cuda")
    L.wide_linear_fwd_dact(XA.ptr(), XA.ld, XA.ps, kp, k_in, M, H, F, has_res, ptr(W), W.stride(0), ptr(b), act,
                           ptr(out), F, P.ptr(), P.ld, P.ps, ptr(dact), dact.stride(0), ptr(ws), ws.numel(), stream())
    return out, P, dact


def run_dpre(stack, glp, Wh, dact, M, H, F, extras, with_bias):
    from spgnn_b200._lib import lib, ptr, stream
    L = lib()
    ws = torch.empty(int(L.wide_dpre_ws(H, F)), dtype=torch.uint8, device="cuda")
    gp = [(ptr(g), g.stride(0)) for g in extras] + [(None, 0)] * (2 - len(extras))
    dpre = stack.Planes(M, H * F, "cuda")
    db = torch.full((H * F,), float("nan"), device="cuda") if with_bias else None
    L.wide_dpre(glp.ptr(), glp.ld, glp.ps, glp.cols, M, H, F, ptr(Wh), Wh.stride(0), ptr(dact), dact.stride(0),
                gp[0][0], gp[0][1], gp[1][0], gp[1][1], dpre.ptr(), dpre.ld, dpre.ps, ptr(db), ptr(ws), ws.numel(),
                stream())
    return dpre, db


# (H, F, k_in, has_res, act, M, extra fp32 sources besides the head, head outputs C, bias): every H, F, act and
# source count at least once, M never a multiple of 128, M = 40 001 wraps both TMEM buffers
CASES = [
    (1, 32, 64, 0, ACT_ELU, 1, 0, 22, True),
    (2, 96, 100, 1, ACT_NONE, 127, 1, 22, True),
    (4, 1024, 192, 1, ACT_TANH, 129, 2, 22, True),
    (2, 1024, 192, 1, ACT_ELU, 40001, 0, 22, True),          # the shipped output layer
    (4, 32, 232, 0, ACT_NONE, 40001, 2, 5, False),
    (1, 1024, 64, 1, ACT_TANH, 40001, 1, 64, True),
    (4, 96, 100, 0, ACT_ELU, 1000, 1, 22, True),
    (1, 96, 192, 1, ACT_ELU, 255, 2, 22, False),
    (2, 32, 64, 0, ACT_TANH, 3, 0, 22, True),
]


@pytest.mark.parametrize("H,F,k_in,has_res,act,M,n_extra,C,bias", CASES)
def test_saved_derivative_and_dpre_from_the_head(mods, H, F, k_in, has_res, act, M, n_extra, C, bias):
    stack = mods["stack"]
    XA, kp, W, b = wide_operands(stack, M, H, F, k_in, has_res, seed=M * 5 + H * F + k_in)
    b = b if bias else None
    HF = H * F

    # forward: outputs bit-identical to plain mode 0, dact bit-identical to the act' of mode 1
    out0, P0 = run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, 0)
    out, P, dact = run_fwd_dact(stack, XA, kp, k_in, M, H, F, has_res, W, b, act)
    torch.cuda.synchronize()
    assert torch.equal(out, out0), "fp32 output differs from mode 0"
    assert torch.equal(P.buf[:, :, :F], P0.buf[:, :, :F]), "planes output differs from mode 0"
    ones = torch.full((M, F), float(H), device="cuda")         # g / H = 1 exactly: mode 1 writes act' itself
    grad1, _ = run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, 1, grads=[ones])
    assert torch.equal(stack.split_planes(dact).buf[:, :, :HF], grad1.buf[:, :, :HF]), "dact differs from mode 1"
    pre = wide_pre64(XA, kp, W, b, M, H, F, k_in, has_res)
    dact_ref = torch.cat([_act_grad64(pre[h], act) for h in range(H)], 1)
    assert rel_err(dact.cpu(), dact_ref) < GEMM_TOL
    assert rel_err(out.cpu(), _act64(pre, act).mean(0)) < GEMM_TOL

    # backward: dpre / dbias from the head's output gradient against mode 1 fed the head's fp32 dX, and fp64
    gen = torch.Generator().manual_seed(M + C + n_extra)
    gl = torch.randn(M, C, generator=gen)
    Wh = torch.randn(C, F, generator=gen) / C ** 0.5
    extras = [torch.randn(M, F, generator=gen) for _ in range(n_extra)]
    glp = stack.split_planes(gl.cuda())
    Whd = Wh.cuda()
    head_dx = stack.planes_linear_bwd_input(glp, Whd, F)
    dpre1, db1 = run_wide(stack, XA, kp, k_in, M, H, F, has_res, W, b, act, 1,
                          grads=[e.cuda() for e in extras] + [head_dx])
    dpre2, db2 = run_dpre(stack, glp, Whd, dact, M, H, F, [e.cuda() for e in extras], b is not None)
    torch.cuda.synchronize()
    d1, d2 = dpre1.float().cpu(), dpre2.float().cpu()
    assert rel_err(d2, d1) < 1e-6, "dpre differs from mode 1 beyond fp32 rounding of the head's dX"
    g64 = (torch.stack(extras).double().sum(0) if extras else 0.0) + glp.float().double().cpu() @ Wh.double()
    dref = torch.cat([g64 / H * _act_grad64(pre[h], act) for h in range(H)], 1)
    assert rel_err(d2, dref) < GEMM_TOL, "dpre against fp64"
    if b is not None:
        assert rel_err(db2.cpu(), db1.cpu()) < 1e-5, "dbias differs from mode 1"
        assert rel_err(db2.cpu(), dref.sum(0)) < GEMM_TOL, "dbias against fp64"
    else:
        assert db2 is None


def test_dpre_rejects_a_head_wider_than_one_k_block(mods):
    from spgnn_b200._lib import SpgnnError
    stack = mods["stack"]
    M, H, F, C = 130, 2, 32, 65
    glp = stack.split_planes(torch.randn(M, C).cuda())
    dact = torch.ones(M, H * F, device="cuda")
    with pytest.raises(SpgnnError, match="1..64 outputs"):
        run_dpre(stack, glp, torch.randn(C, F).cuda(), dact, M, H, F, [], False)


def _net_step(mods, net, g, y, cw, with_emb):
    mods["ops"].manual_seed(11)
    net.zero_grad()
    out = net(g)
    loss = mods["ops"].masked_cross_entropy(out[0], y, cw, mask=torch.ones_like(y, dtype=torch.bool))
    if with_emb:
        loss = loss + 1e-3 * out[1].square().mean()       # a second gradient source on the output layer
    loss.backward()
    return [o.detach().clone() for o in out], {k: p.grad.clone() for k, p in net.named_parameters()
                                               if p.grad is not None}


@pytest.mark.parametrize("name", ["st_gat_3", "st_pgat_spgnn_3"])
@pytest.mark.parametrize("with_emb", [False, True])
def test_train_step_with_and_without_the_saved_derivative(mods, name, with_emb, monkeypatch):
    """The same train-mode step (dropout on, attention dropout on the output layer) with stack.WIDE_SAVED_DACT on and
    off: outputs identical, every parameter gradient within 1e-6 of its largest entry.  The forward keeps dact only
    for a train-mode step that keeps a tape for the head: never in eval or under no_grad."""
    stack = mods["stack"]
    kind, cfg = FULL_MODELS[name]
    scans = _scan_dicts(mods, 3000, 5, ragged=True)
    pos = None
    if kind == "spgnn":
        pos = np.concatenate([mods["ope"].dist_pos_enc(s["adj"], mods["ope"].anchors_39(s["fvs_out"], s["adj"]))[0]
                              for s in scans])
    torch.manual_seed(4)
    net = getattr(mods["sm"], NET_CLS[kind])(**cfg).cuda()
    net.init()
    with torch.no_grad():
        for k, p_ in net.named_parameters():
            if k.endswith("bias"):
                p_.normal_(0, 0.05)
    net.set_gcn_only()
    net.train(True)
    net.gat.gat_layers[-1].attn_drop_p = 0.2
    g = _device_batch(mods, scans, pos)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans])).cuda()
    cw = torch.tensor([0.2] + [0.8] * 21).cuda()

    saved = []
    real = stack._wide_forward

    def spy(*args, **kw):
        out32, P, rec = real(*args, **kw)
        saved.append(rec.dact is not None)
        return out32, P, rec

    monkeypatch.setattr(stack, "_wide_forward", spy)
    res = {}
    for flag in (True, False):
        monkeypatch.setattr(stack, "WIDE_SAVED_DACT", flag)
        saved.clear()
        res[flag] = _net_step(mods, net, g, y, cw, with_emb)
        assert saved == [flag], (name, flag, saved)
    plan = net.gat._stack_plan()
    assert plan.layers[-1].wide
    for a, b in zip(res[True][0], res[False][0]):
        assert torch.equal(a, b), name
    assert set(res[True][1]) == set(res[False][1])
    for k, b in res[False][1].items():
        err = float((res[True][1][k].double() - b.double()).abs().max())
        assert err <= 1e-6 * float(b.abs().max()), (name, k, err, float(b.abs().max()))

    monkeypatch.setattr(stack, "WIDE_SAVED_DACT", True)
    saved.clear()
    net.eval()
    net(g)
    net.train(True)
    with torch.no_grad():
        net(g)
    assert saved == [False, False], saved
