"""Shared helpers for the test-suite (settings dicts, golden loaders, tolerances)."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# tests/golden/make_golden.py:TINY — widths of the committed wiring fixtures
TINY_COMMON = dict(out_ch=22, fv_dim=32, num_hiddens=[16, 8, 8], node_embed_dim=24)
TINY_MODELS = {
    "gat3": ("gat", dict(TINY_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1, attn_drop=0.1,
                         negative_slope=0.2)),
    "gat3_nr": ("gat", dict(TINY_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                            attn_drop=0.1, negative_slope=0.2, res=False)),
    "gat6": ("gat", dict(TINY_COMMON, num_gat_layers=6, num_heads=2, num_out_heads=2, feat_drop=0.1, attn_drop=0.1,
                         negative_slope=0.2, num_hiddens=[16, 8, 8, 8, 8, 8])),
    "gcn3": ("gcn", dict(TINY_COMMON, num_gcn_layers=3)),
    "gin3": ("gin", dict(TINY_COMMON, num_gin_layers=3)),
    "sage3": ("sage", dict(TINY_COMMON, num_layers=3, feat_drop=0.1, node_ks=[2, 2, 2, 2], node_sample_rate=0.3)),
    "spgnn3": ("spgnn", dict(TINY_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                             attn_drop=0.1, negative_slope=0.2, pos_hiddens=[16, 8, 8], num_pos_heads=1,
                             pos_enc_dim=39)),
    "spgnnnl3": ("spgnn", dict(TINY_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                               attn_drop=0.1, negative_slope=0.2, pos_hiddens=[16, 8, 8], num_pos_heads=1,
                               pos_enc_dim=39, mode="PENL")),
}

# exp_settings/*.py MODEL dicts, GNN keys only (SURVEY.md Appendix A)
FULL_COMMON = dict(out_ch=22, fv_dim=1024, num_hiddens=[256, 128, 64], node_embed_dim=1024)
FULL_MODELS = {
    "st_gat_3": ("gat", dict(FULL_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                             attn_drop=0.1, negative_slope=0.2)),
    "st_gat_6": ("gat", dict(FULL_COMMON, num_gat_layers=6, num_heads=2, num_out_heads=2, feat_drop=0.1,
                             attn_drop=0.1, negative_slope=0.2, num_hiddens=[256, 128, 64, 64, 64, 64])),
    "st_gat_6_nr": ("gat", dict(FULL_COMMON, num_gat_layers=6, num_heads=2, num_out_heads=2, feat_drop=0.1,
                                attn_drop=0.1, negative_slope=0.2, num_hiddens=[256, 128, 64, 64, 64, 64],
                                res=False)),
    "st_gcn_3": ("gcn", dict(FULL_COMMON, num_gcn_layers=3)),
    "st_gin_3": ("gin", dict(FULL_COMMON, num_gin_layers=3)),
    "st_sage_3": ("sage", dict(FULL_COMMON, num_layers=3, feat_drop=0.1, node_ks=[2, 2, 2, 2],
                               node_sample_rate=0.3)),
    "st_pgat_spgnn_3": ("spgnn", dict(FULL_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                                      attn_drop=0.1, negative_slope=0.2, pos_hiddens=[256, 128, 64],
                                      num_pos_heads=1, pos_enc_dim=39)),
    "st_pgat_spgnnnl_3": ("spgnn", dict(FULL_COMMON, num_gat_layers=3, num_heads=2, num_out_heads=2, feat_drop=0.1,
                                        attn_drop=0.1, negative_slope=0.2, pos_hiddens=[256, 128, 64],
                                        num_pos_heads=1, pos_enc_dim=39, mode="PENL")),
}


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def golden_state_dict(rec):
    return {k[4:]: torch.from_numpy(v) for k, v in rec.items() if k.startswith("sd::")}


def golden_graph_inputs():
    """The 4-tree batch of tests/golden/graph_pe.npz as python lists."""
    rec = load_golden("graph_pe.npz")
    n = int(rec["n_graphs"])
    scans = [dict(adj=rec[f"adj{i}"], fvs=rec[f"fvs{i}"], fvs_out=rec[f"fvs_out{i}"], labels=rec[f"labels{i}"])
             for i in range(n)]
    return rec, scans


def rel_err(a, b):
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


def rel_err_elementwise(a, b, floor=0.25):
    """max over elements of |a - b| / (|b| + floor * max|b|): the element-wise (numpy.allclose-style) reading of
    north_star's "within 1e-4 relative": |a - b| <= bar * |b| + floor * bar * max|b| for EVERY element.  The additive
    floor is there because a logit is a sum of ~1000 products of the magnitude of the largest logits: an element
    that is ~0 by cancellation still carries the rounding of those terms (measured: 1.2e-5 x max|b|)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    den = b.abs() + floor * float(b.abs().max().clamp(min=1e-30))
    return float(((a - b).abs() / den).max())


def oracle_fp64(onet, og):
    """A float64 copy of an oracle net and of its input graph (same parameters, same inputs): the exact value of
    the function both fp32 implementations approximate — the reference for GRADIENTS, whose softmax backward
    (da - sum a da) cancels and amplifies whatever rounding the forward carries, the oracle's fp32 one included."""
    import copy
    net64 = copy.deepcopy(onet).double()
    net64.train(onet.training)
    g64 = copy.copy(og)
    g64.ndata = {k: (v.double() if v.is_floating_point() else v) for k, v in og.ndata.items()}
    return net64, g64


def launches(run):
    """Short names of the library kernels run() launches, template arguments included ('spmm_kernel<4>',
    'act_bwd_planes_kernel<true>'); torch's own kernels are left out.  A throwaway kernel opens the profiler session:
    the profiler has been seen to drop the first launch of a session."""
    import re
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        run()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if "spgnn::" not in e.name:
            continue
        m = re.search(r"(\w+_kernel)\s*(<[\w,\s]*>)?\s*\(", e.name)
        if m:
            names.add(m.group(1) + re.sub(r"\s+", "", m.group(2) or ""))
    return names


def traced(ops, fn):
    """Runs fn() on the device with spgnn_b200.ops.KINK_TRACE recording; returns (result, records)."""
    ops.KINK_TRACE = []
    try:
        out = fn()
    finally:
        rec, ops.KINK_TRACE = ops.KINK_TRACE, None
    return out, rec


def replay(records, fn, tol=1e-4):
    """Runs fn() on the oracle with the device's decisions replayed (oracle/kinks.py); checks the tape was consumed
    exactly and that every decision on which device and oracle disagree sat within ``tol`` of the kink / tie."""
    from oracle import kinks
    with kinks.use(kinks.Tape(records, tol)) as tape:
        out = fn()
    assert tape.done(), f"oracle consumed {tape.pos} of {len(tape.records)} device decisions"
    assert not tape.violations, tape.violations
    return out, tape


def grad_errors(net, onet):
    """{parameter: max abs gradient error / largest gradient entry of that parameter} (diagnostics)"""
    ograds = dict(onet.named_parameters())
    return {k: float((p.grad.cpu().double() - ograds[k].grad.double()).abs().max() / ograds[k].grad.abs().max().clamp(min=1e-30))
            for k, p in net.named_parameters() if ograds[k].grad is not None and p.grad is not None}


def assert_grads_match(net, onet, grad_tol, tag=""):
    """Every parameter gradient of the device net against the oracle net: relative to the parameter's largest
    gradient entry, with an absolute floor of 1e-6 x the largest gradient in the model (gradients that are ~0
    analytically — d attn_r through the shift-invariant softmax — are cancellation noise on both sides)."""
    ograds = dict(onet.named_parameters())
    gmax = max(float(q.grad.abs().max()) for q in ograds.values() if q.grad is not None)
    bad = []
    for k, p in net.named_parameters():
        r = ograds[k].grad
        if r is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, (tag, k)
            continue
        assert p.grad is not None, (tag, k)
        abs_err = float((p.grad.cpu().double() - r.double()).abs().max())
        if not (abs_err <= grad_tol * float(r.abs().max()) or abs_err <= 1e-6 * gmax):
            bad.append((k, f"{abs_err:.3e}", f"{float(r.abs().max()):.3e}"))
    assert not bad, (tag, f"gmax {gmax:.3e}", bad)
