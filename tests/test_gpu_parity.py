"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the reference-generated fixtures.

Bars (BASELINE.json north_star): batching / index arithmetic bit-exact; fp32 logits and positional encodings
within 1e-4 relative; arg-max decisions identical.
"""
import numpy as np
import pytest
import torch

from helpers import (FULL_MODELS, TINY_MODELS, assert_grads_match, golden_graph_inputs, golden_state_dict, load_golden,
                     oracle_fp64, rel_err, rel_err_elementwise, replay, traced)

pytestmark = pytest.mark.gpu

TOL = 1e-4          # north_star tolerance for fp32 logits / encodings
GRAD_TOL = 2e-4     # gradients vs the fp64 oracle, relative to the parameter's largest entry (eval mode)
# Train mode: attention dropout rescales the surviving attention weights by 1/(1-p) and zeroes others, which makes the
# softmax backward (da - sum a da) cancel harder; the projection's split-bf16 operands carry 2^-18 = 3.8e-6 per value
# (60x the rounding of an fp32 FMA chain, 1/130 of the TF32 the reference's torch 1.9 used by default) and the
# cancellation amplifies it to 2-4e-4 on the attention vectors of the dropped layers (measured, branches pinned).
TRAIN_GRAD_TOL = 5e-4


@pytest.fixture(scope="module")
def mods():
    from oracle import dgl_ops, models as om, pe as ope
    from spgnn_b200 import graph as sg, models as sm, ops, pe as spe, synth
    return dict(dgl_ops=dgl_ops, om=om, ope=ope, sg=sg, sm=sm, ops=ops, spe=spe, synth=synth)


NET_CLS = {"gat": "GATNet", "gcn": "GCNNet", "gin": "GINNet", "sage": "SAGENet", "spgnn": "GATPositionSPGNNNet"}


def _device_batch(m, scans, pos_enc=None):
    g = m["sg"].batch_from_adjs([s["adj"] for s in scans])
    g.ndata["fvs"] = torch.from_numpy(np.concatenate([s["fvs"] for s in scans])).cuda()
    g.ndata["fvs_out"] = torch.from_numpy(np.concatenate([s["fvs_out"] for s in scans])).cuda()
    if pos_enc is not None:
        g.ndata["pos_enc"] = torch.from_numpy(pos_enc).cuda()
    return g


def _oracle_batch(m, scans, pos_encs=None):
    gs = []
    for i, s in enumerate(scans):
        og = m["dgl_ops"].graph_from_adj(s["adj"])
        og.ndata["fvs"] = torch.from_numpy(s["fvs"])
        if pos_encs is not None:
            og.ndata["pos_enc"] = torch.from_numpy(pos_encs[i])
        gs.append(og)
    return m["dgl_ops"].batch(gs)


def _scan_dicts(m, first, count, ragged=True, fv_dim=1024):
    return [dict(adj=s.adj, fvs=s.fvs, fvs_out=s.fvs_out, labels=s.labels)
            for s in m["synth"].make_scans(first, count, ragged=ragged, fv_dim=fv_dim)]


# ------------------------------------------------------------------------------------------------ graph
def test_batch_builder_matches_reference_fixture(mods):
    rec, scans = golden_graph_inputs()
    g = _device_batch(mods, scans)
    assert np.array_equal(g.src.cpu().numpy(), rec["b_src"])
    assert np.array_equal(g.dst.cpu().numpy(), rec["b_dst"])
    assert np.array_equal(g.batch_num_nodes().cpu().numpy(), rec["b_num_nodes"])
    assert np.array_equal(g.batch_num_edges().cpu().numpy(), rec["b_num_edges"])
    assert g.batch_size == len(scans) and g.number_of_nodes() == int(rec["b_num_nodes"].sum())
    # dgl.batch of single graphs built one by one gives the same thing
    singles = [mods["sg"].from_adj(s["adj"]) for s in scans]
    for i, h in enumerate(singles):
        assert np.array_equal(h.src.cpu().numpy(), rec[f"src{i}"]) and np.array_equal(h.dst.cpu().numpy(), rec[f"dst{i}"])
    g2 = mods["sg"].batch(singles)
    assert torch.equal(g2.src, g.src) and torch.equal(g2.dst, g.dst) and torch.equal(g2.in_src, g.in_src)


def test_from_adj_to_graph_ports_line_by_line(mods):
    """job_runner.py:1779-1801 with ``spgnn_b200.graph`` standing in for ``dgl``: DGLGraph(nx.DiGraph(adj)) →
    remove_self_loop → .to('cuda:0') → ndata → add_edges(nodes, nodes) gives the edge lists the reference's own code
    produced (fixture), and equals the one-pass builder."""
    import networkx as nx
    sg = mods["sg"]
    rec, scans = golden_graph_inputs()
    for i, s in enumerate(scans):
        adj_np = np.asarray(s["adj"])
        for first in (nx.DiGraph(adj_np), adj_np, torch.from_numpy(adj_np)):
            g = sg.DGLGraph(first)
            g = sg.remove_self_loop(g)
            g = g.to('cuda:0')
            g.ndata['y'] = torch.from_numpy(np.asarray(s["labels"]).astype(np.int64)).cuda()
            g.add_edges(g.nodes(), g.nodes())
            assert np.array_equal(g.src.cpu().numpy(), rec[f"src{i}"]) and np.array_equal(g.dst.cpu().numpy(), rec[f"dst{i}"])
            assert g.number_of_nodes() == adj_np.shape[0] and g.ndata['y'].shape[0] == adj_np.shape[0]
        h = sg.from_adj(adj_np)
        assert torch.equal(h.in_src, g.in_src) and torch.equal(h.in_ptr, g.in_ptr) and torch.equal(h.out_dst, g.out_dst)
    und = nx.path_graph(4)                                   # an undirected graph contributes both directions
    assert sg.DGLGraph(und).number_of_edges() == 6
    # the host-side helpers of the reference run on g.cpu(): dgl.to_networkx(g.cpu()) (job_runner.py:1763),
    # g.cpu().to_networkx() (:1652), adjacency_matrix().to_dense().numpy() (:1742), in_degrees() (:1633)
    hg = g.cpu()
    G1, G2 = sg.to_networkx(hg), hg.to_networkx()
    by_id = lambda G: [(u, v) for u, v, _ in sorted(G.edges(data="id"), key=lambda e: e[2])]
    assert by_id(G1) == by_id(G2) == list(zip(rec[f"src{i}"].tolist(), rec[f"dst{i}"].tolist()))
    assert list(G1.edges()) == list(g.to_networkx().edges())
    assert nx.diameter(G1) >= 1 and hg.number_of_nodes() == g.number_of_nodes()
    A = hg.adjacency_matrix().to_dense().numpy()
    assert np.array_equal(A, g.adjacency_matrix().cpu().numpy()) and A.sum() == g.number_of_edges()
    assert np.array_equal(hg.in_degrees().numpy(), g.in_degrees().cpu().numpy())
    assert (hg.adjacency_matrix(scipy_fmt="csr") != g.adjacency_matrix(scipy_fmt="csr")).nnz == 0
    assert torch.equal(hg.ndata['y'], g.ndata['y'].cpu()) and hg.to('cuda:0') is g and hg.cpu() is hg


def test_batch_builder_csc_csr_consistency_ragged_64(mods):
    scans = _scan_dicts(mods, 0, 64, ragged=True, fv_dim=4)
    g = mods["sg"].batch_from_adjs([s["adj"] for s in scans])
    og = _oracle_batch(mods, [dict(s, fvs=s["fvs"]) for s in scans])
    src, dst = g.src.cpu(), g.dst.cpu()
    assert torch.equal(src, og.src) and torch.equal(dst, og.dst)
    in_ptr, in_src, in_eid = g.in_ptr.cpu().long(), g.in_src.cpu().long(), g.in_eid.cpu().long()
    # in-CSC: stable counting sort of the edge list by destination
    order = torch.sort(dst, stable=True)[1]
    assert torch.equal(in_eid, order) and torch.equal(in_src, src[order])
    assert torch.equal(in_ptr[1:] - in_ptr[:-1], torch.bincount(dst, minlength=g.num_nodes))
    # out-CSR: every slot appears once, grouped by source, dst consistent
    out_ptr, out_dst, out_slot = g.out_ptr.cpu().long(), g.out_dst.cpu().long(), g.out_slot.cpu().long()
    assert torch.equal(torch.sort(out_slot)[0], torch.arange(g.num_edges))
    owner = torch.repeat_interleave(torch.arange(g.num_nodes), out_ptr[1:] - out_ptr[:-1])
    assert torch.equal(in_src[out_slot], owner)
    assert torch.equal(out_dst, dst[in_eid[out_slot]])
    assert torch.equal(g.node_gid.cpu().long(),
                       torch.repeat_interleave(torch.arange(64), g.batch_num_nodes().cpu()))


def test_graph_errors(mods, monkeypatch):
    sg = mods["sg"]
    from spgnn_b200._lib import SpgnnError
    g = sg.from_edges([0, 1], [1, 2], 3)                     # node 0 has no in-edge
    net = mods["sm"].GAT(1, 8, [8], 8, [1, 1], torch.nn.functional.elu, 0, 0, 0.2, True).cuda()
    with pytest.raises(SpgnnError):
        net(g, torch.zeros(3, 8, device="cuda"))
    with pytest.raises(SpgnnError):
        sg.from_edges([0, 5], [1, 2], 3)                     # endpoint outside the graph
    with pytest.raises(SpgnnError):
        mods["ops"].linear(torch.zeros(4, 4), torch.zeros(4, 4))   # CPU tensors: no fallback
    monkeypatch.setattr(mods["ops"], "GEMM_MODE", 1)                 # no projection path but the planes GEMMs
    with pytest.raises(SpgnnError):
        mods["ops"].linear(torch.zeros(4, 4, device="cuda"), torch.zeros(4, 4, device="cuda"))


# ------------------------------------------------------------------------------------------------ projection
@pytest.mark.parametrize("M,K1,K2,N", [(300, 64, 0, 48), (1000, 1024, 39, 130), (257, 39, 0, 258), (513, 100, 7, 22),
                                       (128, 64, 0, 16), (5000, 1024, 40, 1028), (4096, 192, 0, 4100),
                                       (64, 64, 0, 24), (10, 1024, 0, 256), (1, 128, 128, 64)])   # mini-batch sized
def test_linear_fwd_bwd_against_fp64(mods, M, K1, K2, N):
    """ops.linear (planes + TMA-fed tcgen05 GEMMs) forward and backward against an fp64 reference."""
    ops = mods["ops"]
    tol = 4e-5
    gen = torch.Generator().manual_seed(M + N)
    x1 = torch.randn(M, K1, generator=gen)
    x2 = torch.randn(M, K2, generator=gen) if K2 else None
    W = torch.randn(N, K1 + K2, generator=gen) / (K1 + K2) ** 0.5
    b = torch.randn(N, generator=gen)
    go = torch.randn(M, N, generator=gen)
    xs = [t.cuda().requires_grad_() for t in ([x1, x2] if K2 else [x1])]
    Wc, bc = W.cuda().requires_grad_(), b.cuda().requires_grad_()
    y = ops.linear(xs[0], Wc, bc, "elu", x2=xs[1] if K2 else None)
    y.backward(go.cuda())
    xd = [t.double().requires_grad_() for t in ([x1, x2] if K2 else [x1])]
    Wd, bd = W.double().requires_grad_(), b.double().requires_grad_()
    yd = torch.nn.functional.elu(torch.cat(xd, 1) @ Wd.t() + bd)
    yd.backward(go.double())
    assert rel_err(y.detach().cpu(), yd.detach()) < tol
    for a, r in zip(xs + [Wc, bc], xd + [Wd, bd]):
        assert rel_err(a.grad.cpu(), r.grad) < tol


# ------------------------------------------------------------------------------------------------ models
@pytest.mark.parametrize("name", sorted(TINY_MODELS))
def test_models_match_reference_wiring_fixtures(mods, name):
    """CUDA path vs outputs of the reference's own models.py classes (tests/golden/wiring_*.npz)."""
    rec, scans = golden_graph_inputs()
    w = load_golden(f"wiring_{name}.npz")
    kind, cfg = TINY_MODELS[name]
    net = getattr(mods["sm"], NET_CLS[kind])(**cfg).cuda()
    res = net.load_state_dict(golden_state_dict(w), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    net.eval()
    g = _device_batch(mods, scans, rec["b_pos_enc"])
    with torch.no_grad():
        out = net(g)
    j = 0
    while f"out{j}" in w:
        assert rel_err(out[j].cpu(), w[f"out{j}"]) < TOL, (name, j)
        j += 1
    assert j == len(out)
    dec = mods["ops"].segmented_argmax(out[0], g)
    assert np.array_equal(dec.cpu().numpy(), w["decision"])
    assert np.array_equal(out[0].argmax(1).cpu().numpy(), w["out0"].argmax(1))


def _margin_aware_flips(a, b, tol):
    """arg-max flips whose top-2 margin in the reference exceeds the tolerance (must be zero)."""
    a, b = a.double(), b.double()
    flips = (a.argmax(1) != b.argmax(1)).nonzero().flatten()
    top2 = b.topk(2, dim=1)[0]
    margin = (top2[:, 0] - top2[:, 1]) / b.abs().max()
    return int((margin[flips] > tol).sum())


# every model, and GIN once more with its MLP run module by module (Linear, Dropout, fused LeakyReLU, Linear): the
# branch of nn.GINConv.forward that any apply_func other than the reference's MLP takes
@pytest.mark.parametrize("name,unfused", [pytest.param(n, False, id=n) for n in sorted(FULL_MODELS)] +
                         [pytest.param("st_gin_3", True, id="st_gin_3-unfused")])
def test_full_width_forward_backward_vs_oracle(mods, name, unfused, monkeypatch):
    """exp_settings widths, 6 ragged trees, eval-mode forward + all parameter gradients vs the CPU oracle, at the
    SAME bar (1e-4 outputs, 2e-4 gradients) for every model family.

    The gradient of a LeakyReLU / ReLU / max is a discontinuous function of the forward values: an attention logit,
    an MLP pre-activation or a pair of pooled neighbours within rounding distance of the kink / the tie takes one
    branch on the device and the other in the oracle, and a whole gradient row moves (this is what the 3e-2 bar of
    round 1 and the "in-degree > 4" xfail were hiding: scripts/deg5_bisect.py shows every kernel exact on those
    graphs).  The device therefore records the branch it took at every such decision (ops.KINK_TRACE) and the oracle
    replays it (oracle/kinks.py), verifying that each decision it would have taken differently sat within 1e-4 of
    the kink.  With the branches pinned the two implementations compute the same function and are compared
    exactly."""
    kind, cfg = FULL_MODELS[name]
    ops = mods["ops"]
    if unfused:
        from spgnn_b200 import nn as snn
        monkeypatch.setattr(snn, "_is_gin_mlp", lambda mlp: False)
    scans = _scan_dicts(mods, 1000, 6, ragged=True)
    pos = None
    if kind == "spgnn":
        pos = []
        for s in scans:
            anc = mods["ope"].anchors_39(s["fvs_out"], s["adj"])
            pos.append(mods["ope"].dist_pos_enc(s["adj"], anc)[0])
    torch.manual_seed(0)
    onet = mods["om"].GNNNet(kind, cfg)
    onet.init_like_reference()
    with torch.no_grad():
        for k, p in onet.named_parameters():
            if k.endswith("bias"):
                p.normal_(0, 0.05)
    onet.eval()
    net = getattr(mods["sm"], NET_CLS[kind])(**cfg).cuda()
    net.load_state_dict(onet.state_dict(), strict=True)
    net.eval()
    og = _oracle_batch(mods, scans, pos)
    g = _device_batch(mods, scans, np.concatenate(pos) if pos is not None else None)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]))
    cw = torch.tensor([0.2] + [0.8] * 21)
    mask = torch.from_numpy(np.concatenate([s["labels"] for s in scans]) != 0) | (torch.rand(y.numel(), generator=torch.Generator().manual_seed(1)) < 0.15)

    out, rec = traced(ops, lambda: net(g))
    loss = ops.masked_cross_entropy(out[0], y.cuda(), cw.cuda(), mask=mask.cuda())
    loss.backward()
    ref, tape = replay(rec, lambda: onet(og))                 # fp32, as DGL computes: the reference for the outputs
    loss_ref = mods["om"].cross_entropy_masked(ref[0], y, mask, cw)
    onet64, og64 = oracle_fp64(onet, og)                      # fp64: the reference for the gradients
    ref64, _ = replay(rec, lambda: onet64(og64))
    mods["om"].cross_entropy_masked(ref64[0], y, mask, cw.double()).backward()

    for j in range(len(ref)):
        assert rel_err(out[j].detach().cpu(), ref[j].detach()) < TOL, (name, "output", j)
        # element-wise: logits against 1e-4 x (|ref| + max|ref| / 4); the embeddings (tanh / ELU outputs, whose
        # pre-activations are larger than the outputs) against 1e-4 x (|ref| + max|ref| / 2)
        assert rel_err_elementwise(out[j].detach().cpu(), ref[j].detach(), 0.25 if j == 0 else 0.5) < TOL, \
            (name, "output, element-wise", j)
    assert abs(loss.item() - loss_ref.item()) < TOL * abs(loss_ref.item())
    assert _margin_aware_flips(out[0].detach().cpu(), ref[0].detach(), TOL) == 0
    dec = ops.segmented_argmax(out[0].detach(), g).cpu()
    dec_ref = mods["om"].decide_per_tree(ref[0].detach(), og.batch_num_nodes())
    assert torch.equal(dec, dec_ref)
    assert_grads_match(net, onet64, GRAD_TOL, (name, unfused, f"{tape.flips} of {tape.decisions} decisions pinned"))


@pytest.mark.parametrize("name", ["st_gat_3", "st_gat_6_nr", "st_pgat_spgnn_3", "st_pgat_spgnnnl_3"])
@pytest.mark.parametrize("train", [False, True])
def test_aggregate_first_output_layer_equals_projection_first(mods, name, train, monkeypatch):
    """The head-averaged output layer evaluated aggregate-first (spgnn_gat_aggx_* + spgnn_wide_linear) against the
    projection-first layer kernels on the same weights, inputs and dropout seeds: outputs and every parameter
    gradient agree to fp32 round-off (both paths hold the 1e-4 bar against the oracle separately).  In train mode
    the output layer gets attention dropout as well, so the regenerated masks of both paths are compared too."""
    from spgnn_b200 import stack
    kind, cfg = FULL_MODELS[name]
    scans = _scan_dicts(mods, 2000, 5, ragged=True)
    pos = None
    if kind == "spgnn":
        pos = np.concatenate([mods["ope"].dist_pos_enc(s["adj"], mods["ope"].anchors_39(s["fvs_out"], s["adj"]))[0]
                              for s in scans])
    torch.manual_seed(3)
    net = getattr(mods["sm"], NET_CLS[kind])(**cfg).cuda()
    net.init()
    with torch.no_grad():
        for k, p_ in net.named_parameters():
            if k.endswith("bias"):
                p_.normal_(0, 0.05)
    net.set_gcn_only()
    net.train(train)
    if train:
        net.gat.gat_layers[-1].attn_drop_p = 0.2
    g = _device_batch(mods, scans, pos)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans])).cuda()
    cw = torch.tensor([0.2] + [0.8] * 21).cuda()
    res = {}
    for wide in (True, False):
        monkeypatch.setattr(stack, "WIDE_OUTPUT_LAYER", wide)
        mods["ops"].manual_seed(11)
        net.zero_grad()
        out = net(g)
        loss = mods["ops"].masked_cross_entropy(out[0], y, cw, mask=torch.ones_like(y, dtype=torch.bool))
        (loss + 1e-3 * out[1].square().mean()).backward()
        res[wide] = ([o.detach().clone() for o in out], {k: p_.grad.clone() for k, p_ in net.named_parameters()
                                                         if p_.grad is not None})
    plan = net.gat._stack_plan()
    assert plan.layers[-1].wide, "the output layer of this preset should qualify for the aggregate-first path"
    for a, b in zip(res[True][0], res[False][0]):
        assert rel_err(a.cpu(), b.cpu()) < 2e-5, name
    gmax = max(float(v.abs().max()) for v in res[False][1].values())
    assert set(res[True][1]) == set(res[False][1])
    for k, b in res[False][1].items():
        a = res[True][1][k]
        abs_err = float((a.double() - b.double()).abs().max())
        assert abs_err <= 5e-5 * float(b.abs().max()) or abs_err <= 1e-6 * gmax, (name, k, abs_err, float(b.abs().max()))


def test_state_dict_keys_are_dgl_names(mods):
    kind, cfg = FULL_MODELS["st_pgat_spgnn_3"]
    net = mods["sm"].GATPositionSPGNNNet(**cfg)
    keys = set(net.state_dict())
    for k in ("gat.gat_layers.0.fc.weight", "gat.gat_layers.0.attn_l", "gat.gat_layers.0.attn_r",
              "gat.gat_layers.0.res_fc.weight", "gat.gat_layers.0.bias", "gat.pgnn_layers.2.fc.weight",
              "gnn_out.weight", "gnn_out.bias"):
        assert k in keys
    assert sum(p.numel() for p in net.parameters()) == 2_501_078        # SURVEY.md §8a parameter count
    assert tuple(net.state_dict()["gat.gat_layers.0.fc.weight"].shape) == (512, 1063)


# ------------------------------------------------------------------------------------------------ dropout
def test_train_mode_dropout_statistics_and_determinism(mods):
    ops = mods["ops"]
    x = torch.ones(2000, 64, device="cuda", requires_grad=True)
    ops.manual_seed(7)
    y = ops.concat_dropout(x, None, 0.1, True)
    keep = (y != 0).float().mean().item()
    assert abs(keep - 0.9) < 0.01 and abs(y.mean().item() - 1.0) < 0.02
    assert torch.all((y == 0) | ((y - 1 / 0.9).abs() < 1e-6))
    y.sum().backward()
    assert torch.equal((x.grad != 0), (y != 0))             # backward regenerates the same mask
    ops.manual_seed(7)
    assert torch.equal(ops.concat_dropout(x, None, 0.1, True), y)

    kind, cfg = TINY_MODELS["spgnn3"]
    rec, scans = golden_graph_inputs()
    net = mods["sm"].GATPositionSPGNNNet(**cfg).cuda()
    g = _device_batch(mods, scans, rec["b_pos_enc"])
    net.train()
    ops.manual_seed(3)
    a = net(g)[0]
    ops.manual_seed(3)
    b = net(g)[0]
    ops.manual_seed(4)
    c = net(g)[0]
    assert torch.equal(a, b) and not torch.equal(a, c)
    net.eval()
    assert not torch.equal(net(g)[0], a)


# ------------------------------------------------------------------------------------------------ PE
def test_anchor_select_and_distance_pe_match_reference_fixture(mods):
    rec, scans = golden_graph_inputs()
    g = _device_batch(mods, scans)
    anc = mods["spe"].select_anchors(g).cpu().numpy()
    for i, s in enumerate(scans):
        ref = rec[f"anchors{i}"]
        assert np.array_equal(anc[i, :21], ref[:21])                       # CNN anchors: exact
        assert anc[i].tolist() == mods["ope"].anchors_39(s["fvs_out"], s["adj"])     # distal leaves: deterministic rule
    # with the reference's anchors the encoding is bit-identical to the reference's
    ref_anc = torch.from_numpy(np.stack([rec[f"anchors{i}"] for i in range(len(scans))])).int().cuda()
    pe, diam = mods["spe"].distance_pos_enc(g, ref_anc)
    assert np.array_equal(pe.cpu().numpy(), rec["b_pos_enc"])
    for i, s in enumerate(scans):
        assert int(diam[i]) == mods["ope"].dist_pos_enc(s["adj"], rec[f"anchors{i}"].tolist())[2]


def test_pe_on_64_ragged_trees_vs_oracle(mods):
    scans = _scan_dicts(mods, 500, 64, ragged=True, fv_dim=4)
    g = _device_batch(mods, scans)
    anc = mods["spe"].select_anchors(g)
    pe, _ = mods["spe"].distance_pos_enc(g, anc)
    rw = mods["spe"].rw_pos_enc(g)
    anc, pe, rw = anc.cpu().numpy(), pe.cpu().numpy(), rw.cpu().numpy()
    off = g.node_off.cpu().numpy()
    for i, s in enumerate(scans):
        ref_anc = mods["ope"].anchors_39(s["fvs_out"], s["adj"])
        assert anc[i].tolist() == ref_anc
        assert np.array_equal(pe[off[i]:off[i + 1]], mods["ope"].dist_pos_enc(s["adj"], ref_anc)[0])
    for i in (0, 17, 63):
        ref = mods["ope"].rw_pos_enc(scans[i]["adj"], 39)
        got = rw[off[i]:off[i + 1]]
        assert np.all(got[:, 0::2] == 0)
        assert np.abs(got - ref).max() <= TOL * np.abs(ref).max()
        assert np.allclose(got, ref, rtol=TOL, atol=1e-12)


def test_rw_pe_matches_reference_fixture(mods):
    rec, scans = golden_graph_inputs()
    g = _device_batch(mods, scans)
    rw = mods["spe"].rw_pos_enc(g).cpu().numpy()
    off = g.node_off.cpu().numpy()
    for i in range(len(scans)):
        assert np.allclose(rw[off[i]:off[i + 1]], rec[f"rw_enc{i}"], rtol=TOL, atol=1e-12)


def test_disconnected_graph_raises(mods):
    from spgnn_b200._lib import SpgnnError
    adj = np.eye(30, dtype=np.uint8)
    adj[0, 1] = adj[1, 0] = 1
    g = mods["sg"].from_adj(adj)
    with pytest.raises(SpgnnError):
        mods["spe"].distance_pos_enc(g, torch.zeros(1, 39, dtype=torch.int32, device="cuda"))


# ------------------------------------------------------------------------------------------------ loss / decision
def test_masked_ce_on_device_mask(mods):
    ops = mods["ops"]
    N = 5000
    gen = torch.Generator().manual_seed(0)
    logits = torch.randn(N, 22, generator=gen)
    y = torch.where(torch.rand(N, generator=gen) < 0.07, torch.randint(1, 22, (N,), generator=gen), torch.zeros(N, dtype=torch.long))
    cw = torch.tensor([0.2] + [0.8] * 21)
    lc = logits.cuda().requires_grad_()
    loss = ops.masked_cross_entropy(lc, y.cuda(), cw.cuda(), rate=0.15, seed=99)
    loss.backward()
    kept = lc.grad.abs().sum(1) != 0
    assert torch.all(kept[y.cuda() != 0])                                 # every labelled node survives (job_runner.py:1897)
    frac = kept[y.cuda() == 0].float().mean().item()
    assert abs(frac - 0.15) < 0.02
    lr = logits.clone().requires_grad_()
    ref = torch.nn.functional.cross_entropy(lr[kept.cpu()], y[kept.cpu()], weight=cw)
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * abs(ref.item())
    assert rel_err(lc.grad.cpu(), lr.grad) < 1e-5


# ------------------------------------------------------------------------------------------------ device generator
def test_device_synth_integer_part_is_bit_identical_to_host(mods):
    from spgnn_b200 import synth_device
    for ragged in (False, True):
        scans = mods["synth"].make_scans(40, 8, ragged=ragged, fv_dim=8)
        b = synth_device.make_batch(40, 8, ragged=ragged, fv_dim=8, features=True)
        off = b.graph.node_off.cpu().numpy()
        for i, s in enumerate(scans):
            assert np.array_equal(b.parent[off[i]:off[i + 1]].cpu().numpy(), s.parent)
            assert np.array_equal(b.graph.ndata["y"][off[i]:off[i + 1]].cpu().numpy(), s.labels)
            assert np.allclose(b.graph.ndata["fvs"][off[i]:off[i + 1]].cpu().numpy(), s.fvs, atol=2e-5)
            assert np.allclose(b.graph.ndata["fvs_out"][off[i]:off[i + 1]].cpu().numpy(), s.fvs_out, atol=1e-4)
        ref = mods["sg"].batch_from_adjs([s.adj for s in scans])
        assert torch.equal(ref.src, b.graph.src) and torch.equal(ref.dst, b.graph.dst)


@pytest.mark.parametrize("H,F,K,res", [(2, 256, 1063, True), (1, 64, 39, True), (2, 1024, 192, True), (2, 64, 128, False),
                                       (3, 20, 7, True)])
def test_pack_weight_matches_the_torch_formula(mods, H, F, K, res):
    """spgnn_gat_pack_weight (+bwd) vs [W_fc ; W_res ; (W_fc.view(H,F,K) * attn_l).sum(1) ; ... attn_r] in fp64."""
    ops = mods["ops"]
    gen = torch.Generator().manual_seed(H * 1000 + K)
    w = torch.randn(H * F, K, generator=gen)
    wr = torch.randn(H * F, K, generator=gen) if res else None
    al, ar = torch.randn(1, H, F, generator=gen), torch.randn(1, H, F, generator=gen)
    rows = H * F * (2 if res else 1) + 2 * H
    go = torch.randn(rows, K, generator=gen)
    leaves = [t.cuda().requires_grad_() if t is not None else None for t in (w, wr, al, ar)]
    P = ops.PackWeightFn.apply(*leaves, H, F)
    assert P.shape == (rows, K) and P.stride(0) % 4 == 0 and P.data_ptr() % 16 == 0
    P.backward(go.cuda())
    ref_leaves = [t.double().requires_grad_() if t is not None else None for t in (w, wr, al, ar)]
    w3 = ref_leaves[0].view(H, F, K)
    blocks = [ref_leaves[0]] + ([ref_leaves[1]] if res else []) + \
        [(w3 * ref_leaves[2].view(H, F, 1)).sum(1), (w3 * ref_leaves[3].view(H, F, 1)).sum(1)]
    Pr = torch.cat(blocks, 0)
    Pr.backward(go.double())
    assert rel_err(P.detach().cpu(), Pr.detach()) < 1e-6
    for a, r in zip(leaves, ref_leaves):
        if a is not None:
            assert a.grad.shape == a.shape
            assert rel_err(a.grad.cpu(), r.grad) < 1e-5


def test_sage_forward_batch_on_sampled_blocks_vs_oracle(mods):
    """SAGENet.forward_batch (models.py:685-689, 814-817) on MultiLayerNeighborSampler([2,2,2,2]) blocks: outputs,
    loss and parameter gradients against the oracle run on the SAME blocks (the draw itself is torch's RNG)."""
    from spgnn_b200 import sampling
    kind, cfg = FULL_MODELS["st_sage_3"]
    scans = _scan_dicts(mods, 500, 4, ragged=True)
    g = _device_batch(mods, scans)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]).astype(np.int64))
    g.ndata["y"] = y.cuda()
    torch.manual_seed(0)
    onet = mods["om"].GNNNet(kind, cfg)
    onet.init_like_reference()
    onet.eval()
    net = mods["sm"].SAGENet(**cfg).cuda()
    net.load_state_dict(onet.state_dict(), strict=True)
    net.eval()
    gen = torch.Generator(device="cuda").manual_seed(3)
    seeds = torch.randperm(g.num_nodes, device="cuda", generator=gen)[:64]
    loader = sampling.NodeDataLoader(g, seeds, sampling.MultiLayerNeighborSampler(net.sage.node_ks), batch_size=64,
                                     generator=gen)
    (input_nodes, sd, blocks), = list(loader)
    assert torch.equal(sd, seeds) and len(blocks) == 4 and blocks[-1].num_dst_nodes == 64
    cw = torch.tensor([0.2] + [0.8] * 21)
    out, emb = net.forward_batch(blocks, blocks[0].srcdata["fvs"])
    loss = mods["ops"].masked_cross_entropy(out, blocks[-1].dstdata["y"], cw.cuda(), rate=1.0)
    loss.backward()

    oblocks = []
    for b in blocks:
        s_loc, d_loc = b.edges()
        oblocks.append(mods["dgl_ops"].Block(s_loc.cpu(), d_loc.cpu(), b.num_src_nodes, b.num_dst_nodes))
    ref_out, ref_emb = onet.forward_batch(oblocks, blocks[0].srcdata["fvs"].cpu())
    loss_ref = torch.nn.functional.cross_entropy(ref_out, y[seeds.cpu()], weight=cw)
    loss_ref.backward()
    assert rel_err(out.detach().cpu(), ref_out.detach()) < TOL
    assert rel_err(emb.detach().cpu(), ref_emb.detach()) < TOL
    assert abs(loss.item() - loss_ref.item()) < TOL * abs(loss_ref.item())
    ograds = dict(onet.named_parameters())
    gmax = max(float(q.grad.abs().max()) for q in ograds.values() if q.grad is not None)
    for k, p in net.named_parameters():
        r = ograds[k].grad
        if r is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        abs_err = float((p.grad.cpu().double() - r.double()).abs().max())
        assert abs_err <= 3e-2 * float(r.abs().max()) or abs_err <= 1e-6 * gmax, (k, abs_err, float(r.abs().max()))


@pytest.mark.parametrize("p", [0.0, 0.3])
def test_gin_mlp_function_with_fused_dropout(mods, p):
    """ops.MlpDropFn (GIN's Linear → Dropout → LeakyReLU → Linear → LeakyReLU) against fp64 autograd with the SAME
    dropout mask (regenerated from the seed through spgnn_split_planes): outputs and all five gradients."""
    from spgnn_b200 import stack
    ops = mods["ops"]
    M, a, b = 700, 96, 64
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(M, a, generator=gen)
    W0, b0 = torch.randn(b, a, generator=gen) / a ** 0.5, torch.randn(b, generator=gen) * 0.1
    W3, b3 = torch.randn(b, b, generator=gen) / b ** 0.5, torch.randn(b, generator=gen) * 0.1
    go = torch.randn(M, b, generator=gen)
    seed = 0x1234ABCD
    leaves = [t.cuda().requires_grad_() for t in (x, W0, b0, W3, b3)]
    y = ops.MlpDropFn.apply(*leaves, ops.act_code("leaky_relu"), 0.01, p, seed)
    y.backward(go.cuda())
    # the mask, from the hidden activation and its dropped planes
    with torch.no_grad():
        y1 = ops.linear(leaves[0].detach(), leaves[1].detach(), leaves[2].detach(), "leaky_relu", 0.01)
        dropped = stack.split_planes(y1, p, seed).float()
        scale = torch.where(y1 != 0, dropped / y1, torch.ones_like(y1)).cpu().double()
    if p > 0:
        kept = (scale > 0).double().mean().item()
        assert abs(kept - (1 - p)) < 0.02 and torch.allclose(scale[scale > 0], torch.tensor(1 / (1 - p), dtype=torch.float64), rtol=1e-3)
    ref = [t.double().requires_grad_() for t in (x, W0, b0, W3, b3)]
    # LeakyReLU branches taken from the device outputs: an element within fp32 rounding of the kink would otherwise
    # flip its derivative (1 vs 0.01) between the fp32 and the fp64 evaluation and move a whole gradient row
    s1 = torch.where(y1 > 0, 1.0, 0.01).cpu().double()
    s2 = torch.where(y.detach() > 0, 1.0, 0.01).cpu().double()
    yr = (((ref[0] @ ref[1].t() + ref[2]) * s1 * scale) @ ref[3].t() + ref[4]) * s2
    yr.backward(go.double())
    assert rel_err(y.detach().cpu(), yr.detach()) < 4e-5
    for t, r in zip(leaves, ref):
        assert rel_err(t.grad.cpu(), r.grad) < 1e-4, t.shape


def _random_tree_adj(n, max_children, rng):
    """tree ∪ I as uint8: node i > 0 hangs under a random earlier node that still has room for a child."""
    adj = np.eye(n, dtype=np.uint8)
    kids = np.zeros(n, dtype=np.int64)
    for i in range(1, n):
        cand = np.flatnonzero(kids[:i] < max_children)
        p = int(rng.choice(cand))
        kids[p] += 1
        adj[i, p] = adj[p, i] = 1
    return adj


def _edge_case_adjs(case, rng):
    if case == "tiny_trees":
        return [_random_tree_adj(n, 2, rng) for n in (1, 3, 120, 1, 2)]
    if case == "trifurcations":
        return [_random_tree_adj(n, 4, rng) for n in (150, 90)]
    return [_random_tree_adj(801, 2, rng), _random_tree_adj(60, 2, rng)]


def _model_pair(mods, name, train):
    kind, cfg = FULL_MODELS[name]
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
    return kind, onet, net


def _scans_on(adjs, rng, n_min_anchor=False):
    scans = []
    for a in adjs:
        n = a.shape[0]
        scans.append(dict(adj=a, fvs=np.maximum(rng.standard_normal((n, 1024)), 0).astype(np.float32),
                          fvs_out=(3 * rng.standard_normal((n, 22))).astype(np.float32),
                          labels=rng.integers(0, 22, n).astype(np.int64)))
    return scans


def _compare_step(mods, name, scans, train, tag):
    """One forward + loss + backward of ``name`` on ``scans``: device (decisions recorded) vs oracle (decisions
    replayed); outputs, loss and every parameter gradient at the parity bar."""
    ops = mods["ops"]
    kind, onet, net = _model_pair(mods, name, train)
    pos = None
    if kind == "spgnn":
        pos = [mods["ope"].dist_pos_enc(s["adj"], mods["ope"].anchors_39(s["fvs_out"], s["adj"]))[0] for s in scans]
    og = _oracle_batch(mods, scans, pos)
    g = _device_batch(mods, scans, np.concatenate(pos) if pos is not None else None)
    assert torch.equal(g.src.cpu(), og.src) and torch.equal(g.dst.cpu(), og.dst)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]))
    cw = torch.tensor([0.2] + [0.8] * 21)
    mask = torch.ones(y.numel(), dtype=torch.bool)
    ops.manual_seed(5)
    out, rec = traced(ops, lambda: net(g))
    loss = ops.masked_cross_entropy(out[0], y.cuda(), cw.cuda(), mask=mask.cuda())
    loss.backward()
    ref, tape = replay(rec, lambda: onet(og))                 # fp32 oracle: outputs and loss
    loss_ref = mods["om"].cross_entropy_masked(ref[0], y, mask, cw)
    onet64, og64 = oracle_fp64(onet, og)                      # fp64 oracle: gradients
    ref64, _ = replay(rec, lambda: onet64(og64))
    mods["om"].cross_entropy_masked(ref64[0], y, mask, cw.double()).backward()
    if train and kind != "gcn":                       # GraphConv stacks have no dropout
        assert any(k == "drop" for k, _ in rec), "train mode without a dropout mask on the tape"
    for j in range(len(ref)):
        assert rel_err(out[j].detach().cpu(), ref[j].detach()) < TOL, (tag, j)
    assert abs(loss.item() - loss_ref.item()) < TOL * abs(loss_ref.item())
    assert_grads_match(net, onet64, TRAIN_GRAD_TOL if train else GRAD_TOL,
                       (tag, f"{tape.flips} of {tape.decisions} decisions pinned"))
    return g, tape


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("name", ["st_gat_3", "st_pgat_spgnn_3"])
@pytest.mark.parametrize("case", ["tiny_trees", "trifurcations", "above_384_nodes"])
def test_edge_case_graphs_vs_oracle(mods, case, name, train):
    """Full-width GAT-3 and SPGNN-3 on graphs outside the per-tree kernels' envelope (degree <= 4, <= 384 nodes,
    which the synthetic bifurcating trees never leave): single-node and 3-node trees in a batch, airway trees with
    tri- and quadrifurcations (in-degree up to 6: general-degree branches of gat_layer.cu / gat_wide.cu), a tree of
    801 nodes.  Forward, loss and every parameter gradient vs the oracle, eval and train mode (dropout masks and
    LeakyReLU branches replayed from the device, oracle/kinks.py)."""
    rng = np.random.default_rng(7)
    adjs = _edge_case_adjs(case, rng)
    if name == "st_pgat_spgnn_3":
        adjs = [a for a in adjs if a.shape[0] >= 21] or [_random_tree_adj(30, 2, rng)]   # 21 distinct anchors per tree
    g, _ = _compare_step(mods, name, _scans_on(adjs, rng), train, (case, name, train))
    if case == "trifurcations":
        assert g.max_degree() > 4


def test_random_trees_up_to_six_children_sweep(mods):
    """Hypothesis-style sweep: random batches of random trees with up to 6 children per node (in-degree up to 8),
    random sizes on both sides of the per-tree kernels' limits, GAT-3 and SPGNN-3, eval and train."""
    rng = np.random.default_rng(2026)
    for trial in range(8):
        mc = int(rng.integers(2, 7))
        sizes = [int(rng.integers(21, 420)) for _ in range(int(rng.integers(1, 5)))]
        adjs = [_random_tree_adj(n, mc, rng) for n in sizes]
        name = ("st_gat_3", "st_pgat_spgnn_3")[trial % 2]
        _compare_step(mods, name, _scans_on(adjs, rng), bool((trial // 2) % 2), ("sweep", trial, mc, sizes, name))


def test_batch_builder_csc_csr_consistency_above_degree_4(mods):
    """In-CSC / out-CSR of a batch with in-degree up to 8 (the backward's source side is the only consumer of the
    out-CSR; the bifurcating synthetic trees never exceed degree 4)."""
    rng = np.random.default_rng(11)
    adjs = [_random_tree_adj(n, 6, rng) for n in (150, 90, 33, 301)]
    g = mods["sg"].batch_from_adjs(adjs)
    assert g.max_degree() > 4
    og = _oracle_batch(mods, [dict(adj=a, fvs=np.zeros((a.shape[0], 1), np.float32)) for a in adjs])
    src, dst = g.src.cpu(), g.dst.cpu()
    assert torch.equal(src, og.src) and torch.equal(dst, og.dst)
    in_ptr, in_src, in_eid = g.in_ptr.cpu().long(), g.in_src.cpu().long(), g.in_eid.cpu().long()
    order = torch.sort(dst, stable=True)[1]
    assert torch.equal(in_eid, order) and torch.equal(in_src, src[order])
    assert torch.equal(in_ptr[1:] - in_ptr[:-1], torch.bincount(dst, minlength=g.num_nodes))
    out_ptr, out_dst, out_slot = g.out_ptr.cpu().long(), g.out_dst.cpu().long(), g.out_slot.cpu().long()
    assert torch.equal(torch.sort(out_slot)[0], torch.arange(g.num_edges))          # a permutation of the slots
    owner = torch.repeat_interleave(torch.arange(g.num_nodes), out_ptr[1:] - out_ptr[:-1])
    assert torch.equal(in_src[out_slot], owner)
    assert torch.equal(out_dst, dst[in_eid[out_slot]])
    assert torch.equal(out_ptr[1:] - out_ptr[:-1], torch.bincount(src, minlength=g.num_nodes))
    assert int((in_ptr[1:] - in_ptr[:-1]).max()) == g.max_degree()


@pytest.mark.parametrize("name", sorted(FULL_MODELS))
def test_train_mode_step_matches_oracle_exactly(mods, name):
    """The benchmarked configuration (train mode: feature dropout, attention dropout, GIN's MLP dropout) against the
    oracle with the device's dropout masks injected — the one configuration round 1 only checked statistically."""
    scans = _scan_dicts(mods, 3000, 4, ragged=True)
    _compare_step(mods, name, scans, True, ("train", name))


# ------------------------------------------------------------------------------------------------ optimiser
@pytest.mark.parametrize("kw", [dict(momentum=0.9), dict(momentum=0.0), dict(momentum=0.9, weight_decay=1e-2),
                                dict(momentum=0.9, nesterov=True), dict(momentum=0.8, dampening=0.3, weight_decay=5e-3)])
def test_flat_sgd_matches_torch_optim_sgd(mods, kw):
    """runner.FlatSGD / spgnn_sgd_step against torch.optim.SGD (the reference's optimiser, job_runner.py:239-249,
    1919) over 5 steps including step 0 (momentum buffer = first gradient), with an ExponentialLR decay between
    steps (job_runner.py:1346-1348, gamma 0.9), a parameter that never receives a gradient (torch skips it: no
    momentum-only drift, no weight decay) and one that receives its first gradient at step 2."""
    from spgnn_b200 import runner
    torch.manual_seed(1)
    shapes = [(37, 19), (19,), (5, 7, 3), (11,), (64, 33)]
    init = [torch.randn(*s) for s in shapes]
    ref_p = [torch.nn.Parameter(t.clone().double()) for t in init]
    dev_p = [torch.nn.Parameter(t.clone().cuda()) for t in init]
    lr, gamma = 0.05, 0.9
    ref_opt = torch.optim.SGD(ref_p, lr=lr, **kw)
    sched = torch.optim.lr_scheduler.ExponentialLR(ref_opt, gamma=gamma)
    opt = runner.FlatSGD(dev_p, lr=lr, **kw)
    for step in range(5):
        ref_opt.zero_grad()
        opt.zero_grad()
        for i, (r, d) in enumerate(zip(ref_p, dev_p)):
            if i == 3 or (i == 2 and step < 2):
                continue                                   # no gradient: both optimisers must leave it alone
            g = torch.randn(*shapes[i], generator=torch.Generator().manual_seed(100 * step + i))
            r.grad = g.double()
            d.grad = g.cuda()
        ref_opt.step()
        opt.step()
        sched.step()
        opt.set_lr(opt.lr * gamma)
        for i, (r, d) in enumerate(zip(ref_p, dev_p)):
            assert rel_err(d.detach().cpu(), r.detach()) < 2e-6, (kw, step, i)
    assert torch.equal(dev_p[3].detach().cpu(), init[3])
    sd = opt.state_dict()
    assert 3 not in sd["state"] and (bool(sd["state"]) == (kw["momentum"] != 0.0))
    if kw["momentum"]:
        for i in (0, 1, 2, 4):
            assert rel_err(sd["state"][i]["momentum_buffer"], ref_opt.state[ref_p[i]]["momentum_buffer"]) < 2e-6


# ------------------------------------------------------------------------------------------------ dormant extras
def test_dormant_pe_extras_and_graph_api_leftovers_vs_oracle(mods):
    """SURVEY 8f rank 4 / 8b leftovers: Laplacian-eigenvector PE (job_runner.py:1630-1645), the Laplacian and the
    distance / compactness PE losses (:1803-1861) against their literal restatements in oracle/pe.py, and
    ``adjacency_matrix(scipy_fmt=)`` / ``adjacency_matrix_scipy`` / ``to_networkx`` (:1814, :1632, :1763)."""
    import scipy.sparse as sp
    from spgnn_b200 import pe_extras
    ope, dgl_ops, sg = mods["ope"], mods["dgl_ops"], mods["sg"]
    rng = np.random.default_rng(4)
    adjs = [_random_tree_adj(n, mc, rng) for n, mc in ((60, 2), (45, 3), (30, 2))]
    g = sg.batch_from_adjs(adjs)
    ogs = [dgl_ops.graph_from_adj(a) for a in adjs]
    off = g.node_off.tolist()
    # graph API
    A = g.adjacency_matrix(scipy_fmt="csr")
    assert sp.isspmatrix_csr(A) and A.shape == (g.num_nodes, g.num_nodes) and A.nnz == g.num_edges
    assert np.array_equal(A.toarray(), g.adjacency_matrix().cpu().numpy())
    ids = g.adjacency_matrix_scipy(return_edge_ids=True, fmt="coo")
    assert np.array_equal(np.sort(ids.data), np.arange(g.num_edges))
    G = g.to_networkx()
    assert G.number_of_nodes() == g.num_nodes and G.number_of_edges() == g.num_edges
    assert [(u, v) for u, v, _ in sorted(G.edges(data="id"), key=lambda e: e[2])] == \
        list(zip(g.src.cpu().tolist(), g.dst.cpu().tolist()))
    # eigenvector PE: eigen-pairs of the same Laplacian, same ordering (vectors agree up to sign where non-degenerate)
    ev = pe_extras.compute_eigen_basis(g, 39).cpu().numpy()
    assert ev.shape == (g.num_nodes, 39) and np.array_equal(g.ndata["eigvec"].cpu().numpy(), ev)
    for i, og in enumerate(ogs):
        val, ref = ope.eigen_basis(og, 39)
        L = ope._norm_laplacian(og)
        blk = ev[off[i]:off[i + 1]].astype(np.float64)
        k = min(39, og.num_nodes - 1)
        lam = np.einsum("nk,nk->k", blk[:, :k], L @ blk[:, :k])
        assert np.allclose(lam, val[1:1 + k], atol=1e-5) and np.allclose(L @ blk[:, :k], blk[:, :k] * lam, atol=1e-4)
        assert np.all(blk[:, k:] == 0)
        gaps = np.minimum(np.abs(np.diff(val[:k + 2]))[:-1], np.abs(np.diff(val[:k + 2]))[1:])
        for j in np.nonzero(gaps > 1e-3)[0]:
            assert abs(abs(float(blk[:, j] @ ref[:, j].astype(np.float64))) - 1.0) < 1e-3, (i, j)
    # losses
    gen = torch.Generator().manual_seed(0)
    p = torch.randn(g.num_nodes, 39, generator=gen)
    y = torch.zeros(g.num_nodes, dtype=torch.int64)
    for i in range(len(adjs)):
        nodes = torch.randperm(off[i + 1] - off[i], generator=gen)[:21] + off[i]
        y[nodes] = torch.arange(1, 22)
    y[off[1] + 3] = 0                                         # one label missing in the second tree
    ps = [p[off[i]:off[i + 1]] for i in range(len(adjs))]
    ys = [y[off[i]:off[i + 1]] for i in range(len(adjs))]
    ref = ope.laplacian_pos_loss(ogs, ps, 0.1, 39)
    got = pe_extras.laplacian_pos_loss(g, p.cuda(), 0.1, 39)
    assert abs(float(got) - float(ref)) < 1e-5 * abs(float(ref))
    cache = [torch.from_numpy(ope.dist_pos_enc(a, list(range(21)))[1]) for a in adjs]
    stats0 = torch.rand(len(adjs), 21, 39, generator=gen)
    dev_loss, ref_loss = pe_extras.DistPosLoss(22, 39), ope.DistPosLoss(22, 39)
    for it in range(2):                                        # second call exercises the cached running mean
        pd = (p * (1 + 0.1 * it)).cuda().requires_grad_()
        d1, c1 = dev_loss(g, cache, p=pd, y=y.cuda(), batch_stats_init=stats0)
        d0, c0 = ref_loss([t * (1 + 0.1 * it) for t in ps], ys, cache, stats0)
        assert abs(float(d1) - float(d0)) < 1e-5 * abs(float(d0)) and abs(float(c1) - float(c0)) <= 1e-4 * max(abs(float(c0)), 1e-6)
        (d1 + c1).backward()
        assert torch.isfinite(pd.grad).all()


def test_distance_pe_tree_kernel_equals_all_pairs_kernel_and_oracle(mods, monkeypatch):
    """spgnn_pe_dist_init: the anchor-wave + double-BFS kernel that trees take gives bit-identical encodings and
    diameters to the all-pairs kernel (SPGNN_PE_ALL_PAIRS=1) and to the oracle's hop matrix; a graph with a cycle
    in the same batch is declined by the tree kernel and still comes out right; single-node graphs included."""
    rng = np.random.default_rng(21)
    adjs = [_random_tree_adj(n, mc, rng) for n, mc in ((301, 2), (64, 5), (1, 2), (37, 3), (150, 2), (2, 2))]
    cyc = _random_tree_adj(80, 2, rng)
    cyc[5, 70] = cyc[70, 5] = 1                                  # one extra edge: a cycle, diameter by all pairs
    adjs.insert(2, cyc)
    g = mods["sg"].batch_from_adjs(adjs)
    anchors = torch.stack([torch.from_numpy(rng.integers(0, a.shape[0], 39).astype(np.int32)) for a in adjs]).cuda()
    pe_fast, d_fast = mods["spe"].distance_pos_enc(g, anchors, store=False)
    monkeypatch.setenv("SPGNN_PE_ALL_PAIRS", "1")
    pe_all, d_all = mods["spe"].distance_pos_enc(g, anchors, store=False)
    monkeypatch.delenv("SPGNN_PE_ALL_PAIRS")
    assert torch.equal(pe_fast, pe_all) and torch.equal(d_fast, d_all)
    off = g.node_off.tolist()
    for i, a in enumerate(adjs):
        if a.shape[0] == 1:
            assert float(pe_fast[off[i]].abs().max()) == 0.0 and int(d_fast[i]) == 0
            continue
        ref, _, diam = mods["ope"].dist_pos_enc(a, anchors[i].cpu().tolist())
        assert int(d_fast[i]) == diam and np.array_equal(pe_fast[off[i]:off[i + 1]].cpu().numpy(), ref), i


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,k_off,cc", [(1000, 260, 384, 0, 0), (333, 516, 768, 0, 192), (257, 130, 132, 64, 70)])
def test_dx_gemm_with_the_consumer_dropout_mask_in_its_epilogue(mods, M, N, K, k_off, cc):
    """spgnn_planes_linear_bwd_input_masked == unmasked dX times the feat_drop mask every plane producer derives from
    (seed, row, 4-column chunk) — the mask split_planes applies in the forward (GATConv's feat_drop, models.py:301-314
    via DGL GATConv.forward): the producing layer's backward then reads a finished gradient."""
    from spgnn_b200 import stack
    dev = torch.device("cuda", 0)
    torch.manual_seed(3)
    dC = stack.split_planes(torch.randn(M, N, device=dev))
    W = torch.randn(N, k_off + K, device=dev)
    p, seed = 0.1, 4242
    plain = stack.planes_linear_bwd_input(dC, W, K, k_off=k_off)
    masked = stack.planes_linear_bwd_input(dC, W, K, k_off=k_off, drop_p=p, seed=seed, concat_chunks=cc)
    nch = cc if cc > 0 else (k_off + K + 3) // 4
    keep = stack.split_planes(torch.ones(M, K, device=dev), p=p, seed=seed, concat_chunks=nch, chunk_off=k_off // 4).float()
    frac = float((keep == 0).float().mean())
    assert 0.07 < frac < 0.13
    scale = torch.tensor(1.0, device=dev) / (torch.tensor(1.0, device=dev) - torch.tensor(p, device=dev))   # fp32, as the kernel
    assert torch.equal(masked[:, :K], torch.where(keep != 0, plain[:, :K] * scale, torch.zeros_like(plain[:, :K])))
    again = stack.planes_linear_bwd_input(dC, W, K, k_off=k_off, drop_p=p, seed=seed + 1, concat_chunks=cc)
    assert not torch.equal(again[:, :K], masked[:, :K])


@pytest.mark.gpu
@pytest.mark.parametrize("M,K1,K2,N", [(38017, 512, 256, 516), (40100, 1024, 39, 1028), (37889 + 128, 256, 0, 384)])
def test_cta_pair_projection_gemm_against_fp64_and_the_single_cta_kernel(mods, M, K1, K2, N):
    """nt_pair_kernel (tcgen05 cta_group::2; taken for K >= 256 and N >= 320 once there are >= 4 m-tiles per pair) on
    shapes with an odd number of m-tiles, a ragged last tile and concatenated sources: forward (with bias + ELU in the
    epilogue) and dX against fp64, and bit-for-bit against the same rows pushed through the single-CTA kernel in
    batches too small for the pair path (the projections of GATConv, models.py:301-314 through DGL's fc / res_fc)."""
    from spgnn_b200 import stack
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(M)
    x1 = torch.randn(M, K1, generator=gen).to(dev)
    x2 = torch.randn(M, (K2 + 3) // 4 * 4, generator=gen)[:, :K2].to(dev) if K2 else None
    W = (torch.randn(N, K1 + K2, generator=gen) / (K1 + K2) ** 0.5).to(dev)
    b = torch.randn(N, generator=gen).to(dev)
    P1, P2 = stack.split_planes(x1), (stack.split_planes(x2) if K2 else None)
    y = stack.planes_linear(P1, W, bias=b, act=1, A2=P2)
    xd = torch.cat([x1, x2], 1).double() if K2 else x1.double()
    ref = torch.nn.functional.elu(xd @ W.double().t() + b.double())
    assert rel_err(y[:, :N].cpu(), ref.cpu()) < 4e-5
    go = stack.split_planes(torch.randn(M, N, generator=gen).to(dev))
    dx = stack.planes_linear_bwd_input(go, W, K1 + K2)
    assert rel_err(dx[:, :K1 + K2].cpu(), (go.float().double() @ W.double()).cpu()) < 4e-5
    # the same rows through the single-CTA kernel (small batches never take the pair path): identical bits
    rows = slice(M - 3000, M)
    Ps = stack.split_planes(x1[rows].contiguous())
    P2s = stack.split_planes(x2[rows].contiguous()) if K2 else None
    ys = stack.planes_linear(Ps, W, bias=b, act=1, A2=P2s)
    assert torch.equal(ys[:, :N], y[rows, :N])
    # masked epilogue on the pair path == mask applied afterwards
    dxm = stack.planes_linear_bwd_input(go, W, K1 + K2, drop_p=0.1, seed=99)
    keep = stack.split_planes(torch.ones(M, K1 + K2, device=dev), p=0.1, seed=99).float()
    scale = torch.tensor(1.0, device=dev) / (torch.tensor(1.0, device=dev) - torch.tensor(0.1, device=dev))
    assert torch.equal(dxm[:, :K1 + K2], torch.where(keep != 0, dx[:, :K1 + K2] * scale, torch.zeros_like(dx[:, :K1 + K2])))
