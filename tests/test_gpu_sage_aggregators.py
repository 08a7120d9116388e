"""SAGEConv mean / gcn / lstm on the GPU against the oracle (DGL 0.7's op sequence): full-width forward and backward
in eval and train mode, sampled blocks (with an empty destination), general in-degree, the lstm reducer at 4096
trees, and the exp_settings runners with a non-default aggregator."""
import numpy as np
import pytest
import torch

from sage_oracle import gnn_net
from helpers import FULL_MODELS, assert_grads_match, oracle_fp64, rel_err, rel_err_elementwise, replay, traced
from test_gpu_parity import (TOL, GRAD_TOL, TRAIN_GRAD_TOL, _device_batch, _oracle_batch, _random_tree_adj,
                             _scan_dicts, _scans_on)

pytestmark = pytest.mark.gpu

AGGS = ("mean", "gcn", "lstm")


@pytest.fixture(scope="module")
def mods():
    from oracle import dgl_ops, models as om
    from spgnn_b200 import graph as sg, models as sm, ops, synth
    return dict(dgl_ops=dgl_ops, om=om, sg=sg, sm=sm, ops=ops, synth=synth)


def _cfg(agg):
    kind, cfg = FULL_MODELS["st_sage_3"]
    return dict(cfg, aggregator_type=agg)


def _pair(mods, agg, train):
    cfg = _cfg(agg)
    torch.manual_seed(0)
    onet = gnn_net(cfg)
    onet.init_like_reference()
    with torch.no_grad():
        for k, p in onet.named_parameters():
            if k.endswith("bias"):
                p.normal_(0, 0.05)
    net = mods["sm"].SAGENet(**cfg).cuda()
    net.load_state_dict(onet.state_dict(), strict=True)
    onet.train(train)
    net.train(train)
    return onet, net


def _compare(mods, agg, scans, train, tag):
    """Forward + masked CE + backward: device (dropout masks recorded) vs oracle (masks replayed); logits (global and
    element-wise), per-tree decisions, loss and every parameter gradient against the fp64 oracle."""
    ops = mods["ops"]
    onet, net = _pair(mods, agg, train)
    og = _oracle_batch(mods, scans)
    g = _device_batch(mods, scans)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]).astype(np.int64))
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
        assert any(k == "drop" for k, _ in rec), "train mode without a dropout mask on the tape"
    for j in range(len(ref)):
        assert rel_err(out[j].detach().cpu(), ref[j].detach()) < TOL, (tag, "output", j)
        assert rel_err_elementwise(out[j].detach().cpu(), ref[j].detach(), 0.25 if j == 0 else 0.5) < TOL, (tag, j)
    assert abs(loss.item() - loss_ref.item()) < TOL * abs(loss_ref.item())
    dec = ops.segmented_argmax(out[0].detach(), g).cpu()
    assert torch.equal(dec, mods["om"].decide_per_tree(ref[0].detach(), og.batch_num_nodes())), tag
    assert_grads_match(net, onet64, TRAIN_GRAD_TOL if train else GRAD_TOL, (tag, f"{tape.flips} of {tape.decisions}"))
    return g


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("agg", AGGS)
def test_full_width_step_vs_oracle(mods, agg, train):
    _compare(mods, agg, _scan_dicts(mods, 1000 if not train else 3000, 6 if not train else 4, ragged=True), train,
             (agg, train))


@pytest.mark.parametrize("agg", AGGS)
@pytest.mark.parametrize("case", ["single_node_trees", "trifurcations", "six_children", "above_384_nodes"])
def test_general_degree_vs_oracle(mods, agg, case):
    """Trees outside the synthetic airway envelope: single-node trees (one LSTM step), tri- and quadrifurcations,
    up to six children (in-degree up to 8 with the self loop: up to 8 LSTM steps), a tree of 801 nodes."""
    rng = np.random.default_rng(17)
    adjs = {"single_node_trees": [_random_tree_adj(n, 2, rng) for n in (1, 3, 120, 1, 2)],
            "trifurcations": [_random_tree_adj(n, 4, rng) for n in (150, 90)],
            "six_children": [_random_tree_adj(n, 6, rng) for n in (200, 57, 33)],
            "above_384_nodes": [_random_tree_adj(801, 2, rng), _random_tree_adj(60, 2, rng)]}[case]
    g = _compare(mods, agg, _scans_on(adjs, rng), False, (agg, case))
    if agg == "lstm":
        o = mods["ops"].lstm_order(g)
        deg = (g.in_ptr[1:] - g.in_ptr[:-1]).cpu()
        assert o.steps == [int((deg > t).sum()) for t in range(int(deg.max()))] and o.off[-1] == g.num_edges
        perm = o.perm.cpu().long()
        assert torch.equal(perm, torch.sort(-deg, stable=True)[1])           # descending, stable
        assert torch.equal(o.rank.cpu().long()[perm], torch.arange(g.num_nodes))


def _oracle_blocks(mods, blocks):
    out = []
    for b in blocks:
        s_loc, d_loc = b.edges()
        out.append(mods["dgl_ops"].Block(s_loc.cpu(), d_loc.cpu(), b.num_src_nodes, b.num_dst_nodes))
    return out


@pytest.mark.parametrize("agg", AGGS)
def test_forward_batch_on_sampled_blocks_vs_oracle(mods, agg):
    """SAGENet.forward_batch on MultiLayerNeighborSampler([2,2,2,2]) blocks, and on the same blocks with every in-edge
    of two destinations of the last block removed (zero in-degree: mean / lstm add nothing, gcn keeps x[v])."""
    from spgnn_b200 import sampling
    scans = _scan_dicts(mods, 500, 4, ragged=True)
    g = _device_batch(mods, scans)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]).astype(np.int64))
    g.ndata["y"] = y.cuda()
    onet, net = _pair(mods, agg, False)
    gen = torch.Generator(device="cuda").manual_seed(3)
    seeds = torch.randperm(g.num_nodes, device="cuda", generator=gen)[:64]
    loader = sampling.NodeDataLoader(g, seeds, sampling.MultiLayerNeighborSampler(net.sage.node_ks), batch_size=64,
                                     generator=gen)
    (_, sd, blocks), = list(loader)
    last = blocks[-1]
    s_loc, d_loc = last.edges()
    keep = (d_loc != 5) & (d_loc != 17)
    cut = sampling.Block(s_loc[keep], d_loc[keep], last.src_ids, last.num_dst_nodes)
    assert int((cut.in_ptr[1:] == cut.in_ptr[:-1]).sum()) == 2
    cw = torch.tensor([0.2] + [0.8] * 21)
    x = blocks[0].srcdata["fvs"]
    for tag, bl in (("sampled", blocks), ("empty_destination", blocks[:-1] + [cut])):
        net.zero_grad()
        onet.zero_grad()
        out, emb = net.forward_batch(bl, x)
        loss = mods["ops"].masked_cross_entropy(out, y[seeds.cpu()].cuda(), cw.cuda(), rate=1.0)
        loss.backward()
        onet64 = oracle_fp64(onet, _oracle_batch(mods, scans[:1]))[0]
        ref_out, ref_emb = onet.forward_batch(_oracle_blocks(mods, bl), x.cpu())
        ref64, _ = onet64.forward_batch(_oracle_blocks(mods, bl), x.cpu().double())
        torch.nn.functional.cross_entropy(ref64, y[seeds.cpu()], weight=cw.double()).backward()
        assert rel_err(out.detach().cpu(), ref_out.detach()) < TOL, (agg, tag)
        assert rel_err(emb.detach().cpu(), ref_emb.detach()) < TOL, (agg, tag)
        assert_grads_match(net, onet64, GRAD_TOL, (agg, tag))


B = 4096


@pytest.fixture(scope="module")
def big():
    from spgnn_b200 import synth_device
    return synth_device.make_batch(0, B, ragged=False)


def test_lstm_at_4096_trees_is_deterministic_and_equals_the_sum_over_sub_batches(mods, big):
    """Full-width lstm SAGENet on 4096 trees: two training steps' gradients are bit-identical, and the gradient of
    the batch equals the fp64 sum over 8 sub-batches of 512 trees (disjoint components, a plain sum over nodes) —
    this holds the long dW_hh reduction over ~2.5 M step rows and the 64-bit row offsets to the small-batch path."""
    from spgnn_b200 import synth_device
    torch.manual_seed(5)
    net = mods["sm"].SAGENet(**_cfg("lstm")).cuda()
    with torch.no_grad():
        for k, p in net.named_parameters():
            if k.endswith("bias"):
                p.normal_(0, 0.05)
    net.eval()
    g = big.graph
    N = g.num_nodes
    R = torch.randn(N, 22, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9)) / N ** 0.5

    def grads(graph, rows):
        net.zero_grad(set_to_none=True)
        (net(graph)[0] * rows).sum().backward()
        return {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None}

    g1 = grads(g, R)
    g2 = grads(g, R)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    del g2
    big_grads = {k: v.double() for k, v in g1.items()}
    del g1
    off = g.node_off.cpu().numpy()
    acc = {k: torch.zeros_like(v) for k, v in big_grads.items()}
    step = B // 8
    for first in range(0, B, step):
        sb = synth_device.make_batch(first, step, ragged=False)
        for k, v in grads(sb.graph, R[off[first]:off[first + step]]).items():
            acc[k] += v.double()
    gmax = max(float(v.abs().max()) for v in acc.values())
    for k, v in big_grads.items():
        err = float((v - acc[k]).abs().max())
        assert err <= 1e-4 * float(acc[k].abs().max()) or err <= 1e-6 * gmax, (k, err, float(acc[k].abs().max()))


def test_settings_file_with_lstm_aggregator_trains_checkpoints_and_tests(tmp_path):
    """An exp_settings file that differs from st_sage_3 in aggregator_type only: GCNTrainSAGE takes training steps,
    writes a checkpoint, and GCNTest reloads it and runs inference."""
    from spgnn_b200 import job_runner, ops
    from spgnn_b200.settings import PRESETS, Settings, get_callable_by_name
    torch.manual_seed(0)
    ops.manual_seed(0)
    p = PRESETS["st_sage_3"]
    path = tmp_path / "st_sage_3_lstm.py"
    path.write_text("".join(f"{k} = {v!r}\n" for k, v in dict(p, MODEL=dict(p["MODEL"], aggregator_type="lstm"),
                                                               EXP_NAME="exp", MODEL_ROOT_PATH=str(tmp_path),
                                                               SYNTHETIC_SCANS=3, SYNTHETIC_RAGGED=True,
                                                               TRAIN_BATCH_SIZE=2, TRAIN_SAMPLE_SIZE=2, GCN_STEPS=3,
                                                               LOG_STEPS=1, NUM_EPOCHS=2, SAVE_EPOCHS=1).items()))
    s = Settings(str(path))
    tr = get_callable_by_name(s.JOB_RUNNER_CLS)(s)
    assert isinstance(tr, job_runner.GCNTrainSAGE)
    assert tr.model.sage.g_layers[0]._aggre_type == "lstm"
    hist = tr.run()
    assert len(hist) > 0 and np.isfinite(hist).all()
    ck = sorted((tmp_path / "exp").glob("*.pth"))
    assert ck, "no checkpoint written"
    state = torch.load(ck[-1], weights_only=False)
    assert "sage.g_layers.0.lstm.weight_hh_l0" in state["model_dict"]
    s2 = Settings(str(path))
    s2.RELOAD_CHECKPOINT_PATH = str(ck[-1])
    te = get_callable_by_name(s2.TEST_RUNNER_CLS)(settings_module=s2, output_path=str(tmp_path / "out"))
    for k, v in tr.model.state_dict().items():
        assert torch.equal(v, te.model.state_dict()[k]), k
    res = te.run()
    assert len(res) == 3
    r = next(iter(res.values()))
    assert r["decision"].shape == (21,) and 0.0 <= r["acc"] <= 1.0
