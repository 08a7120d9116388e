"""The device neighbour sampler (csrc/sampling.cu via sampling.DeviceBlockSampler) on the GPU: bit-exact against the
numpy restatement of tests/test_cpu_device_sampler.py, the block invariants, the inclusion distribution, SAGENet's
forward_batch on its blocks against the fp64 oracle, one synchronising call per mini-batch, the GCNTrainSAGE runner
and a 4096-tree batch."""
import warnings

import numpy as np
import pytest
import torch

from helpers import FULL_MODELS, assert_grads_match, oracle_fp64, rel_err
from sage_oracle import gnn_net
from test_cpu_device_sampler import check_invariants, sample_blocks as np_sample_blocks
from test_gpu_parity import GRAD_TOL, TOL, _device_batch, _oracle_batch, _random_tree_adj, _scan_dicts

pytestmark = pytest.mark.gpu

SEED = 0x5EED5A6E


@pytest.fixture(scope="module")
def mods():
    from oracle import dgl_ops, models as om
    from spgnn_b200 import graph as sg, models as sm, ops, sampling, synth
    return dict(dgl_ops=dgl_ops, om=om, sg=sg, sm=sm, ops=ops, sampling=sampling, synth=synth)


def _star(sg, d):
    """Node 0 with in-degree d (d - 1 leaves and a self loop); the leaves have in-degree 0."""
    src = np.concatenate([np.arange(1, d), [0]])
    return sg.from_edges(src, np.zeros(d, np.int64), d)


def _zero_in(sg):
    """Hand-made: a chain 0 -> 1 -> ... -> 5, a fan 6 -> {7, 8, 9} and node 10 isolated; 0, 6 and 10 have no in-edge."""
    src = [0, 1, 2, 3, 4, 6, 6, 6, 7, 8]
    dst = [1, 2, 3, 4, 5, 7, 8, 9, 9, 9]
    return sg.from_edges(src, dst, 11)


def _graph(mods, kind):
    sg = mods["sg"]
    rng = np.random.default_rng(21)
    if kind == "ragged64":
        g = sg.batch_from_adjs([s["adj"] for s in _scan_dicts(mods, 0, 64, ragged=True)])
    elif kind == "six_children":
        g = sg.batch_from_adjs([_random_tree_adj(n, 6, rng) for n in (200, 57, 33, 1)])
    elif kind == "star5000":
        g = _star(sg, 5000)
    else:
        g = _zero_in(sg)
    N = g.num_nodes
    seeds = {"star5000": np.array([0, 17, 4999, 2500]), "zero_in": np.array([0, 9, 6, 10, 5, 2])}.get(
        kind, rng.permutation(N)[:min(N, 150)])
    return g, seeds


def _host(blocks):
    return [dict(src_ids=b.src_ids.cpu().numpy(), in_ptr=b.in_ptr.cpu().numpy().astype(np.int64),
                 in_src=b.in_src.cpu().numpy().astype(np.int64), out_ptr=b.out_ptr.cpu().numpy().astype(np.int64),
                 out_dst=b.out_dst.cpu().numpy().astype(np.int64),
                 out_slot=b.out_slot.cpu().numpy().astype(np.int64), num_dst=b.num_dst_nodes) for b in blocks]


FANOUTS = [[0], [1], [2], [6000], [-1], [2, 2, 2, 2], [1, -1, 0, 3], [6000, 2, -1, 1]]


@pytest.mark.parametrize("fanouts", FANOUTS, ids=lambda f: "_".join(map(str, f)))
@pytest.mark.parametrize("kind", ["ragged64", "six_children", "star5000", "zero_in"])
def test_blocks_equal_the_restatement_and_meet_the_invariants(mods, kind, fanouts):
    g, seeds = _graph(mods, kind)
    in_ptr, in_src = g.in_ptr.cpu().numpy(), g.in_src.cpu().numpy()
    sampler = mods["sampling"].DeviceBlockSampler(fanouts)
    for salt in (0, 1, 2 ** 63 + 5):
        blocks = sampler.sample_blocks(g, torch.from_numpy(seeds).cuda(), seed=SEED, salt=salt, gather=False)
        got, want = _host(blocks), np_sample_blocks(in_ptr, in_src, seeds, fanouts, SEED, salt)
        assert len(got) == len(want) == len(fanouts)
        for l, (a, b) in enumerate(zip(got, want)):
            assert a["num_dst"] == b["num_dst"], (l, "num_dst")
            for k in ("src_ids", "in_ptr", "in_src", "out_ptr", "out_dst", "out_slot"):
                assert np.array_equal(a[k], b[k]), (l, k, salt)
        check_invariants(got, in_ptr, in_src, seeds)
    assert bool((g._sample_pos == -1).all())                    # the scratch is left clean


def test_node_data_gathers_and_refusals(mods):
    sampling = mods["sampling"]
    g, seeds = _graph(mods, "ragged64")
    g.ndata["fvs"] = torch.randn(g.num_nodes, 40, device="cuda")
    g.ndata["y"] = torch.randint(0, 22, (g.num_nodes,), device="cuda")
    blocks = sampling.DeviceBlockSampler([2, 2, 2]).sample_blocks(g, torch.from_numpy(seeds).cuda(), seed=1)
    assert torch.equal(blocks[0].srcdata["fvs"], g.ndata["fvs"][blocks[0].src_ids])
    assert torch.equal(blocks[-1].dstdata["y"], g.ndata["y"][torch.from_numpy(seeds).cuda()])
    from spgnn_b200._lib import SpgnnError
    s = sampling.DeviceBlockSampler([2, 2])
    for bad in ([0, 5, 5], [3, g.num_nodes], [-1, 2]):                       # repeated, out of range, negative
        with pytest.raises(SpgnnError):
            s.sample_blocks(g, torch.tensor(bad, device="cuda"), seed=1)
        assert bool((g._sample_pos == -1).all())
    with pytest.raises(SpgnnError):
        sampling.DeviceNodeDataLoader(g, [0, g.num_nodes], s)
    ok = s.sample_blocks(g, torch.tensor([0, 5], device="cuda"), seed=1)           # still usable after a refusal
    assert torch.equal(ok[-1].dst_ids.cpu(), torch.tensor([0, 5]))


def test_each_in_edge_is_kept_with_probability_min_f_d_over_d(mods):
    """500 copies of a node with six children (in-degree 7 with its self loop) as seeds, 40 salts: the kept count
    of every CSC position follows min(f, d)/d (chi-square, significance 1e-3), for f = 1, 2, 3, 6."""
    from scipy.stats import chisquare
    sg, sampling = mods["sg"], mods["sampling"]
    d, copies = 7, 500
    adj = np.eye(d, dtype=np.uint8)
    adj[0, 1:] = adj[1:, 0] = 1
    g = sg.batch_from_adjs([adj] * copies)
    seeds = torch.arange(copies, device="cuda") * d
    for f in (1, 2, 3, 6):
        counts = np.zeros(d)
        s = sampling.DeviceBlockSampler([f])
        for salt in range(40):
            b, = s.sample_blocks(g, seeds, seed=SEED, salt=salt, gather=False)
            slots = g.in_ptr[seeds.long()].repeat_interleave(f).cpu().numpy()       # first slot of each seed
            src = b.src_ids[b.in_src.long()].cpu().numpy()
            dst = b.dst_ids.repeat_interleave(f).cpu().numpy()
            in_src = g.in_src.cpu().numpy()
            for u, v, beg in zip(src, dst, slots):
                pos = np.flatnonzero(in_src[beg:beg + d] == u)
                counts[pos[0]] += 1
        n = 40 * copies
        assert counts.sum() == n * f
        assert chisquare(counts, np.full(d, n * f / d)).pvalue > 1e-3, (f, counts)


def _oracle_blocks(mods, blocks):
    out = []
    for b in blocks:
        s_loc, d_loc = b.edges()
        out.append(mods["dgl_ops"].Block(s_loc.cpu(), d_loc.cpu(), b.num_src_nodes, b.num_dst_nodes))
    return out


@pytest.mark.parametrize("agg", ["pool", "mean", "gcn", "lstm"])
def test_forward_batch_on_device_blocks_vs_oracle(mods, agg):
    kind, cfg = FULL_MODELS["st_sage_3"]
    cfg = dict(cfg, aggregator_type=agg)
    scans = _scan_dicts(mods, 500, 4, ragged=True)
    g = _device_batch(mods, scans)
    y = torch.from_numpy(np.concatenate([s["labels"] for s in scans]).astype(np.int64))
    g.ndata["y"] = y.cuda()
    torch.manual_seed(0)
    onet = gnn_net(cfg)
    onet.init_like_reference()
    with torch.no_grad():
        for k, p in onet.named_parameters():
            if k.endswith("bias"):
                p.normal_(0, 0.05)
    net = mods["sm"].SAGENet(**cfg).cuda()
    net.load_state_dict(onet.state_dict(), strict=True)
    onet.eval()
    net.eval()
    seeds = torch.from_numpy(np.random.default_rng(4).permutation(g.num_nodes)[:64]).cuda()
    blocks = mods["sampling"].DeviceBlockSampler(net.sage.node_ks).sample_blocks(g, seeds, seed=SEED, salt=3)
    x = blocks[0].srcdata["fvs"]
    cw = torch.tensor([0.2] + [0.8] * 21)
    out, emb = net.forward_batch(blocks, x)
    yd = blocks[-1].dstdata["y"]
    mods["ops"].masked_cross_entropy(out, yd, cw.cuda(), rate=1.0).backward()
    ref_out, ref_emb = onet.forward_batch(_oracle_blocks(mods, blocks), x.cpu())
    onet64 = oracle_fp64(onet, _oracle_batch(mods, scans[:1]))[0]
    ref64, _ = onet64.forward_batch(_oracle_blocks(mods, blocks), x.cpu().double())
    torch.nn.functional.cross_entropy(ref64, yd.cpu(), weight=cw.double()).backward()
    assert rel_err(out.detach().cpu(), ref_out.detach()) < TOL, agg
    assert rel_err(emb.detach().cpu(), ref_emb.detach()) < TOL, agg
    if agg != "pool":
        assert_grads_match(net, onet64, GRAD_TOL, agg)
        return
    # max-pool routes each gradient to one arg-max slot: a near-tie decided differently in fp32 and fp64 moves it,
    # so pool takes the bar of test_gpu_parity's forward_batch test (3e-2 of the parameter's largest gradient)
    ograds = dict(onet64.named_parameters())
    gmax = max(float(q.grad.abs().max()) for q in ograds.values() if q.grad is not None)
    for k, p in net.named_parameters():
        r = ograds[k].grad
        if r is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        err = float((p.grad.cpu().double() - r).abs().max())
        assert err <= 3e-2 * float(r.abs().max()) or err <= 1e-6 * gmax, (k, err, float(r.abs().max()))


def test_one_synchronising_call_per_minibatch(mods):
    sampling = mods["sampling"]
    g, _ = _graph(mods, "ragged64")
    g.ndata["fvs"] = torch.randn(g.num_nodes, 1024, device="cuda")
    g.ndata["y"] = torch.randint(0, 22, (g.num_nodes,), device="cuda")
    nids = np.random.default_rng(5).permutation(g.num_nodes)[:int(0.3 * g.num_nodes)]
    loader = sampling.DeviceNodeDataLoader(g, nids, sampling.DeviceBlockSampler([2, 2, 2, 2]), batch_size=64,
                                           shuffle=True)
    it = iter(loader)
    next(it)                                                    # first call allocates the graph's scratch
    torch.cuda.synchronize()
    # the first window after turning the debug mode on carries a one-time synchronising call of its own (seen with
    # the torch sampler as well), so it is left out of the count
    with warnings.catch_warnings(record=True):
        torch.cuda.set_sync_debug_mode("warn")
        try:
            next(it)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    n_batches, syncs, messages = 0, [], []
    while True:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            torch.cuda.set_sync_debug_mode("warn")
            try:
                item = next(it)
            except StopIteration:
                break
            finally:
                torch.cuda.set_sync_debug_mode("default")
        n_batches += 1
        syncs.append(sum("synchroniz" in str(x.message) for x in w))
        messages += [str(x.message) for x in w]
        assert item[2][0].num_src_nodes > 0
    assert n_batches >= 3 and syncs == [1] * n_batches, (syncs, sorted(set(messages)))


def _write_settings(tmp_path, optimizer):
    from spgnn_b200.settings import PRESETS
    p = PRESETS["st_sage_3"]
    path = tmp_path / "st_sage_3_device.py"
    path.write_text("".join(f"{k} = {v!r}\n" for k, v in dict(p, OPTIMIZER=optimizer, EXP_NAME="exp",
                                                               MODEL_ROOT_PATH=str(tmp_path), SYNTHETIC_SCANS=3,
                                                               SYNTHETIC_RAGGED=True, TRAIN_BATCH_SIZE=2,
                                                               TRAIN_SAMPLE_SIZE=2, GCN_STEPS=3, LOG_STEPS=1,
                                                               NUM_EPOCHS=2, SAVE_EPOCHS=1).items()))
    return str(path)


@pytest.mark.parametrize("optimizer", [{"method": "torch.optim.SGD", "momentum": 0.9, "lr": 1e-3},
                                       {"method": "torch.optim.Adam", "lr": 1e-3}], ids=["FlatSGD", "FlatAdam"])
def test_gcntrain_sage_runs_on_the_device_sampler(tmp_path, monkeypatch, optimizer):
    from spgnn_b200 import job_runner, ops, runner, sampling
    from spgnn_b200.settings import Settings, get_callable_by_name
    calls = []
    orig = sampling.DeviceBlockSampler.sample_blocks
    monkeypatch.setattr(sampling.DeviceBlockSampler, "sample_blocks",
                        lambda self, *a, **k: calls.append(1) or orig(self, *a, **k))
    monkeypatch.setattr(sampling.MultiLayerNeighborSampler, "sample_blocks",
                        lambda *a, **k: pytest.fail("GCNTrainSAGE used the torch sampler"))
    torch.manual_seed(0)
    ops.manual_seed(0)
    path = _write_settings(tmp_path, optimizer)
    s = Settings(path)
    tr = get_callable_by_name(s.JOB_RUNNER_CLS)(s)
    assert isinstance(tr, job_runner.GCNTrainSAGE)
    assert isinstance(tr.optimizer, runner.FlatAdam if "Adam" in optimizer["method"] else runner.FlatSGD)
    hist = tr.run()
    assert len(hist) == 6 and np.isfinite(hist).all() and calls
    ck = sorted((tmp_path / "exp").glob("*.pth"))
    assert ck, "no checkpoint written"
    s2 = Settings(path)
    s2.RELOAD_CHECKPOINT_PATH = str(ck[-1])
    te = get_callable_by_name(s2.TEST_RUNNER_CLS)(settings_module=s2, output_path=str(tmp_path / "out"))
    for k, v in tr.model.state_dict().items():
        assert torch.equal(v, te.model.state_dict()[k]), k
    res = te.run()
    assert len(res) == 3
    r = next(iter(res.values()))
    assert r["decision"].shape == (21,) and 0.0 <= r["acc"] <= 1.0


def test_full_size_batch_invariants_and_repeatability(mods):
    """4096 synthetic trees (1.23 M nodes): 4096 seeds through fanouts [2, 2, 2, 2] and [2, -1, 2, 2]; the blocks meet
    the invariants (checked with torch on the device) and the same salt gives the same blocks twice."""
    from spgnn_b200 import synth_device
    g = synth_device.make_batch(0, 4096, ragged=False).graph
    assert g.num_nodes > 1_200_000
    seeds = torch.randperm(g.num_nodes, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))[:4096]
    for fanouts in ([2, 2, 2, 2], [2, -1, 2, 2]):
        s = mods["sampling"].DeviceBlockSampler(fanouts)
        a = s.sample_blocks(g, seeds, seed=SEED, salt=9, gather=False)
        b = s.sample_blocks(g, seeds, seed=SEED, salt=9, gather=False)
        for x, y in zip(a, b):
            for k in ("src_ids", "in_ptr", "in_src", "out_ptr", "out_dst", "out_slot"):
                assert torch.equal(getattr(x, k), getattr(y, k)), k
        dst_ids = seeds.long()
        for l in reversed(range(len(fanouts))):
            blk, f = a[l], fanouts[l]
            S = dst_ids.numel()
            assert torch.equal(blk.src_ids[:S], dst_ids)
            ex = blk.src_ids[S:]
            assert bool((ex[1:] > ex[:-1]).all())
            assert not bool(torch.isin(ex, dst_ids).any())
            deg = (g.in_ptr[dst_ids + 1] - g.in_ptr[dst_ids]).long()
            cnt = (blk.in_ptr[1:] - blk.in_ptr[:-1]).long()
            assert torch.equal(cnt, deg if f < 0 else deg.clamp(max=f))
            # every kept edge is a graph edge: (global src, global dst) pairs are in the graph's edge set
            src_g, dst_l = blk.src_ids[blk.in_src.long()], torch.repeat_interleave(torch.arange(S, device="cuda"), cnt)
            key = src_g * g.num_nodes + dst_ids[dst_l]
            gkey = torch.sort(g.src * g.num_nodes + g.dst)[0]
            at = torch.searchsorted(gkey, key).clamp(max=gkey.numel() - 1)
            assert torch.equal(gkey[at], key)
            assert torch.unique(key).numel() == key.numel()
            # out-CSR: stable transpose of the in-CSC
            E = blk.num_edges
            osl = blk.out_slot.long()
            assert torch.equal(torch.sort(osl)[0], torch.arange(E, device="cuda"))
            src_of_out = torch.repeat_interleave(torch.arange(blk.num_src_nodes, device="cuda"),
                                                 (blk.out_ptr[1:] - blk.out_ptr[:-1]).long())
            assert torch.equal(blk.in_src.long()[osl], src_of_out)
            assert torch.equal(dst_l[osl], blk.out_dst.long())
            assert torch.equal(torch.sort(src_of_out * E + osl)[0], src_of_out * E + osl)     # stable by source
            dst_ids = blk.src_ids
    assert bool((g._sample_pos == -1).all())
