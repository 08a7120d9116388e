"""Adam and AdamW on the device: spgnn_adam_step against an fp64 restatement of torch's update, runner.FlatAdam
against torch.optim.Adam / AdamW and their state dicts both ways, CUDA-graph replay of an Adam step, and the
settings-driven runners with OPTIMIZER = torch.optim.Adam / AdamW."""
import copy

import numpy as np
import pytest
import torch

from helpers import FULL_MODELS, TINY_MODELS, rel_err

pytestmark = pytest.mark.gpu

PAD = 8                       # guard elements on each side of the bucket (keeps the bucket 16-byte aligned)
GUARD = 7.25
SPGNN3 = 2_501_078


def _sizes(L):
    """Parameter sizes of a bucket of L floats: unaligned offsets, and for SPGNN3 the parameters of st_pgat_spgnn_3."""
    if L == SPGNN3:
        from spgnn_b200 import models as sm
        sizes = [p.numel() for p in sm.GATPositionSPGNNNet(**FULL_MODELS["st_pgat_spgnn_3"][1]).parameters()]
    else:
        sizes = {1: [1], 7: [1, 2, 4], 4097: [1, 4096]}[L]
    assert sum(sizes) == L
    return sizes


def _table(offsets, live, chunk):
    rows = []
    for i in live:
        o, k = offsets[i]
        for c in range(0, k, chunk):
            rows += [PAD + o + c, min(chunk, k - c), i]
    return torch.tensor(rows + list(live), dtype=torch.int64, device="cuda"), len(rows) // 3


# (bucket length, AdamW, amsgrad, maximize, weight_decay, betas, steps, elements per chunk of the launch table)
KERNEL_CASES = [
    (1, False, False, False, 0.0, (0.9, 0.999), 1, 4096),
    (7, True, True, False, 0.05, (0.5, 0.9), 50, 3),
    (7, False, False, True, 0.02, (0.9, 0.999), 50, 4096),
    (4097, True, False, True, 0.0, (0.9, 0.999), 50, 1000),
    (4097, False, True, False, 0.1, (0.5, 0.9), 20, 4096),
    (SPGNN3, False, False, False, 0.0, (0.9, 0.999), 12, 4096),
    (SPGNN3, True, True, True, 0.01, (0.9, 0.999), 4, 4096),
]


@pytest.mark.parametrize("L,decoupled,amsgrad,maximize,wd,betas,steps,chunk", KERNEL_CASES)
def test_adam_kernel_matches_fp64_restatement(L, decoupled, amsgrad, maximize, wd, betas, steps, chunk):
    """spgnn_adam_step called directly, step after step: every live element against the update restated in fp64
    from the kernel's previous state, with t read from the per-parameter device counts; parameters without a
    gradient on a step keep their values and count bit for bit; guard values around the bucket and the gradient
    buffer are never written."""
    from spgnn_b200._lib import lib, ptr, stream
    lr, eps = 1e-2, 1e-8
    b1, b2 = betas
    sizes = _sizes(L)
    offsets = list(zip(np.cumsum([0] + sizes[:-1]).tolist(), sizes))
    P = len(sizes)
    rng = np.random.default_rng(L + steps)
    n = L + 2 * PAD

    def guarded(inside):
        a = np.full(n, GUARD, np.float32)
        a[PAD:PAD + L] = inside
        return a

    host = {"p": guarded(rng.standard_normal(L).astype(np.float32)), "m": guarded(0.0), "v": guarded(0.0),
            "x": guarded(0.0)}
    dev = {k: torch.from_numpy(a).cuda() for k, a in host.items()}
    counts = torch.full((P + 2,), 12345, dtype=torch.int64, device="cuda")
    counts[:P] = 0
    ref_t = np.zeros(P, np.int64)
    sl = slice(PAD, PAD + L)
    par = np.repeat(np.arange(P), sizes)
    for s in range(steps):
        live = [j for j in range(P) if (3 * j + s) % 7 != 2] or [0]
        gh = guarded(rng.standard_normal(L).astype(np.float32))
        gh[PAD + rng.integers(0, L, max(1, L // 50))] = 0.0                  # some zero gradients
        gd = torch.from_numpy(gh).cuda()
        table, n_chunks = _table(offsets, live, chunk)
        before = {k: t.cpu().numpy() for k, t in dev.items()}
        lib().adam_step(ptr(dev["p"]), ptr(gd), ptr(dev["m"]), ptr(dev["v"]), ptr(dev["x"]) if amsgrad else None,
                        ptr(counts), ptr(table), n_chunks, table.data_ptr() + 24 * n_chunks, len(live), lr, b1, b2,
                        eps, wd, int(amsgrad), int(maximize), int(decoupled), stream())
        after = {k: t.cpu().numpy() for k, t in dev.items()}
        ref_t[live] += 1
        assert counts[:P].tolist() == ref_t.tolist() and counts[P:].tolist() == [12345, 12345], s
        assert np.array_equal(gd.cpu().numpy(), gh)
        # fp64 restatement of torch's _single_tensor_adam on the live elements
        on = np.isin(par, live)
        t = np.maximum(ref_t[par], 1).astype(np.float64)                     # parameters never live yet: not compared
        p, m, v, x = (before[k][sl].astype(np.float64) for k in ("p", "m", "v", "x"))
        g = gh[sl].astype(np.float64) * (-1.0 if maximize else 1.0)
        if wd:
            if decoupled:
                p = p * (1.0 - lr * wd)
            else:            # torch hands weight_decay to its fp32 kernel as an fp32 scalar: where g ~ -wd*p its
                g = g + float(np.float32(wd)) * p          # rounding is all that is left of g, so restate it exactly
        m_ref = b1 * m + (1.0 - b1) * g
        v_ref = b2 * v + (1.0 - b2) * g * g
        x_ref = np.maximum(x, v_ref)
        den = np.sqrt(x_ref if amsgrad else v_ref) / np.sqrt(1.0 - b2 ** t) + eps
        p_ref = p - lr / (1.0 - b1 ** t) * m_ref / den
        pa, ma, va, xa = (after[k][sl].astype(np.float64) for k in ("p", "m", "v", "x"))
        d = np.abs(p_ref - before["p"][sl])[on].max()
        assert (np.abs(pa - p_ref)[on] <= 1e-5 * d + 4e-7 * np.abs(p_ref)[on]).all(), s
        assert (np.abs(ma - m_ref)[on] <= 1e-6 * (np.abs(m) + np.abs(g))[on]).all(), s
        assert (np.abs(va - v_ref)[on] <= 1e-6 * v_ref[on] + 1e-30).all(), s
        if amsgrad:
            assert (np.abs(xa - x_ref)[on] <= 1e-6 * x_ref[on] + 1e-30).all(), s
        for k in dev:
            assert np.array_equal(after[k][sl][~on], before[k][sl][~on]), (s, k)              # skipped parameters
            assert (after[k][:PAD] == GUARD).all() and (after[k][PAD + L:] == GUARD).all(), (s, k)


def test_adam_kernel_refuses_bad_arguments_and_writes_nothing():
    from spgnn_b200._lib import SpgnnError, lib, ptr, stream
    p = torch.ones(16, device="cuda")
    g, m, v, x = (torch.ones(16, device="cuda") for _ in range(4))
    counts = torch.zeros(1, dtype=torch.int64, device="cuda")
    table = torch.tensor([0, 16, 0, 0], dtype=torch.int64, device="cuda")

    def call(p_=ptr(p), x_=None, b1=0.9, b2=0.999, eps=1e-8, amsgrad=0):
        lib().adam_step(p_, ptr(g), ptr(m), ptr(v), x_, ptr(counts), ptr(table), 1, table.data_ptr() + 24, 1, 1e-3,
                        b1, b2, eps, 0.0, amsgrad, 0, 0, stream())

    bad = [dict(b1=1.0), dict(b2=1.0), dict(b1=-0.1), dict(b2=float("nan")), dict(eps=-1e-8), dict(x_=ptr(x)),
           dict(amsgrad=1), dict(p_=ptr(p) + 4)]
    for kw in bad:
        with pytest.raises(SpgnnError):
            call(**kw)
    torch.cuda.synchronize()
    assert (p == 1).all() and int(counts) == 0
    call(x_=ptr(x), amsgrad=1)
    assert int(counts) == 1 and not (p == 1).all()


# ------------------------------------------------------------------------------------------ FlatAdam vs torch
OPT_CASES = [("Adam", {}), ("Adam", dict(weight_decay=1e-2, amsgrad=True)), ("AdamW", {}),
             ("AdamW", dict(amsgrad=True, maximize=True, betas=(0.5, 0.9), eps=1e-6, weight_decay=0.1))]
DEAD = 1                                                 # this parameter never receives a gradient


def _feed(pairs, step):
    """Identical gradients to every optimiser's parameters; some parameters get none on some steps."""
    for i, ps in enumerate(zip(*pairs)):
        if i == DEAD or (3 * i + step) % 7 == 2:
            continue
        g = torch.randn(ps[0].shape, generator=torch.Generator().manual_seed(1000 * step + i)).cuda()
        for p in ps:
            p.grad = g.clone()


def _torch_opt(name, params, kw):
    cls = getattr(torch.optim, name)
    return cls(params, foreach=False, **kw)


def _flat_opt(name, params, kw):
    from spgnn_b200 import runner
    return runner.FlatAdam(params, decoupled=name == "AdamW", **dict(dict(weight_decay=1e-2) if name == "AdamW"
                                                                     else {}, **kw))


def _assert_same(flat, ref_opt, dev_p, ref_p, tag):
    for i, (d, r) in enumerate(zip(dev_p, ref_p)):
        assert torch.allclose(d.detach(), r.detach(), atol=1e-6, rtol=1e-5), (tag, i)
    sd = flat.state_dict()
    assert set(sd["state"]) == {i for i, r in enumerate(ref_p) if r in ref_opt.state}, tag
    for i, st in sd["state"].items():
        rs = ref_opt.state[ref_p[i]]
        assert set(st) == set(rs) and float(st["step"]) == float(rs["step"]), (tag, i)
        for k in st:
            if k != "step":
                assert torch.allclose(st[k].cuda(), rs[k], atol=1e-6, rtol=1e-5), (tag, i, k)


def _tiny_net():
    from spgnn_b200 import models as sm
    torch.manual_seed(0)
    net = sm.GATPositionSPGNNNet(**TINY_MODELS["spgnn3"][1]).cuda()
    net.init()
    return net


@pytest.mark.parametrize("name,kw", OPT_CASES)
def test_flat_adam_matches_torch_and_state_dicts_round_trip(name, kw):
    """runner.FlatAdam against torch.optim.Adam / AdamW(foreach=False) on a small SPGNN-3 net and its twin, fed
    identical gradients for 10 steps under an ExponentialLR decay, with one parameter that never gets a gradient
    and others that miss some steps (no step advance, no decay); then each optimiser's state dict is loaded into
    the other kind and both continue 5 steps in lockstep."""
    net = _tiny_net()
    twin = copy.deepcopy(net)
    ref_p, dev_p = list(net.parameters()), list(twin.parameters())
    ref_opt = _torch_opt(name, ref_p, kw)
    sched = torch.optim.lr_scheduler.ExponentialLR(ref_opt, gamma=0.9)
    flat = _flat_opt(name, dev_p, kw)
    assert flat.decoupled == (name == "AdamW") and flat.weight_decay == ref_opt.param_groups[0]["weight_decay"]
    for step in range(10):
        ref_opt.zero_grad()
        flat.zero_grad()
        _feed((ref_p, dev_p), step)
        ref_opt.step()
        flat.step()
        sched.step()
        flat.set_lr(flat.lr * 0.9)
        _assert_same(flat, ref_opt, dev_p, ref_p, ("lockstep", step))
    assert DEAD not in flat.state_dict()["state"] and int(flat.step_t[DEAD]) == 0
    # device -> torch
    p_a = [torch.nn.Parameter(p.detach().clone()) for p in dev_p]
    torch_a = _torch_opt(name, p_a, kw)
    sd = flat.state_dict()
    assert sd["param_groups"][0]["decoupled_weight_decay"] == (name == "AdamW")
    torch_a.load_state_dict(sd)
    # torch -> device, one count given as a number rather than a tensor
    net_b = copy.deepcopy(net)
    p_b = list(net_b.parameters())
    flat_b = _flat_opt(name, p_b, {})
    tsd = copy.deepcopy(ref_opt.state_dict())           # its state entries are the optimiser's own dicts
    tsd["state"][0]["step"] = float(tsd["state"][0]["step"])
    flat_b.load_state_dict(tsd)
    assert flat_b.amsgrad == bool(kw.get("amsgrad")) and flat_b.lr == ref_opt.param_groups[0]["lr"]
    _assert_same(flat_b, ref_opt, p_b, ref_p, "loaded from torch")
    for step in range(10, 15):
        for o in (flat, torch_a, ref_opt, flat_b):
            o.zero_grad()
        _feed((dev_p, p_a, ref_p, p_b), step)
        for o in (flat, torch_a, ref_opt, flat_b):
            o.step()
        _assert_same(flat, torch_a, dev_p, p_a, ("device -> torch", step))
        _assert_same(flat_b, ref_opt, p_b, ref_p, ("torch -> device", step))


def test_flat_adam_is_two_launches_per_step_and_builds_its_table_once():
    from spgnn_b200._lib import lib
    net = _tiny_net()
    params = list(net.parameters())
    flat = _flat_opt("Adam", params, {})
    for step in range(3):
        flat.zero_grad()
        for p in params:
            p.grad = torch.ones_like(p)
        n0 = int(lib().launch_count())
        flat.step()
        assert int(lib().launch_count()) - n0 == 2
    assert len(flat._tables) == 1
    table, n_chunks = flat._tables[tuple(range(len(params)))]
    assert n_chunks == sum(-(-p.numel() // flat.CHUNK) for p in params)


# ------------------------------------------------------------------------------------------ CUDA graph
def test_cuda_graph_replays_advance_the_adam_step_counts():
    """runner.GraphedTrainStep with FlatAdam on a 6-tree batch, no randomness: W warm-up steps and K replays equal
    W + K eager steps, and the device counts read W + K.  The same replays with the count reset before each one —
    what a step count frozen into the graph as a kernel argument would do — move the parameters differently.
    eps = 1e-2 keeps the comparison to what the step count changes: with eps = 1e-8 Adam turns the last-bit noise
    of gradients that cancel to ~0 (sums whose atomics reorder between runs) into steps of +-lr."""
    from spgnn_b200 import models as sm, ops, pe as spe, runner, synth_device
    kind, cfg = FULL_MODELS["st_pgat_spgnn_3"]
    g = synth_device.make_batch(0, 6, ragged=True).graph
    spe.distance_pos_enc(g, pos_enc_dim=39)
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device="cuda")
    W, K = 3, 5

    def fresh():
        torch.manual_seed(0)
        net = sm.GATPositionSPGNNNet(**dict(cfg, feat_drop=0.0, attn_drop=0.0)).cuda()
        net.init()
        net.train()
        net.set_gcn_only()
        ops.manual_seed(3)
        return net, runner.FlatAdam(net.parameters(), lr=5e-3, eps=1e-2)

    net_e, opt_e = fresh()
    p0 = opt_e.flat_p.clone()
    eager = [float(runner.train_step(net_e, g, opt_e, cw, 1.0).item()) for _ in range(W + K)]
    net_g, opt_g = fresh()
    gs = runner.GraphedTrainStep(net_g, g, opt_g, cw, 1.0, warmup=W)
    replayed = [float(gs().item()) for _ in range(K)]
    gs.reset_salt()
    assert np.allclose(replayed, eager[W:], rtol=2e-4), (replayed, eager)
    counts = opt_g.step_t.cpu()
    assert torch.equal(counts, opt_e.step_t.cpu()) and int(counts.max()) == W + K
    assert bool(((counts == 0) | (counts == W + K)).all())
    err = rel_err((opt_g.flat_p - p0).cpu(), (opt_e.flat_p - p0).cpu())
    assert err < 1e-3, err
    net_f, opt_f = fresh()
    gf = runner.GraphedTrainStep(net_f, g, opt_f, cw, 1.0, warmup=W)
    captured = opt_f.step_t.clone()
    for _ in range(K):
        opt_f.step_t.copy_(captured)                     # every replay takes t = W + 1
        gf()
    gf.reset_salt()
    err_frozen = rel_err((opt_f.flat_p - p0).cpu(), (opt_e.flat_p - p0).cpu())
    assert err_frozen > 2e-2 and err_frozen > 20 * err, (err_frozen, err)


# ------------------------------------------------------------------------------------------ settings-driven runners
def _settings_file(tmp_path, optimizer, preset="st_gat_3", scans=3, steps=16):
    from spgnn_b200.settings import PRESETS, Settings
    pr = PRESETS[preset]
    text = "\n".join([
        f"EXP_NAME = 'adam'", f"MODEL_ROOT_PATH = {str(tmp_path)!r}", f"MODEL = {pr['MODEL']!r}",
        f"JOB_RUNNER_CLS = {pr['JOB_RUNNER_CLS']!r}", f"TEST_RUNNER_CLS = {pr['TEST_RUNNER_CLS']!r}",
        f"SAMPLING_RATE = {pr['SAMPLING_RATE']!r}", f"OPTIMIZER = {optimizer!r}",
        "SCHEDULER = {'method': 'torch.optim.lr_scheduler.ExponentialLR', 'gamma': 0.9}",
        f"SYNTHETIC_SCANS = {scans}", "SYNTHETIC_RAGGED = True",
        f"TRAIN_BATCH_SIZE = {scans}", f"TRAIN_SAMPLE_SIZE = {scans}", f"GCN_STEPS = {steps}",
        "LOG_STEPS = 1", "NUM_EPOCHS = 2", "SAVE_EPOCHS = 1", ""])
    f = tmp_path / f"{preset}_{optimizer['method'].rpartition('.')[2].lower()}.py"
    f.write_text(text)
    return Settings(str(f))


@pytest.mark.parametrize("optimizer", [{"method": "torch.optim.Adam", "lr": 1e-3},
                                       {"method": "torch.optim.AdamW", "amsgrad": True}])
def test_settings_file_with_adam_trains_checkpoints_resumes_and_tests(tmp_path, optimizer):
    """An exp_settings file naming torch.optim.Adam / AdamW: two epochs of 16 graphed steps with ExponentialLR,
    checkpoints in torch's Adam layout, a resumed run restores exp_avg, the step counts and the learning rate, and
    the test runner reads the checkpoint.  Unknown Adam keys and other optimisers are refused."""
    from spgnn_b200 import job_runner, ops, runner
    from spgnn_b200.settings import get_callable_by_name
    torch.manual_seed(0)
    ops.manual_seed(0)
    s = _settings_file(tmp_path, optimizer)
    tr = get_callable_by_name(s.JOB_RUNNER_CLS)(s)
    opt = tr.optimizer
    assert isinstance(opt, runner.FlatAdam) and opt.decoupled == optimizer["method"].endswith("AdamW")
    assert opt.lr == 1e-3 and opt.weight_decay == (0.01 if opt.decoupled else 0.0)       # torch's defaults
    assert opt.amsgrad == bool(optimizer.get("amsgrad"))
    hist = tr.run()
    assert len(hist) == 2 * (16 - 3) and np.isfinite(hist).all()      # the 3 warm-up steps of a graph are not logged
    assert np.mean(hist[-4:]) < np.mean(hist[:4])
    assert tr.epoch_n == 2 and abs(opt.lr - 1e-3 * 0.9 ** 2) < 1e-15
    assert int(opt.step_t.max()) == 2 * 16
    ck = max((tmp_path / "adam").glob("*.pth"), key=lambda p: int(p.stem))
    state = torch.load(ck, weights_only=False)
    osd = state["optimizer_dict"]
    assert float(osd["state"][0]["step"]) == 2 * 16 and osd["state"][0]["step"].dtype == torch.float32
    assert ("max_exp_avg_sq" in osd["state"][0]) == opt.amsgrad
    assert abs(state["scheduler_dict"]["_last_lr"][0] - 1e-3 * 0.9) < 1e-15

    s2 = _settings_file(tmp_path, optimizer)
    s2.RELOAD_CHECKPOINT, s2.RELOAD_CHECKPOINT_PATH = True, str(ck)
    s2.RELOAD_DICT_LIST = ["model_dict", "metric", "optimizer_dict", "scheduler_dict"]
    tr2 = get_callable_by_name(s2.JOB_RUNNER_CLS)(s2)
    o2 = tr2.optimizer
    assert abs(o2.lr - 1e-3 * 0.9) < 1e-15 and tr2.epoch_n == 1
    assert torch.equal(o2.exp_avg, opt.exp_avg) and torch.equal(o2.exp_avg_sq, opt.exp_avg_sq)
    assert torch.equal(o2.step_t, opt.step_t) and torch.equal(o2.flat_p, opt.flat_p)
    if opt.amsgrad:
        assert torch.equal(o2.max_exp_avg_sq, opt.max_exp_avg_sq)
    losses = tr2.train_batch([tr2.source(u) for u in tr2.source.uids], steps=2)
    assert np.isfinite(losses).all() and int(o2.step_t.max()) == 2 * 16 + 2

    s3 = _settings_file(tmp_path, optimizer)
    s3.RELOAD_CHECKPOINT_PATH = str(ck)
    te = get_callable_by_name(s3.TEST_RUNNER_CLS)(settings_module=s3, output_path=str(tmp_path / "out"))
    res = te.run()
    assert len(res) == 3 and (tmp_path / "out" / "gnn_predictions.pkl").exists()

    for bad in (dict(optimizer, foreach=False), dict(optimizer, fused=True), {"method": "torch.optim.RMSprop"}):
        with pytest.raises(job_runner.SpgnnError):
            get_callable_by_name(s.JOB_RUNNER_CLS)(_settings_file(tmp_path, bad))


def test_sage_runner_trains_with_adam(tmp_path):
    """GCNTrainSAGE's neighbour-sampled mini-batches: one FlatAdam step per mini-batch."""
    from spgnn_b200 import job_runner, runner
    from spgnn_b200.settings import get_callable_by_name
    torch.manual_seed(0)
    s = _settings_file(tmp_path, {"method": "torch.optim.Adam"}, preset="st_sage_3", scans=2, steps=2)
    tr = get_callable_by_name(s.JOB_RUNNER_CLS)(s)
    assert isinstance(tr, job_runner.GCNTrainSAGE) and isinstance(tr.optimizer, runner.FlatAdam)
    losses = tr.train_batch([tr.source(u) for u in tr.source.uids], steps=2, max_minibatches=3)
    assert len(losses) == 2 and np.isfinite(losses).all()
    assert 2 <= int(tr.optimizer.step_t.max()) <= 6


# ------------------------------------------------------------------------------------------ full size
def test_adam_update_at_4096_trees_is_bit_identical_run_to_run():
    """st_pgat_spgnn_3 on 4096 trees with FlatAdam: a training step from the same seeds gives the same loss twice
    (the forward and backward only reorder the atomics of the bias-gradient sums), and the Adam update of the next
    step, applied again from the same state to the same gradient, is bit-identical."""
    from spgnn_b200 import models as sm, ops, pe as spe, runner, synth_device
    big = synth_device.make_batch(0, 4096, ragged=True)
    spe.distance_pos_enc(big.graph, pos_enc_dim=39)
    cw = torch.tensor(runner.CLASS_WEIGHTS_22, device="cuda")
    losses = []
    for _ in range(2):
        torch.manual_seed(3)
        net = sm.GATPositionSPGNNNet(**FULL_MODELS["st_pgat_spgnn_3"][1]).cuda()
        net.init()
        net.train()
        net.set_gcn_only()
        opt = runner.FlatAdam(net.parameters(), lr=1e-3)
        ops.manual_seed(77)
        losses.append(float(runner.train_step(net, big.graph, opt, cw, 0.15).item()))
    assert np.isfinite(losses).all() and abs(losses[0] - losses[1]) <= 1e-6 * abs(losses[0])
    state = (opt.flat_p, opt.exp_avg, opt.exp_avg_sq, opt.step_t)
    snap = [t.clone() for t in state]
    runner.train_step(net, big.graph, opt, cw, 0.15)     # afterwards p.grad is still the gradient's bucket slot
    first = [t.clone() for t in state]
    for t, v in zip(state, snap):
        t.copy_(v)
    opt.step()
    for a, b in zip(first, state):
        assert torch.equal(a, b)
    assert int(opt.step_t.max()) == 2 and not torch.equal(first[0], snap[0])
