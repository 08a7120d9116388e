"""CPU-side checks (no GPU): the C-ABI library loads and exports every declared symbol, the host generator and
the host-side plumbing behave, and the product refuses to run without CUDA instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_loads_and_exports_every_header_symbol():
    from spgnn_b200 import build
    path = build.build()
    assert os.path.exists(path)
    from spgnn_b200._lib import lib, parse_header
    L = lib()
    protos = parse_header()
    names = {n for n, _, _ in protos}
    header = open(os.path.join(ROOT, "include", "spgnn_b200.h")).read()
    declared = set(re.findall(r"\b(spgnn_[a-z0-9_]+)\s*\(", header))
    assert declared == names and len(names) >= 35
    dll = ctypes.CDLL(path)
    for n in names:
        assert hasattr(dll, n), n
    assert L.abi_version() == 1
    assert L.scan_ws_bytes(10) > 0 and L.batch_ws_bytes(1000, 3000) > 0     # pure host helpers, no GPU needed


def test_library_is_sm100a_with_lineinfo():
    import subprocess
    from spgnn_b200 import build
    from spgnn_b200._lib import LIB_PATH
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")       # the toolkit the library was built with
    out = subprocess.run([cuobjdump, "--list-elf", LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback():
    from spgnn_b200 import graph as sg, ops
    from spgnn_b200._lib import SpgnnError
    if torch.cuda.is_available():
        pytest.skip("only meaningful without a GPU")
    with pytest.raises(SpgnnError):
        sg.from_adj(np.eye(3, dtype=np.uint8))
    with pytest.raises(SpgnnError):
        ops.linear(torch.zeros(2, 2), torch.zeros(2, 2))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "spgnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f


def test_synth_generator_invariants():
    from spgnn_b200 import synth
    for ragged in (False, True):
        for t in (0, 5, 123456):
            s = synth.make_scan(t, ragged=ragged, fv_dim=8)
            n = s.adj.shape[0]
            assert n % 2 == 1 and (n == 301 if not ragged else 241 <= n <= 361)
            assert np.array_equal(s.adj, s.adj.T) and np.all(np.diag(s.adj) == 1)
            assert s.adj.sum() == n + 2 * (n - 1)                         # tree ∪ I
            assert np.all(s.parent[1:] < np.arange(1, n))                 # parent index < child index
            assert sorted(s.labels[s.labels > 0].tolist()) == list(range(1, 22))
            assert s.fvs.min() >= 0 and s.fvs.dtype == np.float32
            deg = s.adj.sum(1) - 1
            assert deg[0] == 2 and set(np.unique(deg[1:])) <= {1, 3}       # full bifurcation
    a, b = synth.make_scan(3, fv_dim=8), synth.make_scan(3, fv_dim=8)
    assert np.array_equal(a.adj, b.adj) and np.array_equal(a.fvs, b.fvs)
    # Philox known-answer (Random123 kat: counter=0,key=0)
    w = synth.philox4x32(0, 0, 0, 0, 0, 0)
    assert [int(x) for x in w] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


def test_models_construct_with_reference_settings_and_dgl_state_dict_names():
    from spgnn_b200 import models as sm
    from helpers import FULL_MODELS
    counts = {"st_pgat_spgnn_3": 2_501_078, "st_gat_3": 1_931_926, "st_gat_6": 2_031_382, "st_gat_6_nr": 1_031_958,
              "st_gcn_3": 392_662, "st_gin_3": 1_537_955, "st_sage_3": 1_897_366,
              "st_pgat_spgnnnl_3": 2_161_558}
    cls = {"gat": sm.GATNet, "gcn": sm.GCNNet, "gin": sm.GINNet, "sage": sm.SAGENet, "spgnn": sm.GATPositionSPGNNNet}
    for name, (kind, cfg) in FULL_MODELS.items():
        # the CNN-trunk keys of settings.MODEL are accepted and ignored
        net = cls[kind](n_layers=3, in_ch_list=[1, 32, 64, 128], base_ch_list=[24, 32, 64, 128],
                        end_ch_list=[32, 64, 128, 256], kernel_sizes=[3, 3, 3, 3],
                        checkpoint_layers=[0, 1, 1, 0, 1, 1, 1], padding_list=[(1, 1, 1)] * 4,
                        conv_strides=[[1, 2]] * 3, dropout=0.0, spatial_size=10, norm_method="bn", act_method="relu",
                        **cfg)
        assert sum(p.numel() for p in net.parameters()) == counts[name], name     # SURVEY.md §8a
        net.set_gcn_only()
        assert all(p.requires_grad for p in net.parameters())
    from oracle import models as om
    kind, cfg = FULL_MODELS["st_pgat_spgnn_3"]
    assert set(om.GNNNet(kind, cfg).state_dict()) == set(sm.GATPositionSPGNNNet(**cfg).state_dict())


def test_settings_loader_and_name_mapping(tmp_path):
    from spgnn_b200.settings import PRESETS, Settings, get_callable_by_name
    from spgnn_b200 import job_runner, models
    f = tmp_path / "st_custom.py"
    f.write_text("EXP_NAME = 'x'\nGCN_STEPS = 7\nlower = 1\nPOS_ENC_DIM = 39\n"
                 "JOB_RUNNER_CLS = 'apps.airways.labeling_base.job_runner.GCNTrain'\n"
                 "TEST_RUNNER_CLS = 'job_runner.GCNTestLSPE'\n"
                 "MODEL = {'method': 'models.GATPositionLSPENet', 'fv_dim': 32}\n")
    s = Settings(str(f))
    assert s.GCN_STEPS == 7 and s.is_overridden("GCN_STEPS") and not hasattr(s, "lower")
    assert s.TRAIN_BATCH_SIZE == 64 and not s.is_overridden("TRAIN_BATCH_SIZE")        # reference default
    assert get_callable_by_name(s.JOB_RUNNER_CLS) is job_runner.GCNTrain               # absent module in the reference
    assert get_callable_by_name(s.TEST_RUNNER_CLS) is job_runner.GCNTestSPGNN          # absent *LSPE names
    assert get_callable_by_name(s.MODEL["method"]) is models.GATPositionSPGNNNet
    assert get_callable_by_name("initializer.HeNorm") is job_runner.HeNorm
    assert get_callable_by_name("torch.optim.SGD") is torch.optim.SGD
    p = Settings("st_pgat_spgnn_3")
    assert p.MODEL["pos_enc_dim"] == 39 and p.SAMPLING_RATE == 0.15 and set(PRESETS) >= {"st_gat_3", "st_gat_6_nr"}
    cw = [p.CLASS_WEIGHTS[k] for k in sorted(p.CLASS_WEIGHTS.keys())][1:]
    assert len(cw) == 22 and cw[0] == 0.2 and set(cw[1:]) == {0.8}                     # job_runner.py:1867


def test_weight_gradient_launch_plan_is_sane():
    """Host-only planner of the dW GEMM (spgnn_planes_linear_bwd_weight_plan): every CTA fits one wave, the splits
    cover all rows, and the gradient goes on the M side exactly where that saves half-empty accumulators."""
    from spgnn_b200._lib import lib
    L = lib()
    M = 4096 * 301
    shapes = {"gat0": (1028, 1024, 39), "gat1": (516, 512, 256), "gat2": (260, 256, 128), "pgnn0": (514, 39, 0),
              "pgnn1": (258, 256, 0), "pgnn2": (130, 128, 0), "head": (22, 1024, 0), "gat_out_head": (1024, 192, 192)}
    plans = {}
    split_sources = {}
    for name, (N, K1, K2) in shapes.items():
        out = (ctypes.c_int32 * 9)()
        assert L.planes_linear_bwd_weight_plan(M, N, K1, K2, out, 9) == 9
        swap, npt, nqt, splits, ctas, rows, npb, nqb, split = list(out)
        plans[name], split_sources[name] = swap, split
        assert 1 <= ctas <= 148 and ctas == npt * nqt * splits
        assert rows % 32 == 0 and rows * splits >= M > rows * (splits - 1)
        assert npt == -(-npb // 4) and nqt == -(-nqb // 4)
        # split == 1: one launch per source, the plan is the first one's (X1 alone)
        xb = -(-K1 // 64) + (-(-K2 // 64) if K2 and not split else 0)
        yb = -(-N // 64)
        assert (npb, nqb) == ((yb, xb) if swap else (xb, yb))
    # X = [Ax_h | x] is 3 + 3 blocks: on the M side it fills 1.5 accumulators per tile, dC (16 blocks) fills them all
    assert plans["gat_out_head"] == 1 and plans["gat0"] == 0
    # gat0's X = [fvs | pos_enc] is 16 + 1 blocks: 17 x 17 blocks tile into 125 CTAs with half-empty accumulators, the
    # two sources on their own into 140 CTAs of full tiles; the evenly tiling concatenations stay one launch
    assert split_sources["gat0"] == 1 and not any(split_sources[k] for k in ("gat1", "gat2", "gat_out_head"))
    small = (ctypes.c_int32 * 8)()
    assert L.planes_linear_bwd_weight_plan(300, 48, 64, 0, small, 8) == 8 and small[3] == 1 and small[4] == 1


def test_descriptor_structs_match_the_library_layout():
    """The ctypes mirrors of spgnn_gat_layer / spgnn_gat_wide (stack.py) must have the size the C side compiled."""
    from spgnn_b200 import stack
    from spgnn_b200._lib import lib
    assert int(lib().gat_layer_sizeof()) == ctypes.sizeof(stack._Layer)
    assert int(lib().gat_wide_sizeof()) == ctypes.sizeof(stack._Wide)
    stack._checked = False
    stack._check_abi()
    assert stack._checked


def test_flat_sgd_gathers_gradients_into_one_bucket():
    """FlatSGD host logic (no kernels): parameters become views of one buffer, gradients are gathered into the flat
    bucket by one multi-tensor copy, parameters without a gradient contribute zeros, zero_grad drops gradients."""
    import torch
    from spgnn_b200.runner import FlatSGD
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 2), torch.nn.Linear(7, 1))   # [2] is unused
    before = [p.detach().clone() for p in net.parameters()]
    opt = FlatSGD(net.parameters(), lr=0.1)
    assert opt.numel == sum(b.numel() for b in before)
    for p, b in zip(net.parameters(), before):
        assert torch.equal(p.detach(), b) and p.grad is None
        assert opt.flat_p.data_ptr() <= p.data_ptr() < opt.flat_p.data_ptr() + 4 * opt.numel
    net[1](net[0](torch.randn(4, 5))).square().sum().backward()
    ref = [p.grad.clone() if p.grad is not None else torch.zeros_like(p) for p in net.parameters()]
    opt.flat_g.fill_(7.0)                                   # stale content must not survive
    live = opt._gather()
    assert live == [0, 1, 2, 3]                             # the unused Linear(7, 1) has no gradient: skipped like torch
    assert torch.equal(opt.flat_g, torch.cat([r.reshape(-1) for r in ref]))
    for i, (p, v) in enumerate(zip(net.parameters(), opt.g_views)):
        assert (p.grad.data_ptr() == v.data_ptr()) if i in live else (p.grad is None)
    assert opt._gather() == live                            # idempotent once p.grad is the slot
    assert torch.equal(opt.flat_g, torch.cat([r.reshape(-1) for r in ref]))
    # update ranges: one contiguous run over the four live parameters, first step; the skipped ones keep no buffer
    assert opt._runs(live) == [(0, sum(b.numel() for b in before[:4]), True)]
    assert opt.has_buf == [True] * 4 + [False] * 2
    assert opt._runs([0, 1, 3]) == [(0, 18, False), (24, 2, False)]
    sd = opt.state_dict()
    assert sd["param_groups"][0]["params"] == list(range(6)) and sd["param_groups"][0]["lr"] == 0.1
    opt.zero_grad()
    assert all(p.grad is None for p in net.parameters())


def test_bench_workloads_and_launch_list_summary():
    """bench.py's preset table covers every BASELINE.json config, the headline keeps its metric name, and the
    committed ncu launch list summarises to the step the docs quote (one training step = 109 launches)."""
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import bench
    for name, kind in (("st_pgat_spgnn_3", "spgnn"), ("st_gat_3", "gat"), ("st_gat_6", "gat"), ("st_gat_6_nr", "gat"),
                       ("st_gcn_3", "gcn"), ("st_gin_3", "gin"), ("st_sage_3", "sage")):
        model, k, method, rate = bench.workload(name)
        assert k == kind and "method" not in model and 0.0 < rate < 1.0 and method.startswith("models.")
    assert bench.metric_name(bench.HEADLINE) == "spgnn3_train_graphs_per_s"
    assert bench.metric_name("st_gcn_3") == "st_gcn_3_train_graphs_per_s"
    csv_path = os.path.join(ROOT, "profiles", "r01_launches_final.csv")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "launch_summary.py"), csv_path],
                         capture_output=True, text=True, check=True).stdout
    first = out.splitlines()[0]
    assert first.startswith("one training step: launches 109"), first
    assert "tn_planes_kernel" in out and "gat_tree_bwd_kernel" in out


def test_bench_dump_outputs_at_headline_size(tmp_path):
    """bench.py --dump-outputs: float32 arrays under 64 MB in all at the headline's shapes (4096 trees x 301 nodes),
    the same logit rows every run; --steps 0 is refused rather than timing nothing."""
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import bench
    from spgnn_b200 import models as sm
    model, _, method, _ = bench.workload(bench.HEADLINE)
    net = getattr(sm, method.split(".")[-1])(**model)
    logits = torch.arange(4096 * 301 * 22, dtype=torch.float32).reshape(-1, 22)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), net, torch.tensor(1.5), logits)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grads.npy", "logits_sample.npy", "loss.npy", "params.npy"]
    arrays = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float32 for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["params"].size == sum(p.numel() for p in net.parameters()) == arrays["grads"].size
    assert arrays["logits_sample"].shape == (bench.DUMP_LOGIT_ROWS, 22) and float(arrays["loss"]) == 1.5
    assert np.array_equal(arrays["logits_sample"], np.load(tmp_path / "b" / "logits_sample.npy"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_host_row_packer_round_trips_on_the_cpu():
    """spgnn_host_pack_rows_* (host code of libspgnn_b200.so, no GPU involved): mask / values / row offsets of
    zero-suppressed rows reproduce the matrix bit for bit when decoded with numpy; multi-threaded == single-threaded."""
    import numpy as np
    import torch
    from spgnn_b200._lib import lib
    rng = np.random.default_rng(0)
    for rows, cols in ((257, 1024), (5, 96), (33, 50), (1, 1)):
        x = np.maximum(rng.standard_normal((rows, cols)), 0).astype(np.float32)
        x[0, 0] = -0.0
        x[:, -3:] = 0.0                                    # rows end in zeros: no write may land in the next row's slots
        xt = torch.from_numpy(x.copy())
        res = []
        for threads in (1, 4):
            row_off = torch.zeros(rows + 1, dtype=torch.int64)
            nnz = int(lib().host_pack_rows_count(xt.data_ptr(), cols, rows, cols, row_off.data_ptr(), threads))
            assert nnz == int((x.view(np.uint32) != 0).sum()) == int(row_off[-1])
            words = (cols + 31) // 32
            mask = torch.zeros(rows, words, dtype=torch.int32)
            vals = torch.full((nnz + 8,), 7.0, dtype=torch.float32)       # guard elements behind the last value
            lib().host_pack_rows_fill(xt.data_ptr(), cols, rows, cols, row_off.data_ptr(), mask.data_ptr(),
                                      vals.data_ptr(), threads)
            assert bool((vals[nnz:] == 7.0).all())
            res.append((row_off.clone(), mask.clone(), vals[:max(nnz, 1)].clone()))
        assert all(torch.equal(a, b) for a, b in zip(res[0], res[1]))
        row_off, mask, vals = (t.numpy() for t in res[0])
        bits = np.unpackbits(mask.view(np.uint8).reshape(rows, -1), axis=1, bitorder="little")[:, :cols].astype(bool)
        back = np.zeros((rows, cols), np.float32)
        back[bits] = vals[:nnz]
        assert np.array_equal(back.view(np.uint32), x.view(np.uint32))
        assert np.array_equal(np.diff(row_off), bits.sum(1))


def test_packed_host_batch_is_built_without_a_gpu():
    """runner.HostBatch(packed=True): edge lists in DGL edge order (row-major off-diagonal non-zeros), the batch's
    largest degree including the self loop, uint8 labels, zero-suppressed features — all host code."""
    import numpy as np
    import torch
    from spgnn_b200 import runner, synth
    scans = synth.make_scans(3, 6, ragged=True)
    n = [s.adj.shape[0] for s in scans]
    hb = runner.HostBatch(n, torch.from_numpy(np.concatenate([s.adj.reshape(-1) for s in scans])),
                          torch.from_numpy(np.concatenate([s.fvs for s in scans])),
                          torch.from_numpy(np.concatenate([s.fvs_out for s in scans])),
                          torch.from_numpy(np.concatenate([s.labels for s in scans]).astype(np.int64)), pin=False, packed=True)
    srcs, dsts, counts = [], [], [0]
    for s in scans:
        r, c = s.adj.nonzero()
        k = r != c
        srcs.append(r[k]); dsts.append(c[k]); counts.append(counts[-1] + int(k.sum()))
    assert np.array_equal(hb.e_src.numpy(), np.concatenate(srcs)) and np.array_equal(hb.e_dst.numpy(), np.concatenate(dsts))
    assert hb.e_off.tolist() == counts and hb.max_degree == 4 and hb.labels.dtype == torch.uint8
    fvs = np.concatenate([s.fvs for s in scans])
    assert hb.f_nnz == int((fvs != 0).sum()) and hb.nbytes() < 0.6 * (fvs.nbytes + sum(k * k for k in n))
