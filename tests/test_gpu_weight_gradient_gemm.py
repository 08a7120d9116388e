"""The dW GEMM (spgnn_planes_linear_bwd_weight: tn_planes_kernel + reduce_splits, planned by tn_plan) against fp64
on shapes chosen so that every branch of its planner is taken and asserted through spgnn_planes_linear_bwd_weight_plan:
either orientation (swap), one launch per source (split sources), one or many row ranges, the "more tile pairs than
SMs" fallback, row ranges longer than the 8192-row accumulator drain, ragged 32-row stages and N / K remainders.  The
drain itself and the split-source choice are also switched by their environment overrides, which are read once per
process, in subprocesses."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMS = 148
T_BK = 32                # rows per pipeline stage
FLUSH_ROWS = 8192        # rows accumulated in TMEM between two drains (default)
TOL = 4e-5               # split-bf16 planes GEMMs vs fp64 (test_linear_fwd_bwd_against_fp64)

# (M, N, K1, K2) -> what its plan must show
SHAPES = {
    (1, 22, 39, 0): dict(swap=0, split=0, splits=1),                       # a single row
    (31, 130, 258, 0): dict(swap=0, split=0, splits=1),                    # one partial stage
    (33, 258, 130, 0): dict(swap=0, split=0, splits=1),                    # a ragged second stage
    (33, 1028, 1024, 39): dict(swap=0, split=0, splits=1),                 # gat0's widths, too few rows to split
    (8191, 1028, 1024, 39): dict(swap=0, split=1, multi=True),             # gat0: one launch per source
    (8193, 1028, 1024, 39): dict(swap=0, split=1, multi=True),
    (8193, 1024, 192, 192): dict(swap=1, split=0, multi=True),             # the output layer's dW: dC on the M side
    (8191, 22, 258, 0): dict(swap=0, split=0, multi=True),
    (8193, 130, 39, 22): dict(swap=0, split=0, multi=True),                # two ragged sources in one launch
    (8191, 39, 130, 22): dict(split=0, multi=True),
    (257, 4100, 2304, 0): dict(swap=0, split=0, splits=1, fallback=True),  # 9 x 17 = 153 tile pairs > 148 SMs
    (620001, 22, 258, 0): dict(swap=0, split=0, multi=True, long=True),    # > 8192 rows per range: two drains
}


def plan_of(M, N, K1, K2):
    from spgnn_b200._lib import lib
    out = (ctypes.c_int32 * 9)()
    assert lib().planes_linear_bwd_weight_plan(M, N, K1, K2, out, 9) == 9
    keys = ("swap", "np_tiles", "nq_tiles", "splits", "ctas", "rows", "npb", "nqb", "split")
    return dict(zip(keys, list(out)))


def operands(M, N, K1, K2):
    """Seeded planes dC [M, N], X1 [M, K1], X2 [M, K2] (from fp32 data drawn on the device)."""
    from spgnn_b200 import stack
    gen = torch.Generator(device="cuda").manual_seed(M * 31 + N * 7 + K1 + K2)
    dC = stack.split_planes(torch.randn(M, N, device="cuda", generator=gen))
    X1 = stack.split_planes(torch.randn(M, K1, device="cuda", generator=gen))
    X2 = stack.split_planes(torch.randn(M, K2, device="cuda", generator=gen)) if K2 else None
    return dC, X1, X2


def dw(M, N, K1, K2):
    from spgnn_b200 import stack
    dC, X1, X2 = operands(M, N, K1, K2)
    return stack.planes_linear_bwd_weight(dC, X1, X2).cpu()


def dw_ref(M, N, K1, K2):
    """fp64 dC^T [X1 | X2] from exactly the values the kernel reads (the planes' hi + lo)."""
    dC, X1, X2 = operands(M, N, K1, K2)
    x = torch.cat([X1.float()] + ([X2.float()] if X2 is not None else []), 1).double().cpu()
    return dC.float().double().cpu().t() @ x


def check_plan(shape, want):
    M, N, K1, K2 = shape
    p = plan_of(*shape)
    for k in ("swap", "split", "splits"):
        if k in want:
            assert p[k] == want[k], (shape, k, p)
    tiles = p["np_tiles"] * p["nq_tiles"]
    assert p["ctas"] == tiles * p["splits"]
    assert p["rows"] % T_BK == 0 and p["rows"] * p["splits"] >= M > p["rows"] * (p["splits"] - 1)
    if want.get("multi"):
        assert p["splits"] > 1, (shape, p)
    if want.get("fallback"):
        assert tiles > SMS and p["splits"] == 1, (shape, p)
    else:
        assert tiles <= SMS, (shape, p)
    drains = -(-(p["rows"] // T_BK) // (FLUSH_ROWS // T_BK))
    assert (drains >= 2) == bool(want.get("long")), (shape, p)
    return p


def test_the_shape_list_takes_every_branch_of_the_planner():
    """Across the shapes: both orientations, both source plans, one and many row ranges, the fallback, a row range
    with two drains, ragged last stages, and N and K remainders 22, 39, 130, 258 mod 64."""
    plans = {s: check_plan(s, w) for s, w in SHAPES.items()}
    assert {p["swap"] for p in plans.values()} == {0, 1}
    assert {p["split"] for p in plans.values()} == {0, 1}
    assert any(p["splits"] == 1 for p in plans.values()) and any(p["splits"] > 1 for p in plans.values())
    assert any(s[0] % T_BK for s in SHAPES)
    rems = {r % 64 for s in SHAPES for r in s[1:] if r}
    assert {22, 39, 130 % 64, 258 % 64} <= rems


@pytest.mark.parametrize("shape", list(SHAPES), ids=lambda s: "x".join(map(str, s)))
def test_weight_gradient_gemm_against_fp64(shape):
    check_plan(shape, SHAPES[shape])
    assert rel_err(dw(*shape), dw_ref(*shape)) < TOL, shape


_SCRIPT = r"""
import sys, torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from test_gpu_weight_gradient_gemm import SHAPES, dw, plan_of
shapes = [s for s in SHAPES if "x".join(map(str, s)) in sys.argv[3].split(",")]
torch.save({s: (dw(*s), plan_of(*s)) for s in shapes}, sys.argv[2])
"""


def _in_subprocess(env, shapes, path):
    r = subprocess.run([sys.executable, "-c", _SCRIPT, ROOT, str(path), ",".join("x".join(map(str, s)) for s in shapes)],
                       env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return torch.load(path, weights_only=False)


def test_many_drains_at_small_row_counts(tmp_path):
    """SPGNN_TN_FLUSH_ROWS=256 drains the accumulators every 8 stages: every row range of every shape (but the
    shortest) then holds several drain chunks.  Same plans, dW within the fp64 tolerance."""
    res = _in_subprocess({"SPGNN_TN_FLUSH_ROWS": "256"}, list(SHAPES), tmp_path / "flush.pt")
    several = 0
    for s in SHAPES:
        got, p = res[s]
        assert p == plan_of(*s), s                              # the drain changes the chunks, not the plan
        several += -(-p["rows"] // 256) >= 2
        assert rel_err(got, dw_ref(*s)) < TOL, s
    assert several >= len(SHAPES) - 4


def test_split_sources_off_gives_the_same_weight_gradient(tmp_path):
    """SPGNN_TN_SPLIT_SOURCES=0 keeps gat0's two sources in one launch (17 x 17 blocks): same dW within tolerance."""
    shapes = [(8191, 1028, 1024, 39), (8193, 1028, 1024, 39)]
    res = _in_subprocess({"SPGNN_TN_SPLIT_SOURCES": "0"}, shapes, tmp_path / "nosplit.pt")
    for s in shapes:
        got, p = res[s]
        assert p["split"] == 0 and plan_of(*s)["split"] == 1, s
        assert p["npb"] + p["nqb"] == 17 + 17, p
        ref = dw_ref(*s)
        assert rel_err(got, ref) < TOL, s
        assert rel_err(got, dw(*s).double()) < TOL, s
