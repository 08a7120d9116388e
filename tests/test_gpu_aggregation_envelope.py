"""The non-attention aggregations of GraphConv, GINConv and SAGEConv over everything their entry points accept, not
just the aligned, 4-column padded, in-degree <= 4 tree batches of the shipped presets.

* spgnn_spmm (csrc/aggs.cu): every combination of pre / post / self_eps / self_in / add / bias, all five activations,
  odd widths and strided views (the scalar ``<1>`` kernel), bipartite shapes with n_self < N < n_src (the transposed
  call SpmmFn.backward makes), in-degree 0, repeated neighbours, a node of in-degree 5,000 and more nodes than one
  pass of the grid.  SpmmFn forward + backward on ``from_adj`` graphs and on sampled blocks.
* spgnn_sage_maxpool_fwd / _bwd: exact ties (the first in-CSC slot wins), empty neighbourhoods, multi-edges, both
  kernel instances; MaxPoolFn against torch's amax scatter.
* spgnn_degree_norms / spgnn_inv_degree: in-degree 0 (clamped to 1), add = 1, more nodes than one pass of the grid.

Inputs are hand-built int32 CSR arrays, so no tree batch limits the shapes.  References are plain fp64 torch or numpy.
Every output starts as NaN (int outputs as -7) and sits inside a wider buffer, so an entry the kernel forgets fails the
comparison and an entry it writes outside its view is caught.  Each case names the kernel instance it is meant to reach
and the profiler trace must show exactly that launch."""
import numpy as np
import pytest
import torch

from helpers import launches, rel_err

pytestmark = pytest.mark.gpu

NONE, ELU, TANH, RELU, LEAKY = 0, 1, 2, 3, 4         # SPGNN_ACT_*
ACTS = [(NONE, 0.0), (ELU, 0.0), (TANH, 0.0), (RELU, 0.0), (LEAKY, 0.2)]
NAN = float("nan")
U = 2.0 ** -24
# fp32 kernels vs fp64, relative to the largest entry of the output: every output entry is a sum of <= 12 terms (in-
# degree <= 6, the self terms, addend and bias); recursive summation of n terms is within (n - 1) u of the sum of their
# magnitudes, which for random-sign inputs is a few times the largest output: ~12 x 6e-8 x 3 = 2e-6.
TOL = 2e-6


@pytest.fixture(scope="module")
def mods():
    from spgnn_b200 import graph as sg, ops, sampling
    from spgnn_b200._lib import SpgnnError, lib, ptr, stream
    return dict(sg=sg, ops=ops, sampling=sampling, SpgnnError=SpgnnError, lib=lib, ptr=ptr, stream=stream)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def node_pass():
    """Nodes of one pass of node_grid (aggs.cu): sm_count x 32 blocks of 8 warps, one warp per node."""
    return _sms() * 32 * 8


def elem_pass():
    """Threads of one pass of elem_grid (aggs.cu): sm_count x 16 blocks of 256 threads."""
    return _sms() * 16 * 256


def act64(x, act, slope):
    f = torch.nn.functional
    if act == ELU:
        return f.elu(x)
    if act == TANH:
        return torch.tanh(x)
    if act == RELU:
        return f.relu(x)
    if act == LEAKY:
        return f.leaky_relu(x, float(np.float32(slope)))
    return x


# ------------------------------------------------------------------------------------------------ buffers
def dense(rows, cols, vec, fill=NAN, values=None):
    """(view, base): an fp32 [rows, cols] view inside a wider device buffer.  vec: leading dimension cols + 4, 16-byte
    aligned base (what the float4 kernels take when cols % 4 == 0); otherwise leading dimension cols + 3 and a base
    one float past alignment (the scalar kernels)."""
    ld = cols + (4 if vec else 3)
    base = torch.full((rows, ld), fill, dtype=torch.float32)
    off = 0 if vec else 1
    if values is not None:
        base[:, off:off + cols] = values
    base = base.cuda()
    return base[:, off:off + cols], base


def outside(view, base):
    """Entries of ``base`` outside ``view`` (must still hold the prefill)."""
    keep = torch.ones(base.shape, dtype=torch.bool)
    off = (view.data_ptr() - base.data_ptr()) // 4
    keep[:, off:off + view.shape[1]] = False
    return base.cpu()[keep]


def csr(deg, n_src, rng):
    """in_ptr int32 [N + 1] and in_src int32 [E]: node v has deg[v] in-neighbours drawn from [0, n_src)."""
    ptr = np.zeros(len(deg) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(deg)
    src = rng.integers(0, n_src, size=int(ptr[-1]))
    return ptr.astype(np.int32), src.astype(np.int32)


def plant_repeats(ptr, src, every=5):
    """Every ``every``-th node with in-degree >= 3 reads its first neighbour three times."""
    n = 0
    for v in range(len(ptr) - 1):
        if ptr[v + 1] - ptr[v] >= 3:
            n += 1
            if n % every == 0:
                src[ptr[v] + 1] = src[ptr[v] + 2] = src[ptr[v]]
    return src


def out_csr(ptr, src, n_src):
    """(out_ptr, out_dst, out_slot) of an in-CSC: edges sorted by source, stable (the layout Graph / Block keep)."""
    dst = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    order = np.argsort(src, kind="stable")
    optr = np.zeros(n_src + 1, dtype=np.int64)
    optr[1:] = np.cumsum(np.bincount(src, minlength=n_src))
    return optr.astype(np.int32), dst[order].astype(np.int32), order.astype(np.int32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------------ spmm
def spmm_ref(x, ptr, src, N, pre, post, eps, self_in, n_self, add, bias, act, slope):
    """ops.SpmmFn's formula in fp64: act(post (Σ_{u→v} pre[u] x[u] + [self_in, v < n_self] pre[v] x[v])
    + [eps given, v < n_self] (1 + eps) x[v] + add[v] + bias).  Differentiable in x, eps, bias, add."""
    F = x.shape[1]
    dst = torch.from_numpy(np.repeat(np.arange(N), np.diff(ptr.astype(np.int64))))
    s = torch.from_numpy(src.astype(np.int64))
    w = pre[s] if pre is not None else torch.ones(len(s), dtype=torch.float64)
    acc = torch.zeros(N, F, dtype=torch.float64).index_add(0, dst, w[:, None] * x[s])
    if self_in:
        sw = pre[:n_self] if pre is not None else torch.ones(n_self, dtype=torch.float64)
        acc = torch.cat([acc[:n_self] + sw[:, None] * x[:n_self], acc[n_self:]])
    r = acc * post[:, None] if post is not None else acc
    if eps is not None:
        r = torch.cat([r[:n_self] + (1.0 + eps) * x[:n_self], r[n_self:]])
    if add is not None:
        r = r + add
    if bias is not None:
        r = r + bias
    return act64(r, act, slope)


def run_spmm(mods, x, ptr, src, N, F, pre, post, eps, self_in, n_self, add, bias, act, slope, vec, want):
    """One spgnn_spmm call under the profiler (x, add: (view, base) pairs on the device); checks the launch and the
    output against spmm_ref, and that nothing outside the output view was written."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    out, obase = dense(N, F, vec)
    xv, av = x[0], (add[0] if add is not None else None)
    pre_d, post_d = (dev(t) if t is not None else None for t in (pre, post))
    eps_d = torch.tensor([eps], dtype=torch.float32).cuda() if eps is not None else None
    bias_d = dev(bias) if bias is not None else None
    ptr_d, src_d = dev(ptr), dev(src)
    torch.cuda.synchronize()

    def run():
        lib().spmm(P(xv), xv.stride(0), P(ptr_d), P(src_d), P(pre_d), P(post_d), P(eps_d), int(self_in), n_self,
                   P(av), av.stride(0) if av is not None else 0, P(bias_d), act, slope, P(out), out.stride(0), N, F,
                   stream())

    names = launches(run)
    assert names == {f"spmm_kernel<{want}>"}, names
    d64 = lambda t: torch.from_numpy(np.asarray(t, dtype=np.float64)) if t is not None else None
    ref = spmm_ref(xv.cpu().double(), ptr, src, N, d64(pre), d64(post),
                   float(np.float32(eps)) if eps is not None else None, self_in, n_self,
                   av.cpu().double() if av is not None else None, d64(bias), act, slope)
    got = out.cpu()
    assert not torch.isnan(got).any(), "rows or columns left unwritten"
    assert torch.isnan(outside(out, obase)).all(), "written outside the output view"
    return got, ref


# the 64 combinations of (pre, post, self_eps, self_in, add, bias); the activation and F cycle through their lists,
# vec alternates every 8 cases so that every F % 4 == 0 width runs both instances
SPMM_FS = [1, 3, 4, 5, 64, 127, 129, 1024]


def _combo(i):
    flags = [bool(i >> b & 1) for b in range(6)]
    F = SPMM_FS[i % 8]
    vec = (i // 8) % 2 == 0 and F % 4 == 0
    act, slope = ACTS[i % 5]
    return flags, F, vec, act, slope


@pytest.mark.parametrize("i", range(64), ids=lambda i: "pre{}_post{}_eps{}_selfin{}_add{}_bias{}".format(
    *(int(b) for b in _combo(i)[0])) + f"_F{_combo(i)[1]}_{'vec4' if _combo(i)[2] else 'scalar'}_act{_combo(i)[3]}")
def test_spmm_every_term_combination_on_a_bipartite_block(mods, i):
    """N = 300 destinations, n_src = 420 source rows, self terms for the first n_self = 200 (n_self < N < n_src),
    in-degrees 0..6 with repeated neighbours.  <4> when F % 4 == 0 and every operand is a 16-byte aligned view with
    ld % 4 == 0; <1> for odd F and for strided views (odd ld, base one float past alignment)."""
    (use_pre, use_post, use_eps, self_in, use_add, use_bias), F, vec, act, slope = _combo(i)
    rng = np.random.default_rng(100 + i)
    N, n_src, n_self = 300, 420, 200
    deg = rng.integers(0, 7, size=N)
    deg[::17] = 0
    ptr, src = csr(deg, n_src, rng)
    src = plant_repeats(ptr, src)
    x = dense(n_src, F, vec, values=torch.from_numpy(rng.standard_normal((n_src, F)).astype(np.float32)))
    pre = rng.uniform(0.2, 1.5, n_src).astype(np.float32) if use_pre else None
    post = rng.uniform(0.2, 1.5, N).astype(np.float32) if use_post else None
    eps = float(rng.uniform(-0.5, 0.5)) if use_eps else None
    add = dense(N, F, vec, values=torch.from_numpy(rng.standard_normal((N, F)).astype(np.float32))) if use_add else None
    bias = rng.standard_normal(F).astype(np.float32) if use_bias else None
    got, ref = run_spmm(mods, x, ptr, src, N, F, pre, post, eps, self_in, n_self, add, bias, act, slope, vec,
                        4 if vec else 1)
    assert rel_err(got, ref) < TOL


@pytest.mark.parametrize("F,vec", [(128, True), (129, False), (4, False)])
def test_spmm_node_of_in_degree_5000(mods, F, vec):
    """One destination reads 5,000 neighbours (with repeats), the others 0..3.  x holds multiples of 1/4 in [-2, 2]
    and there is no pre norm, so every partial sum is exact in fp32 and only the post-scale, addend and bias round:
    the 1e-6 bar holds however many terms the hub adds."""
    rng = np.random.default_rng(F)
    N, n_src = 60, 3000
    deg = rng.integers(0, 4, size=N)
    deg[7] = 5000
    ptr, src = csr(deg, n_src, rng)
    xs = torch.from_numpy(rng.integers(-8, 9, size=(n_src, F)).astype(np.float32) / 4)
    x = dense(n_src, F, vec, values=xs)
    post = rng.uniform(0.2, 1.5, N).astype(np.float32)
    add = dense(N, F, vec, values=torch.from_numpy(rng.standard_normal((N, F)).astype(np.float32)))
    bias = rng.standard_normal(F).astype(np.float32)
    got, ref = run_spmm(mods, x, ptr, src, N, F, None, post, 0.25, True, N, add, bias, ELU, 0.0, vec,
                        4 if vec else 1)
    assert rel_err(got, ref) < 1e-6


@pytest.mark.parametrize("F,vec", [(4, True), (3, False)])
def test_spmm_more_nodes_than_one_grid_pass(mods, F, vec):
    """N = 40,001 destinations: node_grid caps at sm_count x 32 blocks of 8 warps, so warps take a second node."""
    N = 40001
    assert N > node_pass()
    rng = np.random.default_rng(7)
    n_src, n_self = N + 100, N - 50
    deg = rng.integers(0, 6, size=N)
    ptr, src = csr(deg, n_src, rng)
    x = dense(n_src, F, vec, values=torch.from_numpy(rng.standard_normal((n_src, F)).astype(np.float32)))
    pre = rng.uniform(0.2, 1.5, n_src).astype(np.float32)
    post = rng.uniform(0.2, 1.5, N).astype(np.float32)
    got, ref = run_spmm(mods, x, ptr, src, N, F, pre, post, 0.1, True, n_self, None,
                        rng.standard_normal(F).astype(np.float32), LEAKY, 0.2, vec, 4 if vec else 1)
    assert rel_err(got, ref) < TOL


def _grad_sum_close(got, ref, mag, what, tol=1e-5):
    """A gradient that is a long fp32 reduction (torch's sum for d eps, spgnn_colsum for d bias): within tol of the
    sum of the magnitudes of its terms.  A term dropped or counted twice moves it by ~1/n of that sum (n <= 10^3 here),
    far outside the bar."""
    err = (got.double() - ref).abs()
    assert bool((err <= tol * mag + 1e-30).all()), (what, float((err / mag).max()))


def _spmm_backward_case(mods, graph, n_src, act, slope, pre, post, use_eps, self_in, use_add, use_bias, seed):
    """SpmmFn forward + backward against fp64 autograd of spmm_ref on the graph's own in-CSC."""
    ops = mods["ops"]
    F = 36
    N = ops._n_dst(graph)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(n_src, F, generator=gen)
    eps = torch.tensor([0.3]) if use_eps else None
    bias = torch.randn(F, generator=gen) if use_bias else None
    add = torch.randn(N, F, generator=gen) if use_add else None
    gw = torch.randn(N, F, generator=gen, dtype=torch.float64)
    leaf = lambda t: t.cuda().requires_grad_() if t is not None else None
    xd, ed, bd, ad = leaf(x), leaf(eps), leaf(bias), leaf(add)
    out = ops.SpmmFn.apply(xd, ed, bd, graph, pre, post, act, slope, ad, self_in)
    names = launches(lambda: (out * gw.float().cuda()).sum().backward())
    want = {"spmm_kernel<4>"} | ({"act_bwd_kernel<4>"} if act else set())
    if use_bias:
        want |= {"colsum_partial_kernel", "colsum_final_kernel"}
    assert names == want, (sorted(names), sorted(want))

    ptr, src = graph.in_ptr.cpu().numpy(), graph.in_src.cpu().numpy()
    c64 = lambda t: t.detach().cpu().double() if t is not None else None
    x64, e64, b64, a64 = (c64(t).requires_grad_() if t is not None else None for t in (x, eps, bias, add))
    ref = spmm_ref(x64, ptr, src, N, c64(pre), c64(post), e64[0] if e64 is not None else None, self_in, N, a64, b64,
                   act, slope)
    assert rel_err(out.detach().cpu(), ref.detach()) < TOL, "forward"
    (ref * gw).sum().backward()
    assert rel_err(xd.grad.cpu(), x64.grad) < TOL, "dx"
    dp = _dpre(ref, gw, act, slope)           # gradient at the pre-activation: the terms of d add, d bias, d eps
    if use_add:
        assert rel_err(ad.grad.cpu(), a64.grad) < 1e-6, "d add"
    if use_bias:
        _grad_sum_close(bd.grad.cpu(), b64.grad, dp.abs().sum(0), "d bias")
    if use_eps:
        _grad_sum_close(ed.grad.cpu(), e64.grad, (dp * x64.detach()[:N]).abs().sum().reshape(1), "d eps")


def _dpre(ref, gw, act, slope):
    """gradient of sum(out * gw) with respect to the pre-activation, from the fp64 output"""
    y = ref.detach()
    if act == ELU:
        return gw * torch.where(y > 0, torch.ones_like(y), y + 1)
    if act == TANH:
        return gw * (1 - y * y)
    if act == RELU:
        return gw * (y > 0)
    if act == LEAKY:
        return gw * torch.where(y > 0, 1.0, float(np.float32(slope)))
    return gw


def _random_adj(n, p, rng):
    a = (rng.random((n, n)) < p).astype(np.uint8)
    np.fill_diagonal(a, 1)
    return a


@pytest.mark.parametrize("kind", ["graphconv_both", "gin_mean", "sage_gcn_leaky", "block_sage_gcn", "block_mean"])
def test_spmm_function_backward_against_fp64_autograd(mods, kind):
    """SpmmFn forward + backward (dx by the transposed spmm call, d eps, d bias by spgnn_colsum, d add) on a random
    directed graph from ``from_adj`` (in-degrees 1..~15) and on sampled SAGE blocks (n_src > N, self terms for the
    destinations only)."""
    sg, ops, sampling = mods["sg"], mods["ops"], mods["sampling"]
    rng = np.random.default_rng(len(kind))
    g = sg.from_adj(_random_adj(240, 0.03, rng))
    o_s, i_s, i_i, _ = g.norms()
    if kind == "graphconv_both":
        _spmm_backward_case(mods, g, g.num_nodes, RELU, 0.0, o_s, i_s, False, False, False, True, 1)
    elif kind == "gin_mean":
        _spmm_backward_case(mods, g, g.num_nodes, NONE, 0.0, None, i_i, True, False, False, False, 2)
    elif kind == "sage_gcn_leaky":
        _spmm_backward_case(mods, g, g.num_nodes, LEAKY, 0.2, None, ops.inv_degree(g, 1.0), False, True, True, True,
                            3)
    else:
        seeds = torch.from_numpy(rng.choice(g.num_nodes, 64, replace=False)).cuda()
        blk = sampling.MultiLayerNeighborSampler([4]).sample_blocks(g, seeds,
                                                                    torch.Generator(device="cuda").manual_seed(5))[0]
        assert blk.num_src_nodes > blk.num_dst_nodes
        if kind == "block_sage_gcn":
            _spmm_backward_case(mods, blk, blk.num_src_nodes, ELU, 0.0, None, ops.inv_degree(blk, 1.0), True, True,
                                True, True, 4)
        else:
            _spmm_backward_case(mods, blk, blk.num_src_nodes, TANH, 0.0, None, ops.inv_degree(blk, 0.0), False, False,
                                False, True, 5)


# ------------------------------------------------------------------------------------------------ max-pool
def maxpool_ref(m, ptr, src, N):
    """(out, arg): elementwise max over the in-neighbours, arg = FIRST in-CSC slot reaching it; empty: 0 and -1."""
    F = m.shape[1]
    out = np.zeros((N, F), dtype=np.float32)
    arg = np.full((N, F), -1, dtype=np.int32)
    for v in range(N):
        b, e = int(ptr[v]), int(ptr[v + 1])
        if b == e:
            continue
        vals = m[src[b:e]]
        out[v] = vals.max(0)
        arg[v] = b + np.argmax(vals == out[v], axis=0)
    return out, arg


def maxpool_bwd_ref(g, arg, src, n_src):
    """dm[u] = sum of g[v] over the (v, column) whose arg slot reads u: one slot per (v, column), however many
    edges u -> v there are."""
    dm = np.zeros((n_src, g.shape[1]), dtype=np.float64)
    v, c = np.nonzero(arg >= 0)
    np.add.at(dm, (src[arg[v, c]], c), g[v, c].astype(np.float64))
    return dm


@pytest.mark.parametrize("F,vec_m,vec_g,N", [(4, True, True, 300), (64, False, True, 300), (64, True, False, 300),
                                              (3, False, False, 300), (129, False, False, 300), (1, False, False, 300),
                                              (4, True, True, 40001)])
def test_maxpool_exact_against_numpy(mods, F, vec_m, vec_g, N):
    """out = numpy's max exactly; arg = the first in-CSC slot that reaches it, on values drawn from 9 levels so that
    most maxima are exact ties between different sources and multi-edges; empty neighbourhoods give 0 and -1.  The
    backward scatter against fp64: only the arg slot of a multi-edge gets the gradient.  The forward takes <4> when
    m is 16-byte aligned with ld % 4 == 0 and F % 4 == 0, the backward when g and dm are; N = 40,001 needs more than
    one pass of node_grid."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    rng = np.random.default_rng(F * 7 + N)
    n_src = N + 50
    deg = rng.integers(0, 7, size=N)
    deg[::13] = 0
    ptr, src = csr(deg, n_src, rng)
    src = plant_repeats(ptr, src, every=3)
    assert (N > node_pass()) == (N == 40001)
    mv = (rng.integers(-4, 5, size=(n_src, F)) * 0.5).astype(np.float32)
    m, _ = dense(n_src, F, vec_m, values=torch.from_numpy(mv))
    out, obase = dense(N, F, vec_m)
    arg = torch.full((N, F), -7, dtype=torch.int32, device="cuda")
    ptr_d, src_d = dev(ptr), dev(src)
    torch.cuda.synchronize()
    fwd = launches(lambda: lib().sage_maxpool_fwd(P(m), m.stride(0), P(ptr_d), P(src_d), P(out), out.stride(0),
                                                  P(arg), N, F, stream()))
    assert fwd == {f"maxpool_fwd_kernel<{4 if vec_m else 1}>"}, fwd
    ro, ra = maxpool_ref(mv, ptr, src, N)
    assert np.array_equal(out.cpu().numpy(), ro), "max values"
    assert np.array_equal(arg.cpu().numpy(), ra), "arg slots"
    assert torch.isnan(outside(out, obase)).all()
    ties = np.array([(mv[src[ptr[v]:ptr[v + 1]]] == ro[v]).sum(0) for v in range(min(N, 300))])
    assert (ties > 1).mean() > 0.05, "the inputs should hold many exact ties"

    optr, odst, oslot = out_csr(ptr, src, n_src)
    gv = rng.standard_normal((N, F)).astype(np.float32)
    g, _ = dense(N, F, vec_g, values=torch.from_numpy(gv))
    dm, dbase = dense(n_src, F, vec_g)
    optr_d, odst_d, oslot_d = dev(optr), dev(odst), dev(oslot)
    torch.cuda.synchronize()
    bwd = launches(lambda: lib().sage_maxpool_bwd(P(g), g.stride(0), P(arg), P(optr_d), P(odst_d), P(oslot_d), P(dm),
                                                  dm.stride(0), n_src, F, stream()))
    assert bwd == {f"maxpool_bwd_kernel<{4 if vec_g else 1}>"}, bwd
    ref = maxpool_bwd_ref(gv, ra, src, n_src)
    got = dm.cpu()
    assert not torch.isnan(got).any() and torch.isnan(outside(dm, dbase)).all()
    assert rel_err(got, ref) < TOL


def test_maxpool_function_against_torch_amax(mods):
    """MaxPoolFn forward + backward on a from_adj graph and on a sampled block against fp64 torch scatter_reduce
    ('amax') autograd, on continuous inputs (no ties, where torch would split the gradient)."""
    sg, ops, sampling = mods["sg"], mods["ops"], mods["sampling"]
    rng = np.random.default_rng(11)
    g = sg.from_adj(_random_adj(200, 0.04, rng))
    seeds = torch.from_numpy(rng.choice(200, 50, replace=False)).cuda()
    blk = sampling.MultiLayerNeighborSampler([3]).sample_blocks(g, seeds,
                                                                torch.Generator(device="cuda").manual_seed(1))[0]
    for graph, n_src, n_dst in ((g, 200, 200), (blk, blk.num_src_nodes, blk.num_dst_nodes)):
        m = torch.randn(n_src, 20, dtype=torch.float64)
        gw = torch.randn(n_dst, 20, dtype=torch.float64)
        md = m.float().cuda().requires_grad_()
        out = ops.MaxPoolFn.apply(md, graph)
        (out * gw.float().cuda()).sum().backward()
        dst = torch.repeat_interleave(torch.arange(n_dst), (graph.in_ptr[1:] - graph.in_ptr[:-1]).long().cpu())
        m64 = m.float().double().requires_grad_()
        ref = torch.zeros(n_dst, 20, dtype=torch.float64).scatter_reduce(
            0, dst[:, None].expand(-1, 20), m64[graph.in_src.long().cpu()], "amax", include_self=False)
        (ref * gw).sum().backward()
        assert torch.equal(out.detach().cpu().double(), ref.detach())
        assert rel_err(md.grad.cpu(), m64.grad) < 1e-6


# ------------------------------------------------------------------------------------------------ degree norms
def test_degree_norms_and_inv_degree(mods):
    """degree_norms: deg^-1/2 within 2 ulp of fp64 (powf) and 1/deg bit for bit (IEEE division), degrees clamped to
    1; inv_degree: 1 / max(deg + add, 1) bit for bit for add = 0 and 1.  In-degrees 0, 1, 2, 5,000 and random, over
    more nodes than one pass of elem_grid."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    N = elem_pass() + 1001
    rng = np.random.default_rng(3)
    deg = rng.integers(0, 9, size=N)
    deg[:4] = [0, 1, 2, 5000]
    deg[-1] = 0
    ptr = np.zeros(N + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(deg)
    ptr_d = dev(ptr.astype(np.int32))
    ns, ni = torch.full((N + 4,), NAN, device="cuda"), torch.full((N + 4,), NAN, device="cuda")
    i0, i1 = torch.full((N + 4,), NAN, device="cuda"), torch.full((N + 4,), NAN, device="cuda")
    only = torch.full((N,), NAN, device="cuda")

    def run():
        lib().degree_norms(P(ptr_d), N, P(ns), P(ni), stream())
        lib().degree_norms(P(ptr_d), N, None, P(only), stream())
        lib().inv_degree(P(ptr_d), N, 0.0, P(i0), stream())
        lib().inv_degree(P(ptr_d), N, 1.0, P(i1), stream())

    assert launches(run) == {"degree_norms_kernel", "inv_degree_kernel"}
    d = np.maximum(deg, 1).astype(np.float32)
    ref_s = np.maximum(deg, 1).astype(np.float64) ** -0.5
    got_s = ns.cpu().numpy()
    assert np.isnan(got_s[N:]).all() and np.isnan(ni.cpu().numpy()[N:]).all()
    assert (np.abs(got_s[:N] - ref_s) <= 2 * U * 2 * ref_s).all(), "deg^-1/2"
    one = np.float32(1)
    assert np.array_equal(ni.cpu().numpy()[:N], one / d)
    assert np.array_equal(only.cpu().numpy(), one / d)
    for got, add in ((i0, 0), (i1, 1)):
        ref = one / np.maximum(deg.astype(np.float32) + np.float32(add), one)
        g = got.cpu().numpy()
        assert np.array_equal(g[:N], ref) and np.isnan(g[N:]).all(), add
