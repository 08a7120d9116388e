"""The elementwise glue between projections, the dropout masks, the loss and the decision over everything their entry
points accept, not just the shipped widths on aligned tree batches.

* spgnn_bias_act / spgnn_act_bwd (csrc/aggs.cu): every activation and LeakyReLU slope against torch.nn.functional in
  fp64, both kernel instances, more elements than one pass of the grid.
* The two mask hashes restated on the host (mix64 / u01 and fmix32 / chunk_hash, csrc/common.cuh) pin every mask bit
  for bit: concat_dropout and its backward, split_planes (with chunk_off > 0 inside a concatenation), the masked dX
  epilogue of planes_linear_bwd_input_masked, act_bwd_planes(drop_p) and the drawn node mask of masked_ce.  A defect
  shared by a mask's producer and its consumer cannot cancel out against a definition written outside CUDA.
* The planes split (split2, csrc/tc_ptx.cuh) restated in numpy: split_planes and act_bwd_planes write exactly those
  bits, padding columns 0 in both planes.
* spgnn_act_bwd_planes over ragged N, several column groups, one row band and many; its column sums; its refusals.
* spgnn_colsum over partial row bands, several column blocks and strided rows; bit-identical run to run.
* spgnn_masked_ce_fwd / _bwd and spgnn_segmented_argmax against F.cross_entropy and numpy's first-index argmax.

Every output starts as NaN (planes as the bf16 NaN pattern 0x7FC0, int outputs as a sentinel) inside a wider buffer.
Each case names the kernel instance it is meant to reach and the profiler trace must show exactly that launch."""
import numpy as np
import pytest
import torch

from helpers import launches, rel_err

pytestmark = pytest.mark.gpu

NONE, ELU, TANH, RELU, LEAKY = 0, 1, 2, 3, 4         # SPGNN_ACT_*
NAN = float("nan")
U = 2.0 ** -24
BF16_NAN = 0x7FC0
SEED = 0xD1B54A32D192ED03          # both 32-bit halves of a seed enter chunk_hash
F = torch.nn.functional


@pytest.fixture(scope="module")
def mods():
    from spgnn_b200 import ops, stack
    from spgnn_b200._lib import SpgnnError, lib, ptr, stream
    # the per-step seed salt is 0 outside a replayed CUDA graph; reset it as test_seed_salt_changes_every_mask_and_resets
    # does, so that salted(seed) == seed below
    zero = torch.zeros(1, dtype=torch.int64, device="cuda")
    lib().seed_salt_set(ptr(zero), stream())
    torch.cuda.synchronize()
    return dict(ops=ops, stack=stack, SpgnnError=SpgnnError, lib=lib, ptr=ptr, stream=stream)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def elem_pass():
    """Threads of one pass of elem_grid (aggs.cu): sm_count x 16 blocks of 256 threads."""
    return _sms() * 16 * 256


# ------------------------------------------------------------------------------------------------ host restatements
def mix64(x):
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def u01(seed, idx):
    """common.cuh u01 with salted(seed) = seed: 24 bits of mix64(seed ^ mix64(idx)) over 2^24, fp32."""
    h = mix64(np.uint64(seed) ^ mix64(np.asarray(idx, dtype=np.uint64)))
    return (h >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def fmix32(h):
    h = h ^ (h >> np.uint32(16))
    h = h * np.uint32(0x85EBCA6B)
    h = h ^ (h >> np.uint32(13))
    h = h * np.uint32(0xC2B2AE35)
    return h ^ (h >> np.uint32(16))


def chunk_hash(seed, idx):
    """common.cuh chunk_hash with salted(seed) = seed: 64 mask bits of one 4-column chunk, 16 per element."""
    idx = np.asarray(idx, dtype=np.uint64)
    lo, hi = (idx & np.uint64(0xFFFFFFFF)).astype(np.uint32), (idx >> np.uint64(32)).astype(np.uint32)
    s_lo, s_hi = np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32)
    a = fmix32((s_lo ^ (lo * np.uint32(0x9E3779B1))) + hi * np.uint32(0x85EBCA77))
    b = fmix32((s_hi ^ (lo * np.uint32(0xC2B2AE3D)) ^ a) + hi * np.uint32(0x27D4EB2F))
    return a.astype(np.uint64) | (b.astype(np.uint64) << np.uint64(32))


def thr16(p):
    """round(p * 65536) as the entry points form it in fp32"""
    return int(np.float32(np.float32(p) * np.float32(65536.0) + np.float32(0.5)))


def scale32(p):
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def planes_keep(seed, p, rows, cols, concat_chunks, chunk_off):
    """[rows, cols] bool: the planes dropout mask of element (r, c), chunk r * concat_chunks + chunk_off + c / 4,
    bits 16 (c % 4) .. + 15 kept iff >= round(p * 65536)."""
    r = np.arange(rows, dtype=np.uint64)[:, None]
    c = np.arange(cols, dtype=np.uint64)[None, :]
    h = chunk_hash(seed, r * np.uint64(concat_chunks) + np.uint64(chunk_off) + c // np.uint64(4))
    return ((h >> (np.uint64(16) * (c % np.uint64(4)))) & np.uint64(0xFFFF)) >= np.uint64(thr16(p))


def elem_keep(seed, p, rows, cols):
    """[rows, cols] bool: the concat_dropout mask, u01(seed, r * cols + c) >= p"""
    idx = np.arange(rows, dtype=np.uint64)[:, None] * np.uint64(cols) + np.arange(cols, dtype=np.uint64)[None, :]
    return u01(seed, idx) >= np.float32(p)


def apply_keep(x, keep, p):
    """fp32 x * 1/(1 - p) where kept, 0 elsewhere (the kernels' arithmetic)"""
    return np.where(keep, x.astype(np.float32) * scale32(p), np.float32(0)).astype(np.float32)


def bf16_rne(x):
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    return ((b + np.uint64(0x7FFF) + ((b >> np.uint64(16)) & np.uint64(1))) >> np.uint64(16)).astype(np.uint16)


def bf16_up(h):
    return (h.astype(np.uint32) << np.uint32(16)).view(np.float32)


def split2(x):
    """tc_ptx.cuh split2: hi = bf16 round-to-nearest-even of x, lo = the same rounding of the fp32 x - hi."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    hi = bf16_rne(x)
    lo = bf16_rne((x - bf16_up(hi)).astype(np.float32))
    return hi, lo


def planes_buffer(rows, ldo):
    """[2, rows, ldo] int16 planes buffer filled with the bf16 NaN pattern; ps = rows * ldo"""
    return torch.full((2, rows, ldo), BF16_NAN, dtype=torch.int16, device="cuda")


def check_planes(buf, d, cols):
    """The planes hold exactly split2(d) in columns [0, cols), exact zeros in both planes up to the next multiple of
    4, and the NaN prefill beyond."""
    b = buf.cpu().numpy().view(np.uint16)
    hi, lo = split2(d)
    n4 = (cols + 3) // 4 * 4
    assert np.array_equal(b[0, :, :cols], hi), "hi plane"
    assert np.array_equal(b[1, :, :cols], lo), "lo plane"
    assert (b[:, :, cols:n4] == 0).all(), "padding columns must be 0 in both planes"
    assert (b[:, :, n4:] == BF16_NAN).all(), "written past the padded row"


def test_the_seed_salt_is_zero_and_the_restated_masks_hold_their_rate(mods):
    """After the reset, ops.drop_mask (concat_dropout on ones) is the host restatement of u01 bit for bit, so the salt
    is 0; both restated hashes draw their nominal rates."""
    ops = mods["ops"]
    m = ops.drop_mask(301, 37, 0.3, SEED, "cuda").cpu().numpy()
    keep = elem_keep(SEED, 0.3, 301, 37)
    assert np.array_equal(m, np.where(keep, scale32(0.3), np.float32(0)))
    for p in (0.1, 0.5, 0.99):
        assert abs(elem_keep(SEED, p, 400, 250).mean() - (1 - p)) < 0.01
        assert abs(planes_keep(SEED, p, 400, 250, 63, 0).mean() - (1 - p)) < 0.01


# ------------------------------------------------------------------------------------------------ bias_act / act_bwd
def act64(x, act, slope):
    if act == ELU:
        return F.elu(x)
    if act == TANH:
        return torch.tanh(x)
    if act == RELU:
        return F.relu(x)
    if act == LEAKY:
        return F.leaky_relu(x, float(np.float32(slope)))
    return x


def dense(rows, cols, vec, values=None, fill=NAN):
    """(view, base): fp32 [rows, cols] inside a wider device buffer; vec: ld = cols + 4, aligned base; otherwise
    ld = cols + 3 and a base one float past 16-byte alignment."""
    ld = cols + (4 if vec else 3)
    off = 0 if vec else 1
    base = torch.full((rows, ld), fill, dtype=torch.float32)
    if values is not None:
        base[:, off:off + cols] = torch.as_tensor(values)
    base = base.cuda()
    return base[:, off:off + cols], base


def outside_ok(view, base, fill_nan=True):
    keep = torch.ones(base.shape, dtype=torch.bool)
    off = (view.data_ptr() - base.data_ptr()) // 4
    keep[:, off:off + view.shape[1]] = False
    return bool(torch.isnan(base.cpu()[keep]).all())


def glue_inputs(M, N, seed):
    """x with exact zeros, -0.0, tiny negatives (ELU outputs near 0) and values up to +-6"""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((M, N)) * 2).astype(np.float32)
    flat = x.reshape(-1)
    flat[::7] = 0.0
    flat[3::11] = -0.0
    flat[5::13] = -np.float32(10.0) ** -rng.integers(3, 30, size=len(flat[5::13]))
    return x


def _big(k):
    """rows of a case whose elements (k per thread) exceed one pass of elem_grid"""
    return lambda N: elem_pass() * k // N + 37


# (act, slope, M, N, vec): every activation through both instances, LeakyReLU at 0.01 and 0.2, and one grid-stride size
# per instance
GLUE_CASES = [
    (NONE, 0.0, 300, 64, True), (NONE, 0.0, 300, 63, False),
    (ELU, 0.0, 300, 128, True), (ELU, 0.0, 301, 5, False),
    (TANH, 0.0, 200, 36, True), (TANH, 0.0, 200, 36, False),
    (RELU, 0.0, 150, 4, True), (RELU, 0.0, 150, 1, False),
    (LEAKY, 0.01, 120, 256, True), (LEAKY, 0.2, 120, 255, False), (LEAKY, 0.2, 77, 8, True),
    (ELU, 0.0, _big(4), 128, True), (LEAKY, 0.2, _big(1), 127, False),
]


@pytest.mark.parametrize("act,slope,M,N,vec", GLUE_CASES)
@pytest.mark.parametrize("bias", [True, False])
def test_bias_act_and_act_bwd_against_torch(mods, act, slope, M, N, vec, bias):
    """bias_act: y = act(x + b) within 5e-7 of each fp64 value (one fp32 rounding of x + b, which the activations
    carry through with a condition number <= 1, and <= 2 ulp of expm1f / tanhf).  act_bwd: dx = g act'(x) from the
    fp32 output y, within 4 u |g| of torch's fp64 autograd (act' from y: y + 1 and 1 - y^2 round twice); at exact
    zeros both take torch's branch (ReLU' = 0, LeakyReLU' = slope, ELU' = 1)."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    grid_stride = callable(M)
    M = M(N) if grid_stride else M
    inst = 4 if vec else 1
    assert (M * N // inst > elem_pass()) == grid_stride
    x = glue_inputs(M, N, M + N + act)
    b = np.random.default_rng(N).standard_normal(N).astype(np.float32) if bias else None
    xv, _ = dense(M, N, vec, x)
    y, ybase = dense(M, N, vec)
    bd = torch.from_numpy(b).cuda() if bias else None
    torch.cuda.synchronize()
    names = launches(lambda: lib().bias_act(P(xv), xv.stride(0), P(bd), act, slope, P(y), y.stride(0), M, N,
                                            stream()))
    assert names == {f"bias_act_kernel<{inst}>"}, names
    s64 = torch.from_numpy(x).double() + (torch.from_numpy(b).double() if bias else 0)
    ref = act64(s64, act, slope)
    got = y.cpu().double()
    assert outside_ok(y, ybase) and not torch.isnan(got).any()
    err = (got - ref).abs()
    assert bool((err <= 5e-7 * ref.abs() + 1e-37).all()), float((err / ref.abs().clamp(min=1e-37)).max())

    # backward from the forward output of fp64 pre-activations
    x64 = torch.from_numpy(glue_inputs(M, N, M * 3 + N)).double().requires_grad_()
    y64 = act64(x64, act, slope)
    g = np.random.default_rng(M).standard_normal((M, N)).astype(np.float32)
    (y64 * torch.from_numpy(g).double()).sum().backward()
    yd, _ = dense(M, N, vec, y64.detach().float())
    gd, _ = dense(M, N, vec, g)
    dx, dbase = dense(M, N, vec)
    torch.cuda.synchronize()
    names = launches(lambda: lib().act_bwd(P(gd), gd.stride(0), P(yd), yd.stride(0), act, slope, P(dx), dx.stride(0),
                                           M, N, stream()))
    assert names == {f"act_bwd_kernel<{inst}>"}, names
    got = dx.cpu().double()
    assert outside_ok(dx, dbase) and not torch.isnan(got).any()
    err = (got - x64.grad).abs()
    assert bool((err <= 4 * U * torch.from_numpy(g).double().abs() + 1e-37).all())


def test_bias_act_function_against_torch_autograd(mods):
    """BiasActFn forward + backward (act_bwd, then colsum for the bias) against fp64 autograd."""
    ops = mods["ops"]
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(500, 30, generator=gen)
    b = torch.randn(30, generator=gen)
    gw = torch.randn(500, 30, generator=gen, dtype=torch.float64)
    xd, bd = x.cuda().requires_grad_(), b.cuda().requires_grad_()
    y = ops.BiasActFn.apply(xd, bd, LEAKY, 0.2)
    (y * gw.float().cuda()).sum().backward()
    x64, b64 = x.double().requires_grad_(), b.double().requires_grad_()
    r = act64(x64 + b64, LEAKY, 0.2)
    (r * gw).sum().backward()
    assert rel_err(y.detach().cpu(), r.detach()) < 1e-6
    assert rel_err(xd.grad.cpu(), x64.grad) < 1e-6
    assert bool(((bd.grad.cpu().double() - b64.grad).abs() <= 1e-5 * (x64.grad.abs().sum(0))).all())


# ------------------------------------------------------------------------------------------------ concat_dropout
# (M, K1, K2, p, vec, ldg_extra, d1, d2): the <4> instance needs K1, K2 % 4 == 0 and 16-byte aligned rows; K1 % 4 != 0
# or a strided view takes <1>; the gradient's ld differs from K1 + K2 in most cases
CAT_CASES = [
    (300, 64, 36, 0.1, True, 4, True, True),
    (301, 13, 22, 0.5, False, 5, True, True),
    (77, 5, 0, 0.99, False, 0, True, False),
    (200, 128, 0, 0.5, True, 8, True, False),
    (150, 36, 64, 0.1, True, 4, False, True),
    (150, 36, 64, 0.99, True, 0, True, False),
    (90, 7, 9, 0.0, False, 3, True, True),
    (lambda: elem_pass() * 4 // 64 + 11, 32, 32, 0.5, True, 4, True, True),
    (lambda: elem_pass() // 5 + 11, 3, 2, 0.1, False, 1, True, True),
]


@pytest.mark.parametrize("M,K1,K2,p,vec,ldg_extra,w1,w2", CAT_CASES)
def test_concat_dropout_masks_bit_for_bit(mods, M, K1, K2, p, vec, ldg_extra, w1, w2):
    """out = [x1 | x2] * keep / (1 - p) and its backward d1 | d2 = g * keep / (1 - p), keep = u01(seed, r (K1 + K2)
    + c) >= p restated on the host, bit for bit (p = 0: a plain concatenation).  d1 or d2 NULL writes only the
    other.  The last two cases need more than one pass of elem_grid."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    M = M() if callable(M) else M
    K = K1 + K2
    inst = 4 if vec else 1
    assert (M * K // inst > elem_pass()) == (M > 20000)
    rng = np.random.default_rng(K1 * 100 + K2)
    x1 = rng.standard_normal((M, K1)).astype(np.float32)
    x2 = rng.standard_normal((M, K2)).astype(np.float32)
    x1d, _ = dense(M, K1, vec, x1)
    x2d = dense(M, K2, vec, x2)[0] if K2 else None
    out, obase = dense(M, K, vec)
    seed = SEED ^ (K1 << 7)
    torch.cuda.synchronize()
    names = launches(lambda: lib().concat_dropout(P(x1d), x1d.stride(0), K1, P(x2d), x2d.stride(0) if K2 else 0, K2,
                                                  p, seed, P(out), out.stride(0), M, stream()))
    assert names == {f"concat_dropout_kernel<{inst}>"}, names
    xcat = np.concatenate([x1, x2], 1)
    keep = elem_keep(seed, p, M, K) if p > 0 else np.ones((M, K), dtype=bool)
    ref = apply_keep(xcat, keep, p) if p > 0 else xcat
    assert np.array_equal(out.cpu().numpy(), ref) and outside_ok(out, obase)

    g = rng.standard_normal((M, K)).astype(np.float32)
    gbase = torch.full((M, K + ldg_extra + (0 if vec else 1)), NAN)
    off = 0 if vec else 1
    gbase[:, off:off + K] = torch.from_numpy(g)
    gbase = gbase.cuda()
    gd = gbase[:, off:off + K]
    d1, b1 = dense(M, K1, vec) if w1 else (None, None)
    d2, b2 = dense(M, K2, vec) if (w2 and K2) else (None, None)
    torch.cuda.synchronize()
    names = launches(lambda: lib().concat_dropout_bwd(P(gd), gd.stride(0), K1, K2, p, seed, P(d1),
                                                      d1.stride(0) if d1 is not None else 0, P(d2),
                                                      d2.stride(0) if d2 is not None else 0, M, stream()))
    assert names == {f"concat_dropout_bwd_kernel<{inst}>"}, names
    gref = apply_keep(g, keep, p) if p > 0 else g
    if d1 is not None:
        assert np.array_equal(d1.cpu().numpy(), gref[:, :K1]) and outside_ok(d1, b1)
    if d2 is not None:
        assert np.array_equal(d2.cpu().numpy(), gref[:, K1:]) and outside_ok(d2, b2)


def test_concat_dropout_function_against_torch_autograd(mods):
    """ConcatDropoutFn forward + backward against fp64 autograd of cat -> multiply by the restated mask / (1 - p)."""
    ops = mods["ops"]
    gen = torch.Generator().manual_seed(6)
    x1, x2 = torch.randn(200, 21, generator=gen), torch.randn(200, 11, generator=gen)
    gw = torch.randn(200, 32, generator=gen, dtype=torch.float64)
    a, b = x1.cuda().requires_grad_(), x2.cuda().requires_grad_()
    out = ops.ConcatDropoutFn.apply(a, b, 0.2, SEED)
    (out * gw.float().cuda()).sum().backward()
    keep = torch.from_numpy(elem_keep(SEED, 0.2, 200, 32))
    a64, b64 = x1.double().requires_grad_(), x2.double().requires_grad_()
    r = torch.cat([a64, b64], 1) * keep / (1 - 0.2)
    (r * gw).sum().backward()
    assert rel_err(out.detach().cpu(), r.detach()) < 1e-7
    assert rel_err(a.grad.cpu(), a64.grad) < 1e-7 and rel_err(b.grad.cpu(), b64.grad) < 1e-7


# ------------------------------------------------------------------------------------------------ split_planes
SPECIALS = np.array([0.0, -0.0, 1e-40, -3e-39, 1.1754944e-38, -1.1754944e-38, 1e30, -1e30, 1.0, -1.0, 3.0000002,
                     65535.0, 1e-7, -2.5e-20], dtype=np.float32)


# (M, K1, K2, p, concat_chunks, chunk_off): ragged widths, a concatenation with K1 % 4 != 0, masks standing alone and
# placed inside a wider concatenation (chunk_off > 0), p = 0 on special values
SPLIT_CASES = [
    (100, 37, 0, 0.1, 0, 0),
    (257, 13, 22, 0.5, 20, 3),
    (64, 64, 64, 0.99, 40, 5),
    (33, 6, 5, 0.1, 0, 0),
    (40, 14, 0, 0.0, 0, 0),
    (500, 1, 2, 0.5, 9, 7),
]


@pytest.mark.parametrize("M,K1,K2,p,cc,off", SPLIT_CASES)
def test_split_planes_bit_for_bit(mods, M, K1, K2, p, cc, off):
    """split_planes writes split2(dropout([x1 | x2])) exactly: the mask is chunk_hash(seed, r * concat_chunks +
    chunk_off + c / 4) restated on the host (concat_chunks 0: ceil(K / 4) and no offset), 16 bits per element against
    round(p * 65536), the scale fp32 1 / (1 - p); the padding columns up to the next multiple of 4 are 0 in both planes
    and nothing past them is written.  x1 is a strided view (odd ld), so the scalar loads run next to the float4 ones."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    K = K1 + K2
    rng = np.random.default_rng(M + K)
    x = (rng.standard_normal((M, K)) * np.exp(rng.uniform(-8, 8, (M, K)))).astype(np.float32)
    if p == 0:
        x.reshape(-1)[:len(SPECIALS) * 20] = np.tile(SPECIALS, 20)[:x.size]
    x1d, _ = dense(M, K1, False, x[:, :K1])
    x2d = dense(M, K2, True, x[:, K1:])[0] if K2 else None
    n4 = (K + 3) // 4 * 4
    ldo = n4 + 8
    buf = planes_buffer(M, ldo)
    seed = SEED + K
    torch.cuda.synchronize()
    names = launches(lambda: lib().split_planes(P(x1d), x1d.stride(0), K1, P(x2d), x2d.stride(0) if K2 else 0, K2, p,
                                                seed, cc, off, buf.data_ptr(), ldo, M * ldo, M, stream()))
    assert names == {"split_planes_kernel"}, names
    nch = cc if cc > 0 else (K + 3) // 4
    choff = off if cc > 0 else 0
    d = apply_keep(x, planes_keep(seed, p, M, K, nch, choff), p) if p > 0 else x
    check_planes(buf, d, K)


def test_split2_residual_bound_on_special_values():
    """The restated split on +-0, -0.0, subnormals, the smallest normals and +-1e30 (the bits the kernels write are
    checked against it above): |x - hi - lo| <= 2^-17 |x| for normal x (the exhaustive maximum over one binade is
    2^-17.003, see tc_ptx.cuh), and <= 2^-134, half the smallest bf16 subnormal, where lo underflows."""
    rng = np.random.default_rng(0)
    x = np.concatenate([SPECIALS, (rng.standard_normal(100000) * np.exp(rng.uniform(-80, 80, 100000))).astype(np.float32)])
    x = x.astype(np.float32)
    hi, lo = split2(x)
    r = np.abs(x.astype(np.float64) - bf16_up(hi).astype(np.float64) - bf16_up(lo).astype(np.float64))
    assert (r <= np.maximum(2.0 ** -17 * np.abs(x.astype(np.float64)), 2.0 ** -134)).all()
    normal = np.abs(x) >= 2.0 ** -100
    assert (r[normal] <= 2.0 ** -17 * np.abs(x[normal].astype(np.float64))).all()
    assert hi[1] == 0x8000 and lo[1] == 0 and hi[0] == 0 and lo[0] == 0          # -0.0 keeps its sign in hi


def test_masked_dx_epilogue_against_the_restated_mask(mods):
    """planes_linear_bwd_input_masked == the unmasked dX times the restated planes mask (chunk r * concat_chunks +
    (k_off + c) / 4) and the fp32 scale, bit for bit, for p in {0.1, 0.5, 0.99}, a ragged K and k_off > 0."""
    stack = mods["stack"]
    dev = torch.device("cuda", 0)
    torch.manual_seed(3)
    M, N, K, k_off, cc = 257, 130, 130, 64, 70
    dC = stack.split_planes(torch.randn(M, N, device=dev))
    W = torch.randn(N, k_off + K, device=dev)
    plain = stack.planes_linear_bwd_input(dC, W, K, k_off=k_off)[:, :K].cpu().numpy()
    for p in (0.1, 0.5, 0.99):
        seed = SEED + int(p * 100)
        masked = stack.planes_linear_bwd_input(dC, W, K, k_off=k_off, drop_p=p, seed=seed, concat_chunks=cc)
        keep = planes_keep(seed, p, M, K, cc, k_off // 4)
        assert np.array_equal(masked[:, :K].cpu().numpy(), apply_keep(plain, keep, p)), p


# ------------------------------------------------------------------------------------------------ act_bwd_planes
def _abp_ref(g, y, act, slope, p, seed):
    """d = keep(g) * act'(y) in the kernel's fp32 arithmetic (keep: the standalone planes mask, chunk r * ceil(N/4)
    + c / 4)"""
    M, N = g.shape
    d = apply_keep(g, planes_keep(seed, p, M, N, (N + 3) // 4, 0), p) if p > 0 else g.astype(np.float32)
    if y is None or act == NONE:
        return d
    if act == ELU:
        gr = np.where(y > 0, np.float32(1), (y + np.float32(1)).astype(np.float32))
    elif act == RELU:
        gr = np.where(y > 0, np.float32(1), np.float32(0))
    elif act == LEAKY:
        gr = np.where(y > 0, np.float32(1), np.float32(slope))
    else:
        raise AssertionError("no bit-exact restatement: 1 - y * y may be contracted to an FMA")
    return (d * gr.astype(np.float32)).astype(np.float32)


# (M, N, act, y given, p, column sums): N over ragged widths, one and several 128-column groups; M below one 8-row band,
# at it, above it and over 40,000 rows; y NULL and act NONE; sums on and off
ABP_CASES = [
    (1, 1, RELU, True, 0.0, True), (7, 3, LEAKY, True, 0.5, True), (8, 5, NONE, True, 0.0, True),
    (9, 127, ELU, True, 0.1, False), (40001, 128, RELU, True, 0.5, True), (300, 129, LEAKY, True, 0.99, True),
    (40001, 1028, NONE, False, 0.5, True), (9, 1028, ELU, True, 0.0, False), (1, 129, TANH, True, 0.1, True),
    (40001, 3, TANH, True, 0.0, False), (8, 127, ELU, False, 0.0, True), (7, 1, LEAKY, True, 0.1, False),
]


@pytest.mark.parametrize("M,N,act,with_y,p,sums", ABP_CASES)
def test_act_bwd_planes_against_restatement_and_fp64(mods, M, N, act, with_y, p, sums):
    """Planes of d = keep(g) act'(y) bit for bit against the restated mask and split (TANH, whose 1 - y^2 may be an
    FMA, against fp64 within 2^-17 + 3 u of the largest entry); padding columns 0 in both planes although g and y hold
    values there.  Column sums: g holds multiples of 1/16 up to 2 and act' is 0, 1 or 0.25 (or the mask's exact
    scale 2), so every partial sum is exact and the sums equal fp64 exactly; with other masks and activations within
    the recursive-sum bound (rows per band + 8 + bands) u sum |d|.  Two runs are bit-identical; nothing is written past
    N columns of the sums."""
    lib, P, stream, SpgnnError = mods["lib"], mods["ptr"], mods["stream"], mods["SpgnnError"]
    rng = np.random.default_rng(M * 7 + N)
    n4 = (N + 3) // 4 * 4
    slope = 0.25
    exact = act in (NONE, RELU, LEAKY) and p in (0.0, 0.5)
    gfull = (rng.integers(-32, 33, size=(M, n4 + 4)) / 16).astype(np.float32)
    gfull[:, N:] = 5.0                                        # padding values the kernel must not pass on
    yfull = rng.standard_normal((M, n4 + 4)).astype(np.float32)
    if act == TANH:
        yfull = np.tanh(yfull).astype(np.float32)
    if act == ELU:
        yfull = np.where(yfull > 0, yfull, np.expm1(yfull)).astype(np.float32)
    yfull.reshape(-1)[::9] = 0.0
    gd = torch.from_numpy(gfull).cuda()
    yd = torch.from_numpy(yfull).cuda() if with_y else None
    ldo = n4 + 4
    buf = planes_buffer(M, ldo)
    cs = torch.full((N + 4,), NAN, device="cuda") if sums else None
    ws = torch.full((int(lib().act_bwd_planes_ws(N)) // 4,), NAN, device="cuda") if sums else None
    seed = SEED ^ N

    def run():
        lib().act_bwd_planes(P(gd), gd.stride(0), P(yd), yd.stride(0) if with_y else 0, act, slope, p, seed,
                             buf.data_ptr(), ldo, M * ldo, M, N, P(cs), P(ws), stream())

    torch.cuda.synchronize()
    names = launches(run)
    assert names == ({"act_bwd_planes_kernel<true>", "sum_bands_kernel"} if sums else {"act_bwd_planes_kernel<false>"})
    g = gfull[:, :N]
    y = yfull[:, :N] if with_y else None
    if act == TANH:
        keep = planes_keep(seed, p, M, N, (N + 3) // 4, 0) if p > 0 else np.ones((M, N), bool)
        d64 = np.where(keep, g.astype(np.float64) * float(scale32(p)) if p > 0 else g, 0.0) * (
            1.0 - y.astype(np.float64) ** 2)
        b = buf.cpu().numpy().view(np.uint16)
        got = bf16_up(b[0, :, :N]).astype(np.float64) + bf16_up(b[1, :, :N]).astype(np.float64)
        assert np.abs(got - d64).max() <= (2.0 ** -17 + 3 * U) * np.abs(d64).max()
        assert (b[:, :, N:n4] == 0).all() and (b[:, :, n4:] == BF16_NAN).all()
    else:
        d64 = _abp_ref(g, y, act, slope, p, seed).astype(np.float64)
        check_planes(buf, d64.astype(np.float32), N)
    if sums:
        got = cs.cpu().numpy()
        assert np.isnan(got[N:]).all(), "written past N column sums"
        ref = d64.sum(0)
        if exact:
            assert np.array_equal(got[:N].astype(np.float64), ref), "column sums (exact inputs)"
        else:
            bands = min(-(-1184 // -(-n4 // 128)), -(-M // 8))
            depth = -(-M // bands) + 8 + bands
            assert (np.abs(got[:N] - ref) <= depth * U * np.abs(d64).sum(0) + 1e-30).all(), "column sums"
        first = got.copy()
        cs.fill_(NAN)
        run()
        assert np.array_equal(cs.cpu().numpy(), first, equal_nan=True), "run-to-run"


def test_act_bwd_planes_refusals_touch_nothing(mods):
    """A misaligned g, ldg < the padded row, column sums without a workspace and p >= 1 are host-side SpgnnErrors
    raised before any launch: planes and sums keep their prefill."""
    lib, P, stream, SpgnnError = mods["lib"], mods["ptr"], mods["stream"], mods["SpgnnError"]
    M, N = 40, 10
    g = torch.randn(M, 16, device="cuda")
    buf = planes_buffer(M, 16)
    cs = torch.full((N,), NAN, device="cuda")
    ws = torch.empty(int(lib().act_bwd_planes_ws(N)), dtype=torch.uint8, device="cuda")
    bad = [
        dict(gp=g.data_ptr() + 4, ldg=16, w=ws, p=0.0, match="16-byte aligned"),
        dict(gp=g.data_ptr(), ldg=8, w=ws, p=0.0, match="padded"),
        dict(gp=g.data_ptr(), ldg=16, w=None, p=0.0, match="workspace"),
        dict(gp=g.data_ptr(), ldg=16, w=ws, p=1.0, match="dropout p"),
    ]
    for b in bad:
        with pytest.raises(SpgnnError, match=b["match"]):
            lib().act_bwd_planes(b["gp"], b["ldg"], None, 0, NONE, 0.0, b["p"], 1, buf.data_ptr(), 16, M * 16, M, N,
                                 P(cs), P(b["w"]), stream())
    torch.cuda.synchronize()
    assert (buf.cpu() == BF16_NAN).all() and torch.isnan(cs).all()


def test_planes_linear_and_mlp_backward_against_fp64_autograd(mods):
    """PlanesLinearFn backward (act_bwd_planes with and without the bias sums) and MlpDropFn (the hidden dropout mask
    in split_planes forward and act_bwd_planes backward, the restated planes mask) against fp64 autograd.  The planes
    GEMMs carry ~2^-17 relative per operand, hence the 1e-4 bar of the other planes tests."""
    ops = mods["ops"]
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(300, 40, generator=gen)
    for bias in (True, False):
        # 28 outputs: the gradient of y has 16-byte rows, which is what takes the fused pass
        W = torch.randn(28, 40, generator=gen) * 0.2
        b = torch.randn(28, generator=gen) if bias else None
        gw = torch.randn(300, 28, generator=gen, dtype=torch.float64)
        xd, Wd = x.cuda().requires_grad_(), W.cuda().requires_grad_()
        bd = b.cuda().requires_grad_() if bias else None
        y = ops.PlanesLinearFn.apply(xd, None, Wd, bd, ELU, 0.0)
        names = launches(lambda: (y * gw.float().cuda()).sum().backward())
        assert f"act_bwd_planes_kernel<{'true' if bias else 'false'}>" in names, names
        x64, W64 = x.double().requires_grad_(), W.double().requires_grad_()
        b64 = b.double().requires_grad_() if bias else None
        r = F.elu(x64 @ W64.T + (b64 if bias else 0))
        (r * gw).sum().backward()
        assert rel_err(xd.grad.cpu(), x64.grad) < 1e-4 and rel_err(Wd.grad.cpu(), W64.grad) < 1e-4
        if bias:
            assert rel_err(bd.grad.cpu(), b64.grad) < 1e-4

    p, seed, slope = 0.3, SEED + 5, 0.01
    W0, b0 = torch.randn(23, 40, generator=gen) * 0.2, torch.randn(23, generator=gen)
    W3, b3 = torch.randn(17, 23, generator=gen) * 0.2, torch.randn(17, generator=gen)
    gw = torch.randn(300, 17, generator=gen, dtype=torch.float64)
    leaves = [t.cuda().requires_grad_() for t in (x, W0, b0, W3, b3)]
    y = ops.MlpDropFn.apply(*leaves, LEAKY, slope, p, seed)
    names = launches(lambda: (y * gw.float().cuda()).sum().backward())
    assert {"act_bwd_planes_kernel<true>", "sum_bands_kernel"} <= names, names
    keep = torch.from_numpy(planes_keep(seed, p, 300, 23, (23 + 3) // 4, 0)).double()
    l64 = [t.double().requires_grad_() for t in (x, W0, b0, W3, b3)]
    h = F.leaky_relu(l64[0] @ l64[1].T + l64[2], slope)
    r = F.leaky_relu((h * keep / (1 - p)) @ l64[3].T + l64[4], slope)
    assert rel_err(y.detach().cpu(), r.detach()) < 1e-4
    (r * gw).sum().backward()
    for a, b_ in zip(leaves, l64):
        assert rel_err(a.grad.cpu(), b_.grad) < 1e-4


# ------------------------------------------------------------------------------------------------ colsum
@pytest.mark.parametrize("M", [1, 591, 592, 593, 300001])
@pytest.mark.parametrize("N", [1, 22, 128, 129, 1028])
def test_colsum_against_fp64(mods, M, N):
    """spgnn_colsum over a strided X (odd ld, misaligned base): with multiples of 1/16 up to 2 every partial sum is
    exact and the sums equal fp64 exactly; with random floats within (rows per band + parts / 32 + 5) u sum |x| of
    fp64 (the depth of the band / lane / butterfly tree) and bit-identical run to run.  M < 592 gives one row per band,
    M >= 592 partial bands; N > 128 several column blocks."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    gen = torch.Generator(device="cuda").manual_seed(M + N)
    base = torch.full((M, N + 3), NAN, device="cuda")
    X = base[:, 1:N + 1]
    out = torch.full((N + 4,), NAN, device="cuda")
    ws = torch.full((int(lib().colsum_ws(N)) // 4,), NAN, device="cuda")

    def run():
        lib().colsum(P(X), X.stride(0), M, N, P(out), P(ws), stream())

    X.copy_(torch.randint(-32, 33, (M, N), device="cuda", generator=gen).float() / 16)
    names = launches(run)
    assert names == {"colsum_partial_kernel", "colsum_final_kernel"}
    ref = X.double().sum(0)
    got = out.cpu()
    assert torch.isnan(got[N:]).all()
    assert torch.equal(got[:N].double(), ref.cpu()), "exact inputs"

    X.copy_(torch.randn(M, N, device="cuda", generator=gen) * 3)
    out.fill_(NAN)
    run()
    first = out.clone()
    parts = min(M, 592)
    rpb = -(-M // parts)
    depth = rpb + -(-(-(-M // rpb)) // 32) + 5
    err = (first[:N].double() - X.double().sum(0)).abs()
    assert bool((err <= depth * U * X.double().abs().sum(0) + 1e-30).all())
    out.fill_(NAN)
    run()
    assert torch.equal(out[:N], first[:N]) and bool(torch.isnan(out[N:]).all()), "run-to-run"


# ------------------------------------------------------------------------------------------------ masked CE
def ce_call(mods, logits, y, mask, rate, seed, cw, N, C, ldd_extra=3):
    """spgnn_masked_ce_fwd + _bwd (scale 1); returns (sums, dlogits view, its base)"""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    sums = torch.full((2,), NAN, dtype=torch.float64, device="cuda")
    dbase = torch.full((N, C + ldd_extra), NAN, device="cuda")
    dl = dbase[:, :C]

    def run():
        lib().masked_ce_fwd(P(logits), logits.stride(0), C, P(y), P(mask), rate, seed, P(cw), N, P(sums), stream())
        lib().masked_ce_bwd(P(logits), logits.stride(0), C, P(y), P(mask), rate, seed, P(cw), P(sums), 1.0, N, P(dl),
                            dl.stride(0), stream())

    torch.cuda.synchronize()
    assert launches(run) == {"masked_ce_fwd_kernel", "masked_ce_bwd_kernel"}
    return sums.cpu(), dl.cpu(), dbase.cpu()


@pytest.mark.parametrize("C,N,drawn", [(2, 3000, False), (22, 5000, True), (40, 2000, False), (22, 310000, True),
                                       (2, 310000, False), (40, 7000, True)])
def test_masked_ce_against_torch(mods, C, N, drawn):
    """Loss and gradient against F.cross_entropy(logits[keep], y[keep], weight=) in fp64, logits with ld > C,
    non-uniform class weights.  The drawn mask (y != 0 or u01(seed, i) < rate, restated on the host) is pinned exactly
    through sums[1] = sum of the kept class weights, which a double accumulates exactly in any order; the rate is one
    of the drawn u01 values, so '<' and '<=' differ at that node.  N = 310,000 is more than one pass of the grid
    (sm_count x 8 blocks of 256 threads).  Loss within 2e-6 (per-row nll rounds a few fp32 terms of size <= 10),
    gradient within 1e-6 of its largest entry; rows not kept get exact zeros."""
    rng = np.random.default_rng(C * N)
    assert (N > _sms() * 8 * 256) == (N == 310000)
    logits = (rng.standard_normal((N, C)) * 2).astype(np.float32)
    yl = np.where(rng.random(N) < 0.1, rng.integers(1, C, N), 0).astype(np.int64)
    cw = rng.uniform(0.1, 2.0, C).astype(np.float32)
    seed = SEED + C
    if drawn:
        u = u01(seed, np.arange(N))
        cand = np.nonzero((yl == 0) & (u > 0.1) & (u < 0.3))[0]
        rate = float(u[cand[0]])
        keep = (yl != 0) | (u < np.float32(rate))
        assert not keep[cand[0]]
        mask_d = None
    else:
        rate = 1.0
        keep = rng.random(N) < 0.4
        mask_d = torch.from_numpy(keep.astype(np.uint8)).cuda()
    lbase = torch.full((N, C + 5), NAN)
    lbase[:, :C] = torch.from_numpy(logits)
    ld = lbase.cuda()[:, :C]
    sums, dl, dbase = ce_call(mods, ld, torch.from_numpy(yl).cuda(), mask_d, rate, seed, torch.from_numpy(cw).cuda(),
                              N, C)
    assert float(sums[1]) == float(cw[yl[keep]].astype(np.float64).sum()), "kept set"
    l64 = torch.from_numpy(logits).double().requires_grad_()
    kt = torch.from_numpy(keep)
    ref = F.cross_entropy(l64[kt], torch.from_numpy(yl)[kt], weight=torch.from_numpy(cw).double())
    ref.backward()
    loss, ref = float(sums[0] / sums[1]), float(ref.detach())
    assert abs(loss - ref) <= 2e-6 * abs(ref)
    assert not torch.isnan(dl).any() and torch.isnan(dbase[:, C:]).all()
    assert torch.equal(dl[~kt], torch.zeros_like(dl[~kt]))
    assert rel_err(dl, l64.grad) < 1e-6


def test_masked_ce_with_nothing_kept_matches_torch_on_an_empty_selection(mods):
    """No node kept: torch's weighted cross-entropy over an empty selection is NaN with an all-zero gradient (checked
    here, not assumed); the kernels give sums (0, 0), hence a NaN loss, and write zeros to every row."""
    N, C = 500, 22
    gen = torch.Generator().manual_seed(2)
    logits = torch.randn(N, C, generator=gen)
    y = torch.randint(0, C, (N,), generator=gen)
    cw = torch.rand(C, generator=gen) + 0.1
    l64 = logits.double().requires_grad_()
    keep = torch.zeros(N, dtype=torch.bool)
    ref = F.cross_entropy(l64[keep], y[keep], weight=cw.double())
    ref.backward()
    assert torch.isnan(ref) and torch.equal(l64.grad, torch.zeros_like(l64.grad))
    # given mask of zeros, and a drawn mask with every label 0 and rate 0
    for mask, yy, rate in ((torch.zeros(N, dtype=torch.uint8, device="cuda"), y, 1.0),
                           (None, torch.zeros_like(y), 0.0)):
        sums, dl, _ = ce_call(mods, logits.cuda(), yy.cuda(), mask, rate, 9, cw.cuda(), N, C)
        assert sums.tolist() == [0.0, 0.0] and np.isnan(float(sums[0] / sums[1]))
        assert torch.equal(dl, torch.zeros_like(dl))


def test_masked_ce_function_against_torch_autograd(mods):
    """MaskedCEFn forward + backward (given mask) against fp64 autograd of F.cross_entropy on the selection."""
    ops = mods["ops"]
    gen = torch.Generator().manual_seed(5)
    N, C = 4000, 22
    logits = torch.randn(N, C, generator=gen) * 2
    y = torch.randint(0, C, (N,), generator=gen)
    cw = torch.rand(C, generator=gen) + 0.1
    keep = torch.rand(N, generator=gen) < 0.5
    ld = logits.cuda().requires_grad_()
    loss = ops.MaskedCEFn.apply(ld, y.cuda(), keep.cuda(), 1.0, 0, cw.cuda(), None)
    (loss * 3.0).backward()
    l64 = logits.double().requires_grad_()
    ref = F.cross_entropy(l64[keep], y[keep], weight=cw.double())
    (ref * 3.0).backward()
    assert abs(float(loss.detach()) - float(ref.detach())) <= 2e-6 * abs(float(ref.detach()))
    assert rel_err(ld.grad.cpu(), l64.grad) < 1e-6


# ------------------------------------------------------------------------------------------------ segmented_argmax
@pytest.mark.parametrize("C", [2, 22])
def test_segmented_argmax_first_index_with_planted_ties(mods, C):
    """Trees of 1, 255, 256, 257 and 1,500 nodes (the kernel's 256 threads take several nodes each in the last two).
    Per tree and class the winner's logit is raised by 3 over random logits, so fp32 cannot reorder winners; copies of
    the winning row are planted at nodes another lane, another warp, or the same thread in a later pass handles, and
    the lowest node id must win, as numpy's argmax of the fp64 softmax picks it."""
    lib, P, stream = mods["lib"], mods["ptr"], mods["stream"]
    sizes = [1, 255, 256, 257, 1500]
    rng = np.random.default_rng(C)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(off[-1])
    logits = rng.standard_normal((N, C)).astype(np.float32)
    planted = 0
    for t, n in enumerate(sizes):
        base = int(off[t])
        for c in range(1, C):
            w = int(rng.integers(0, min(n, 40)))
            logits[base + w, c] += 3.0
            for other in (w + 1, w + 33, w + 256):          # another lane, another warp, the same thread's next pass
                if other < n and (c + other) % 2 == 0:
                    logits[base + other] = logits[base + w]
                    planted += 1
    assert planted > 5
    # the winners stand apart from every row that is not a copy of them by far more than fp32 rounding
    l64 = logits.astype(np.float64)
    prob = np.exp(l64 - l64.max(1, keepdims=True))
    prob /= prob.sum(1, keepdims=True)
    for t in range(len(sizes)):
        for c in range(1, C):
            q = np.unique(prob[off[t]:off[t + 1], c])
            assert len(q) == 1 or q[-1] - q[-2] > 1e-4 * q[-1], (t, c)
    B = len(sizes)
    lbase = torch.full((N, C + 3), NAN)
    lbase[:, :C] = torch.from_numpy(logits)
    ld = lbase.cuda()[:, :C]
    out = torch.full((B, C - 1), -7, dtype=torch.int64, device="cuda")
    off_d = torch.from_numpy(off).cuda()
    torch.cuda.synchronize()
    names = launches(lambda: lib().segmented_argmax(P(ld), ld.stride(0), C, P(off_d), B, P(out), stream()))
    assert names == {"segmented_argmax_kernel"}
    ref = np.array([[off[t] + np.argmax(prob[off[t]:off[t + 1], c]) for c in range(1, C)] for t in range(B)])
    assert np.array_equal(out.cpu().numpy(), ref)
