"""-m gpu: the BatchNorm+ReLU (+ max-pool) kernels, their backward and the channel-slice copy / add, exact or tightly bounded
against fp64 (tests/ew_check.py), at every call form UNetEngine.forward / backward makes.

Exact: the forward activation, the pooled values and window positions (fmaf emulated exactly; planted inputs take its
double-rounding branch and windows hold ties), maxpool2x2, nhwc_copy / nhwc_add, dy of a frozen BatchNorm, and in the sparse
regime dgamma / dbeta (small-integer y, g1, g_pool at low density, integer mean, power-of-two rstd and gamma: every partial
sum is an integer below 2^24, whatever the order). Dense regime (y ~ N(mu, sigma), |mu| / sigma up to 30, so
Sum da y - mean Sum da cancels): dgamma / dbeta within ew_check.sum_bounds and dy within ew_check.dy_bound, element by element.

Buffers are laid out as the engine lays them out - the activation in the left half of a concat buffer, dy written over y,
g1 the skip half of the concat gradient - with sentinels in every channel and element a call must not touch. Shapes cover
every channel count the networks use, ragged pixel counts, totals on both sides of the grid strides (from the formulas of
ew_check, asserted per case) and config 2's level 0 at full size. The bounds and the edge cases assume the default grid: the
module skips when an environment variable changes it."""
import os

import pytest
import torch

import conv_check as C
import ew_check as E

pytestmark = pytest.mark.gpu

_ENV = [v for v in E.GRID_ENV if v in os.environ]
if _ENV:
    pytest.skip(f"{', '.join(_ENV)} set: the launch grid differs from the one the bounds and edge cases are derived from",
                allow_module_level=True)

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
SPARSE, DENSE = "sparse", "dense"
CHUNK = 1 << 25   # elements per fp64 reference chunk


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200  # noqa: F401
    from unet_torch_b200 import ops as _ops

    return _ops


def _report(form, **kv):
    print(f"[bn_relu_exact] {form}: " + ", ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}" for k, v in kv.items()))


def _chunks(n, h, w, c):
    step = max(1, CHUNK // (h * w * c))
    return [slice(i, min(n, i + step)) for i in range(0, n, step)]


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# ------------------------------------------------------------------------------------------------ operands
def _ints(shape, m, density, g):
    v = torch.randint(-m, m + 1, shape, generator=g, device="cuda")
    return (v * (torch.rand(shape, generator=g, device="cuda") < density)).to(BF16)


def _bn_params(c, regime, g, y=None):
    """(gamma, mean, rstd, scale, shift) fp32. Sparse: power-of-two gamma and rstd, integer mean. Dense: batch statistics of y."""
    if regime == SPARSE:
        gamma = torch.exp2(torch.randint(-1, 2, (c,), generator=g, device="cuda").float())
        gamma = gamma * torch.where(torch.rand(c, generator=g, device="cuda") < 0.25, -1.0, 1.0)
        mean = torch.randint(-1, 2, (c,), generator=g, device="cuda").float()
        rstd = torch.exp2(torch.randint(-1, 2, (c,), generator=g, device="cuda").float())
    else:
        gamma = (torch.rand(c, generator=g, device="cuda") + 0.5) * torch.where(torch.rand(c, generator=g, device="cuda") < 0.25,
                                                                                 -1.0, 1.0)
        yd = y.reshape(-1, c).to(F64)
        mean = yd.mean(0).float()
        rstd = (yd.var(0, unbiased=False) + 1e-5).rsqrt().float()
    beta = torch.randn(c, generator=g, device="cuda") * 0.3
    scale = (gamma.double() * rstd.double()).float()
    shift = beta - mean * scale
    return gamma, mean, rstd, scale, shift


def _y(n, h, w, c, regime, g):
    if regime == SPARSE:
        return _ints((n, h, w, c), 3, 0.3, g)
    sigma = torch.exp2(torch.rand(c, generator=g, device="cuda") * 4 - 2)
    ratio = torch.rand(c, generator=g, device="cuda") * 60 - 30
    ratio[:2] = torch.tensor([30.0, -30.0], device="cuda")
    y = torch.randn((n, h, w, c), generator=g, device="cuda") * sigma + ratio * sigma
    return y.to(BF16)


def _grad(shape, regime, g):
    return _ints(shape, 4, 0.3, g) if regime == SPARSE else torch.randn(shape, generator=g, device="cuda").to(BF16)


def _plant_ties(y, g):
    """Equal values in a share of the windows: positions 0 = 1 and 2 = 3."""
    for (r0, c0), (r1, c1) in (((0, 0), (0, 1)), ((1, 0), (1, 1))):
        pick = torch.rand(y[:, r0::2, c0::2].shape[:-1], generator=g, device="cuda") < 0.2
        dst = y[:, r1::2, c1::2]
        dst[pick] = y[:, r0::2, c0::2][pick]


# ------------------------------------------------------------------------------------------------ shapes
WIDTHS = [64, 128, 256, 512, 1024]


def _edge_shapes(kind, pool, c=64):
    """(n, h, w) with the work-item total one item-row (C / 8 items) below, at and above the grid stride and 4 x stride of
    `kind`'s grid at its cap, for channel count c."""
    cgs = c // 8
    stride = (E.EW_MAX_BLOCKS if kind != "bwd" else E.BWD_MAX_BLOCKS) * E.EW_THREADS
    out = []
    for mult in sorted({1, E.UNROLL[pool]}):
        base = mult * stride // cgs          # pixels (or windows) at the edge
        for d in (-1, 0, 1):
            out.append((1, 2, 2 * (base + d)) if pool else (1, 1, base + d))
    return out


def _assert_on_edge(kind, n, h, w, c, pool):
    items = E.work_items(n, h, w, c, pool)
    _, stride = E.grid(kind, items)
    assert stride == (E.EW_MAX_BLOCKS if kind != "bwd" else E.BWD_MAX_BLOCKS) * E.EW_THREADS
    assert any(abs(items - m * stride) <= c // 8 for m in (1, 4)), (items, stride)


FWD_CASES = ([(2, 6, 10, c) for c in WIDTHS] + [(16, 32, 32, 2048), (1, 2, 2, 64), (3, 2, 6, 128)] +
             [s + (64,) for s in _edge_shapes("fwd", True)])
FWD_PLAIN_ONLY = [(1, 1, 3, 64), (1, 3, 5, 256), (3, 5, 7, 512)] + [s + (64,) for s in _edge_shapes("fwd", False)]


def _shape_id(s):
    return "x".join(map(str, s))


# ------------------------------------------------------------------------------------------------ forward
def _check_fwd(ops, n, h, w, c, pool, layout, seed):
    g = _gen(seed)
    y = _y(n, h, w, c, DENSE, g)
    if pool:
        _plant_ties(y, g)
    gamma, mean, rstd, scale, shift = _bn_params(c, DENSE, g, y)
    E.plant_midpoints(scale, shift, y, torch.Generator().manual_seed(seed), channels=min(8, c))
    if layout == "canvas" or pool:
        cv, a = E.canvas2(n, h, w, c)
    else:
        abuf, a = E.guarded((n, h, w, c), BF16)
    pooled = idx = None
    if pool:
        pbuf, pooled = E.guarded((n, h // 2, w // 2, c), BF16)
        ibuf, idx = E.guarded((n, h // 2, w // 2, c), torch.uint8)
    ops.bn_relu_fwd(y, scale, shift, a, pooled, idx)
    mids = 0
    for sl in _chunks(n, h, w, c):
        want, _, mid = E.bn_relu_fwd(y[sl], scale, shift)
        mids += int(mid.sum())
        E.assert_equal(a[sl], want, "a")
        if pool:
            pv, pi = E.maxpool2x2(a[sl])   # the kernel pools the bf16 values it stores: a itself is already checked
            E.assert_equal(pooled[sl], pv, "pooled")
            E.assert_equal(idx[sl], pi, "pool_idx")
        del want, mid
    if layout == "canvas" or pool:
        E.assert_right_half(cv, "a")
    else:
        E.assert_guard(abuf, a.numel(), "a")
    if pool:
        E.assert_guard(pbuf, pooled.numel(), "pooled")
        E.assert_guard(ibuf, idx.numel(), "pool_idx")
    assert mids > 0, "no element took the double-rounding branch of fmaf"
    _report(f"fwd {'pooled' if pool else 'plain'} {layout} {_shape_id((n, h, w, c))}", midpoint_share=mids / y.numel())


@pytest.mark.parametrize("shape", FWD_CASES, ids=_shape_id)
@pytest.mark.parametrize("form", ["plain", "plain_canvas", "pooled"])
def test_bn_relu_fwd_exact(ops, shape, form):
    n, h, w, c = shape
    if form == "pooled" and shape[:3] in _edge_shapes("fwd", True):
        _assert_on_edge("fwd", n, h, w, c, True)
    _check_fwd(ops, n, h, w, c, form == "pooled", "canvas" if form != "plain" else "contig", seed=hash(shape) % 1000)


@pytest.mark.parametrize("shape", FWD_PLAIN_ONLY, ids=_shape_id)
def test_bn_relu_fwd_plain_ragged_and_edges_exact(ops, shape):
    n, h, w, c = shape
    if shape[:3] in _edge_shapes("fwd", False):
        _assert_on_edge("fwd", n, h, w, c, False)
    _check_fwd(ops, n, h, w, c, False, "contig", seed=7 + w)


@pytest.mark.parametrize("pool", [False, True], ids=["plain", "pooled"])
def test_bn_relu_fwd_full_size_exact(ops, pool):
    """Config 2, level 0: 16 x 512 x 512 x 64."""
    _check_fwd(ops, 16, 512, 512, 64, pool, "canvas", seed=21 + pool)
    torch.cuda.empty_cache()


@pytest.mark.parametrize("with_idx", [False, True])
@pytest.mark.parametrize("shape", [(2, 6, 10, 64), (1, 2, 2, 1024), (16, 32, 32, 2048)] +
                         [s + (64,) for s in _edge_shapes("ew", True)], ids=_shape_id)
def test_maxpool2x2_exact(ops, shape, with_idx):
    """Folded inference: the input is the left half of a concat buffer whose right half is NaN; some inputs are NaN too
    (a NaN wins) and windows hold ties."""
    n, h, w, c = shape
    g = _gen(31 + c)
    cv, a = E.canvas2(n, h, w, c)
    a.copy_(torch.relu(torch.randn((n, h, w, c), generator=g, device="cuda")).to(BF16))
    _plant_ties(a, g)
    nan = torch.rand((n, h, w, c), generator=g, device="cuda") < 0.01
    a[nan] = float("nan")
    pbuf, pooled = E.guarded((n, h // 2, w // 2, c), BF16)
    ibuf = idx = None
    if with_idx:
        ibuf, idx = E.guarded((n, h // 2, w // 2, c), torch.uint8)
    ops.maxpool2x2(a, pooled, idx)
    pv, pi = E.maxpool2x2(a)
    E.assert_equal(pooled, pv, "pooled")
    E.assert_guard(pbuf, pooled.numel(), "pooled")
    if with_idx:
        E.assert_equal(idx, pi, "pool_idx")
        E.assert_guard(ibuf, idx.numel(), "pool_idx")
    assert bool((cv[..., c:].view(torch.int16) == E.BF16_SENTINEL).all())


# ------------------------------------------------------------------------------------------------ backward
class FakeSyncBN:
    """The part of DataParallelContext that bn_relu_bwd uses, for one GPU: no fused rows path, and an all-reduce that adds
    a known second rank's sums."""

    def __init__(self, other):
        self.other = other

    def supports_rows(self, c):
        return False

    def all_reduce_sum(self, sums):
        sums += self.other


def _check_bwd(ops, n, h, w, c, pool, regime, form, seed):
    """One bn_relu_bwd call in `form` ('plain', 'plain_canvas', 'pooled_skip', 'frozen', 'syncbn') against the fp64 reference.
    Returns the worst error of (dgamma, dbeta, dy) as a fraction of its bound."""
    g = _gen(seed)
    y = _y(n, h, w, c, regime, g)
    if pool:
        _plant_ties(y, g)
    gamma, mean, rstd, scale, shift = _bn_params(c, regime, g, y)
    if regime == DENSE:
        E.plant_midpoints(scale, shift, y, torch.Generator().manual_seed(seed), channels=8)
    if form == "frozen":  # eval() under autograd: the statistics are the running ones
        rm = torch.randint(-2, 3, (c,), generator=g, device="cuda").float() if regime == SPARSE else mean
        rv = torch.rand(c, generator=g, device="cuda") + 0.5
        mean, rstd = torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
        ops.bn_eval_stats(rm, rv, 1e-5, mean, rstd)
        scale = (gamma.double() * rstd.double()).float()
    g1 = _grad((n, h, w, c), regime, g)
    g_pool = idx = None
    if pool:  # the forward above: its positions, and the skip half of the concat gradient as g1
        cva, a = E.canvas2(n, h, w, c)
        pooled = torch.empty((n, h // 2, w // 2, c), dtype=BF16, device="cuda")
        idx = torch.empty((n, h // 2, w // 2, c), dtype=torch.uint8, device="cuda")
        ops.bn_relu_fwd(y, scale, shift, a, pooled, idx)
        g_pool = _grad(pooled.shape, regime, g)
    if pool or form == "plain_canvas":
        cvg, g1s = E.canvas2(n, h, w, c)
        g1s.copy_(g1)
        g1 = g1s
    y_in = y.clone()
    dgb, dgamma = E.guarded((c,), F32)
    dbb, dbeta = E.guarded((c,), F32)
    count, allreduce, other = n * h * w, None, None
    if form == "syncbn":
        other = torch.randint(-1000, 1000, (2 * c,), generator=g, device="cuda").double()
        allreduce, count = FakeSyncBN(other), 2 * n * h * w
    ops.bn_relu_bwd(g1, g_pool, idx, y, gamma, scale, shift, mean, rstd, y, dgamma, dbeta, count=count, allreduce=allreduce,
                    frozen=form == "frozen")   # dy written over y, as in the engine
    dy = y
    # reference: pass 1 the exact sums, pass 2 dy
    sums = torch.zeros((4, c), dtype=F64, device="cuda")
    for sl in _chunks(n, h, w, c):
        sums += E.bwd_sums(E.bwd_da(y_in[sl], g1[sl], None if g_pool is None else g_pool[sl], None if idx is None else idx[sl],
                                    scale, shift), y_in[sl])
    k = E.terms_per_thread(n, h, w, c, pool)
    bg, bb = E.sum_bounds(sums, mean, rstd, k)
    rg, rb = E.param_grads(sums, mean, rstd)
    worst = {}
    exact_params = regime == SPARSE and form != "frozen"
    if exact_params:
        lim = 2.0 ** 24
        assert float(sums[2].max()) < lim and float((rstd.double() * (sums[3] + mean.double().abs() * sums[2])).max()) < lim, \
            "sparse: a partial sum may reach 2^24; the case breaks its regime"
        E.assert_equal(dgamma, rg, "dgamma")
        E.assert_equal(dbeta, rb, "dbeta")
        worst["dgamma"] = worst["dbeta"] = 0.0
    else:
        worst["dgamma"] = E.assert_within(dgamma, rg, bg, "dgamma")
        worst["dbeta"] = E.assert_within(dbeta, rb, bb, "dbeta")
    E.assert_guard(dgb, c, "dgamma")
    E.assert_guard(dbb, c, "dbeta")
    # the apply pass sums: exact (sparse) or within bg / bb of exact; zero when frozen; the second rank's added under SyncBN
    if form == "frozen":
        app = torch.zeros((2, c), dtype=F64, device="cuda")
    else:
        app = torch.stack([rb, rg])
        if other is not None:
            app = app + other.view(2, c)
    sum_err = regime == DENSE and form != "frozen"
    worst["dy"] = 0.0
    for sl in _chunks(n, h, w, c):
        da = E.bwd_da(y_in[sl], g1[sl], None if g_pool is None else g_pool[sl], None if idx is None else idx[sl], scale, shift)
        if form == "frozen":
            k1 = (gamma.double() * rstd.double()).float().double()
            E.assert_equal(dy[sl], E.to_bf16((k1 * da).to(F32).to(F64)), "dy (frozen)")
            continue
        ref, mag = E.dy_ref(da, y_in[sl], gamma, mean, rstd, app, count)
        bound = E.dy_bound(ref, mag, y_in[sl], gamma, mean, rstd, count, bg if sum_err else None, bb if sum_err else None)
        worst["dy"] = max(worst["dy"], E.assert_within(dy[sl], ref, bound, "dy"))
        del da, ref, mag, bound
    if pool or form == "plain_canvas":
        assert bool((cvg[..., c:].view(torch.int16) == E.BF16_SENTINEL).all()), "g1 canvas: the other half was written"
    if pool:
        E.assert_right_half(cva, "a")
    return worst


BWD_SHAPES = ([(2, 6, 10, c) for c in WIDTHS] + [(16, 32, 32, 2048), (1, 2, 2, 64), (3, 2, 6, 128)])
BWD_EDGES_PLAIN = [s + (64,) for s in _edge_shapes("bwd", False)] + [(1, 1, 3, 64), (1, 3, 5, 256)]
BWD_EDGES_POOL = [s + (64,) for s in _edge_shapes("bwd", True)]


@pytest.mark.parametrize("regime", [SPARSE, DENSE])
@pytest.mark.parametrize("shape", BWD_SHAPES, ids=_shape_id)
@pytest.mark.parametrize("pool", [False, True], ids=["plain", "pooled"])
def test_bn_relu_bwd_widths(ops, shape, pool, regime):
    worst = _check_bwd(ops, *shape, pool, regime, "pooled_skip" if pool else "plain", seed=hash((shape, pool)) % 997)
    _report(f"bwd {'pooled' if pool else 'plain'} {regime} {_shape_id(shape)}", **worst)


@pytest.mark.parametrize("regime", [SPARSE, DENSE])
@pytest.mark.parametrize("shape", BWD_EDGES_PLAIN + BWD_EDGES_POOL, ids=_shape_id)
def test_bn_relu_bwd_grid_edges(ops, shape, regime):
    pool = shape in BWD_EDGES_POOL
    n, h, w, c = shape
    if shape[:3] in _edge_shapes("bwd", pool):
        _assert_on_edge("bwd", n, h, w, c, pool)
    worst = _check_bwd(ops, *shape, pool, regime, "pooled_skip" if pool else "plain", seed=w % 991)
    _report(f"bwd edge {'pooled' if pool else 'plain'} {regime} {_shape_id(shape)}", **worst)


@pytest.mark.parametrize("regime", [SPARSE, DENSE])
@pytest.mark.parametrize("form", ["plain_canvas", "frozen", "syncbn", "pooled_frozen", "pooled_syncbn"])
def test_bn_relu_bwd_forms(ops, form, regime):
    pool = form.startswith("pooled")
    worst = _check_bwd(ops, 2, 16, 32, 128, pool, regime, form.replace("pooled_", ""), seed=len(form) + 5 * (regime == DENSE))
    _report(f"bwd {form} {regime}", **worst)


@pytest.mark.parametrize("regime", [SPARSE, DENSE])
@pytest.mark.parametrize("pool", [False, True], ids=["plain", "pooled"])
def test_bn_relu_bwd_full_size(ops, pool, regime):
    """Config 2, level 0: 16 x 512 x 512 x 64 (443 pixels per thread plain, 444 pooled)."""
    worst = _check_bwd(ops, 16, 512, 512, 64, pool, regime, "pooled_skip" if pool else "plain", seed=41 + pool)
    _report(f"bwd full-size {'pooled' if pool else 'plain'} {regime}", **worst)
    torch.cuda.empty_cache()


def test_bn_relu_bwd_with_fused_partials_is_bit_identical(ops):
    """pre = the partial sums of ops.conv3x3_dgrad_bnred (the backward-data convolution that produces g1) on sparse integer
    operands: dgamma, dbeta and dy are bit-identical to the same call with the separate reduce pass, and exact."""
    n, h, w, c = 2, 16, 32, 64
    gc = torch.Generator().manual_seed(51)
    g = _gen(51)
    dy_up = C.operand((n, c, h, w), C.SPARSE, 9 * c, gc)
    wt = C.operand((c, c, 3, 3), C.SPARSE, 9 * c, gc, sparse_input=False)
    _, wd = ops.prep_conv3x3_weight(wt.float().cuda())
    y = _y(n, h, w, c, SPARSE, g)
    gamma, mean, rstd, scale, shift = _bn_params(c, SPARSE, g)
    g1 = torch.empty((n, h, w, c), dtype=BF16, device="cuda")
    pre = ops.conv3x3_dgrad_bnred(C.nhwc(dy_up).contiguous().to(device="cuda", dtype=BF16), wd, g1, y, scale, shift, mean, rstd)
    assert pre is not None, "no fused form at 2 x 16 x 32, 64 -> 64"
    E.assert_equal(g1, C.nhwc(C.conv3x3_dgrad(dy_up, wt)).cuda(), "g1 (dgrad)")
    out = []
    for p in (pre, None):
        yy = y.clone()
        dgamma, dbeta = torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
        ops.bn_relu_bwd(g1, None, None, yy, gamma, scale, shift, mean, rstd, yy, dgamma, dbeta, pre=p)
        out.append((yy, dgamma, dbeta))
    for (a, b), what in zip(zip(out[0], out[1]), ("dy", "dgamma", "dbeta")):
        assert torch.equal(a.view(torch.int16) if a.dtype == BF16 else a.view(torch.int32),
                           b.view(torch.int16) if b.dtype == BF16 else b.view(torch.int32)), f"{what}: pre changes the bits"
    sums = E.bwd_sums(E.bwd_da(y, g1, None, None, scale, shift), y)
    rg, rb = E.param_grads(sums, mean, rstd)
    E.assert_equal(out[0][1], rg, "dgamma")
    E.assert_equal(out[0][2], rb, "dbeta")


# ------------------------------------------------------------------------------------------------ channel-slice copy / add
COPY_SHAPES = [(2, 6, 10, 64), (1, 1, 3, 128), (16, 32, 32, 1024)] + [s + (64,) for s in _edge_shapes("ew", False)]


@pytest.mark.parametrize("shape", COPY_SHAPES, ids=_shape_id)
def test_nhwc_copy_and_add_exact(ops, shape):
    """The multitask and gate forms: the skip half of one concat buffer copied into a second one; an in-place add into the
    skip half of a concat gradient (2C pitch); an add of two contiguous tensors into the first."""
    n, h, w, c = shape
    g = _gen(61 + w)
    src_cv, src = E.canvas2(n, h, w, c)
    bits = torch.randint(-32768, 32768, (n, h, w, c), generator=g, device="cuda", dtype=torch.int32).to(torch.int16)
    bits[bits == E.BF16_SENTINEL] = 0
    src.view(torch.int16).copy_(bits)
    dst_cv, dst = E.canvas2(n, h, w, c)
    ops.nhwc_copy(src, dst)
    assert torch.equal(dst.view(torch.int16), bits), "nhwc_copy: not a bit copy"
    assert bool((dst_cv[..., c:].view(torch.int16) == E.BF16_SENTINEL).all()), "nhwc_copy: wrote the other half"

    def values(shape_):  # magnitudes over 16 binades: the fp32 sum is rounded to bf16, often at a tie
        v = torch.randn(shape_, generator=g, device="cuda") * torch.exp2(torch.randint(-8, 8, shape_, generator=g, device="cuda"))
        return v.to(BF16)

    acv, a = E.canvas2(n, h, w, c)
    a.copy_(values((n, h, w, c)))
    b = values((n, h, w, c))
    want = E.to_bf16((a.to(F64) + b.to(F64)).to(F32).to(F64))
    ops.nhwc_add(a, b)
    E.assert_equal(a, want, "nhwc_add (in place, 2C pitch)")
    assert bool((acv[..., c:].view(torch.int16) == E.BF16_SENTINEL).all()), "nhwc_add: wrote the other half"
    xbuf, x = E.guarded((n, h, w, c), BF16)
    x.copy_(values((n, h, w, c)))
    want = E.to_bf16((x.to(F64) + b.to(F64)).to(F32).to(F64))
    ops.nhwc_add(x, b)
    E.assert_equal(x, want, "nhwc_add (contiguous)")
    assert int((xbuf.view(torch.int16)[x.numel():] != E.BF16_SENTINEL).sum()) == 0, "nhwc_add: written past the end"


# ------------------------------------------------------------------------------------------------ argument validation
def test_pool_arguments_are_validated_before_any_launch(ops):
    """pooled, pool_idx and g_pool are addressed at pixel pitch C by the kernels: a channel slice, a wrong shape or dtype,
    or a pooled gradient without positions is an error raised before anything is launched."""
    from unet_torch_b200 import _lib

    n, h, w, c = 2, 4, 6, 64
    y = torch.zeros((n, h, w, c), dtype=BF16, device="cuda")
    a = torch.empty_like(y)
    v = torch.ones(c, device="cuda")
    pooled = torch.empty((n, h // 2, w // 2, c), dtype=BF16, device="cuda")
    idx = torch.empty((n, h // 2, w // 2, c), dtype=torch.uint8, device="cuda")
    wide = torch.empty((n, h // 2, w // 2, 2 * c), dtype=BF16, device="cuda")
    wide_idx = torch.empty((n, h // 2, w // 2, 2 * c), dtype=torch.uint8, device="cuda")
    bad_pooled = [wide[..., :c], pooled[:, :1], pooled.float(), pooled.view(torch.int16)]
    bad_idx = [wide_idx[..., :c], idx[:, :, :1], idx.to(torch.int16)]
    calls = []
    for p in bad_pooled:
        calls.append(lambda p=p: ops.bn_relu_fwd(y, v, v, a, p, idx))
    for i in bad_idx:
        calls.append(lambda i=i: ops.bn_relu_fwd(y, v, v, a, pooled, i))
        calls.append(lambda i=i: ops.maxpool2x2(y, pooled, i))
        calls.append(lambda i=i: ops.bn_relu_bwd(y, pooled, i, y, v, v, v, v, v, y, v.clone(), v.clone()))
    for p in bad_pooled:
        calls.append(lambda p=p: ops.bn_relu_bwd(y, p, idx, y, v, v, v, v, v, y, v.clone(), v.clone()))
    calls += [lambda: ops.bn_relu_fwd(y, v, v, a, None, idx),                        # positions without a pooled output
              lambda: ops.bn_relu_fwd(y, v, v, a[:, :2], pooled, idx),               # a of another shape
              lambda: ops.bn_relu_bwd(y, pooled, None, y, v, v, v, v, v, y, v.clone(), v.clone()),
              lambda: ops.bn_relu_bwd(None, None, None, y, v, v, v, v, v, y, v.clone(), v.clone())]
    torch.cuda.synchronize()
    launches = _lib.query("b200unet_launch_count")
    for i, call in enumerate(calls):
        with pytest.raises(ValueError):
            call()
        assert _lib.query("b200unet_launch_count") == launches, f"call {i} launched a kernel before failing"
    ops.bn_relu_fwd(y, v, v, a, pooled, idx)   # the well-formed call still runs
    ops.maxpool2x2(y, pooled, idx)
    torch.cuda.synchronize()
    assert _lib.query("b200unet_launch_count") > launches
