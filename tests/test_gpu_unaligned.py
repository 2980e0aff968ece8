"""-m gpu: UNet and UNet_multitask on the tensor-core engine at H and W that are not multiples of 16
(`allow_unaligned_sizes()`): floor-mode pooling (Model.py:36,42) and the zero pad strip F.pad leaves in the concat buffer
(Model.py:69-73), operator by operator and through whole networks against the oracle.

Operators: the floor-mode BatchNorm+ReLU(+pool) forward, max-pool and BatchNorm backward exactly or within the bounds of
tests/ew_check.py at (odd, even), (even, odd) and (odd, odd) maps; the ConvTranspose2d into an odd canvas and the strip fill;
the ConvTranspose2d bias gradient with a large gradient planted in the strip, without and with dropout.
Networks: one training step against the fp32 oracle with the bf16-storage emulation as yardstick (the assertions of
test_gpu_configs.py::test_training_step_at_config_yml_size_against_oracle), dropout with the engine's masks, the two-decoder
network, CUDA-graph replay, and eval (fused heads, logits, predict_tiled)."""
import statistics

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import ew_check as E
from gpu_util import cos, from_nhwc, host_step, rel_l2, to_nhwc_bf16
from oracle import cpu_baseline
from oracle import philox as PX
from oracle import unet_oracle as O
from test_gpu_dropout import _engine_step, _errors, _judge

pytestmark = pytest.mark.gpu

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
MAPS = [(2, 7, 10), (2, 6, 11), (1, 9, 13)]   # (odd, even), (even, odd), (odd, odd)


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200  # noqa: F401
    from unet_torch_b200 import ops as _ops

    return _ops


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _region(t, h, w):
    """The leading 2*(h//2) x 2*(w//2) pixels of an NHWC tensor: what the 2x2 windows cover."""
    return t[:, : 2 * (h // 2), : 2 * (w // 2)]


def _strip_mask(n, h, w):
    m = torch.ones((n, h, w), dtype=torch.bool, device="cuda")
    m[:, : 2 * (h // 2), : 2 * (w // 2)] = False
    return m


# ------------------------------------------------------------------------------------------------ operators
@pytest.mark.parametrize("c", [64, 1024])
@pytest.mark.parametrize("shape", MAPS, ids=lambda s: "x".join(map(str, s)))
def test_floor_bn_relu_pool_forward_exact(ops, shape, c):
    """a (strip pixels included) into the left half of a concat buffer, pooled values and positions: bit-exact; nothing
    outside the slice and the pooled tensors is written."""
    n, h, w = shape
    g = _gen(h * 31 + w + c)
    y = (torch.randn((n, h, w, c), generator=g, device="cuda") * 2 + 0.3).to(BF16)
    r = _region(y, h, w)   # ties between the two rows of a share of the windows
    r[:, 1::2] = torch.where(torch.rand(r[:, 1::2].shape, generator=g, device="cuda") < 0.2, r[:, 0::2], r[:, 1::2])
    scale = torch.rand(c, generator=g, device="cuda") + 0.5
    shift = torch.randn(c, generator=g, device="cuda") * 0.3
    E.plant_midpoints(scale, shift, y, torch.Generator().manual_seed(c + h), channels=8)
    cv, a = E.canvas2(n, h, w, c)
    pbuf, pooled = E.guarded((n, h // 2, w // 2, c), BF16)
    ibuf, idx = E.guarded((n, h // 2, w // 2, c), torch.uint8)
    ops.bn_relu_fwd(y, scale, shift, a, pooled, idx)
    want, _, _ = E.bn_relu_fwd(y, scale, shift)
    E.assert_equal(a, want, "a")
    pv, pi = E.maxpool2x2(_region(a, h, w))
    E.assert_equal(pooled, pv, "pooled")
    E.assert_equal(idx, pi, "pool_idx")
    E.assert_right_half(cv, "a")   # every pixel of the slice written (the strip too), the other half untouched
    E.assert_guard(pbuf, pooled.numel(), "pooled")
    E.assert_guard(ibuf, idx.numel(), "pool_idx")
    # the standalone max-pool of the inference path on the same slice
    pbuf2, pooled2 = E.guarded((n, h // 2, w // 2, c), BF16)
    ibuf2, idx2 = E.guarded((n, h // 2, w // 2, c), torch.uint8)
    ops.maxpool2x2(a, pooled2, idx2)
    E.assert_equal(pooled2, pv, "maxpool2x2")
    E.assert_equal(idx2, pi, "maxpool2x2 positions")
    E.assert_guard(pbuf2, pooled2.numel(), "maxpool2x2")
    E.assert_guard(ibuf2, idx2.numel(), "maxpool2x2 positions")


def _floor_da(y, g1, g_pool, idx, scale, shift):
    """da of the floor-mode pooled backward: the unpooled gradient inside the windows, g1 alone on the strip."""
    n, h, w, _ = y.shape
    da = E.bwd_da(y, g1, None, None, scale, shift)
    r = (slice(None), slice(0, 2 * (h // 2)), slice(0, 2 * (w // 2)))
    da[r] = E.bwd_da(y[r], g1[r], g_pool, idx, scale, shift)
    return da


@pytest.mark.parametrize("regime", ["sparse", "dense"])
@pytest.mark.parametrize("c", [64, 1024])
@pytest.mark.parametrize("shape", MAPS, ids=lambda s: "x".join(map(str, s)))
def test_floor_bn_relu_pool_backward(ops, shape, c, regime):
    """Reduce + apply with the skip half of a concat gradient as g1 and a pooled gradient: dgamma / dbeta exact (sparse:
    every partial sum is an integer below 2^24) or within ew_check.sum_bounds (dense); dy within ew_check.dy_bound on every
    pixel, strip included; dy written over y."""
    n, h, w = shape
    g = _gen(h * 7 + w * 3 + c + (regime == "dense"))

    def ints(shp, m, density):
        v = torch.randint(-m, m + 1, shp, generator=g, device="cuda")
        return (v * (torch.rand(shp, generator=g, device="cuda") < density)).to(BF16)

    if regime == "sparse":
        y = ints((n, h, w, c), 3, 0.3)
        gamma = torch.exp2(torch.randint(-1, 2, (c,), generator=g, device="cuda").float())
        mean = torch.randint(-1, 2, (c,), generator=g, device="cuda").float()
        rstd = torch.exp2(torch.randint(-1, 2, (c,), generator=g, device="cuda").float())
    else:
        y = (torch.randn((n, h, w, c), generator=g, device="cuda") * 2 + 1).to(BF16)
        gamma = torch.rand(c, generator=g, device="cuda") + 0.5
        yd = y.reshape(-1, c).to(F64)
        mean, rstd = yd.mean(0).float(), (yd.var(0, unbiased=False) + 1e-5).rsqrt().float()
    beta = torch.randn(c, generator=g, device="cuda") * 0.3
    scale = (gamma.double() * rstd.double()).float()
    shift = beta - mean * scale
    cva, a = E.canvas2(n, h, w, c)
    pooled = torch.empty((n, h // 2, w // 2, c), dtype=BF16, device="cuda")
    idx = torch.empty((n, h // 2, w // 2, c), dtype=torch.uint8, device="cuda")
    ops.bn_relu_fwd(y, scale, shift, a, pooled, idx)
    grad = (lambda s: ints(s, 4, 0.3)) if regime == "sparse" else (lambda s: torch.randn(s, generator=g, device="cuda").to(BF16))
    g_pool = grad(pooled.shape)
    cvg, g1 = E.canvas2(n, h, w, c)
    g1.copy_(grad((n, h, w, c)))
    y_in = y.clone()
    dgb, dgamma = E.guarded((c,), F32)
    dbb, dbeta = E.guarded((c,), F32)
    count = n * h * w
    ops.bn_relu_bwd(g1, g_pool, idx, y, gamma, scale, shift, mean, rstd, y, dgamma, dbeta, count=count)
    dy = y
    da = _floor_da(y_in, g1, g_pool, idx, scale, shift)
    sums = E.bwd_sums(da, y_in)
    strip_px = n * h * w - n * (h // 2) * (w // 2) * 4
    k = E.terms_per_thread(n, h, w, c, True) + E.terms_per_thread(1, 1, strip_px, c, False)
    bg, bb = E.sum_bounds(sums, mean, rstd, k)
    rg, rb = E.param_grads(sums, mean, rstd)
    if regime == "sparse":
        E.assert_equal(dgamma, rg, "dgamma")
        E.assert_equal(dbeta, rb, "dbeta")
    else:
        E.assert_within(dgamma, rg, bg, "dgamma")
        E.assert_within(dbeta, rb, bb, "dbeta")
    E.assert_guard(dgb, c, "dgamma")
    E.assert_guard(dbb, c, "dbeta")
    ref, mag = E.dy_ref(da, y_in, gamma, mean, rstd, torch.stack([rb, rg]), count)
    dense = regime == "dense"
    bound = E.dy_bound(ref, mag, y_in, gamma, mean, rstd, count, bg if dense else None, bb if dense else None)
    E.assert_within(dy, ref, bound, "dy")
    assert bool(_strip_mask(n, h, w).any()) and bool((da[_strip_mask(n, h, w)] != 0).any()), "the strip carried no gradient"
    assert bool((cvg[..., c:].view(torch.int16) == E.BF16_SENTINEL).all()), "g1 canvas: the other half was written"


_REDUCE_AT_THE_GRID_CAP = r"""
import ctypes, os, sys
sys.path.insert(0, os.getcwd())
import torch
from unet_torch_b200 import _lib
n, h, w, c = 16, 125, 125, 256          # level 2 of 16 x 3 x 500^2
g = torch.Generator(device="cuda").manual_seed(5)
bf = torch.bfloat16
y = torch.randn((n, h, w, c), generator=g, device="cuda").to(bf)
g1 = torch.randn((n, h, w, c), generator=g, device="cuda").to(bf)
gp = torch.randn((n, h // 2, w // 2, c), generator=g, device="cuda").to(bf)
idx = torch.randint(0, 4, (n, h // 2, w // 2, c), generator=g, device="cuda").to(torch.uint8)
one, zero = torch.ones(c, device="cuda"), torch.zeros(c, device="cuda")
ws = _lib.query("b200unet_bn_bwd_workspace_floats", n, h, w, c)
guard = 148 * 8 * 2 * c
buf = torch.full((ws + guard,), float("nan"), device="cuda")
rows = ctypes.c_int(0)
_lib.call("b200unet_bn_relu_bwd_reduce_rows_floor", g1.data_ptr(), c, gp.data_ptr(), idx.data_ptr(), y.data_ptr(), c,
          one.data_ptr(), zero.data_ptr(), zero.data_ptr(), one.data_ptr(), buf.data_ptr(), ctypes.byref(rows), n, h, w, c,
          torch.cuda.current_stream().cuda_stream)
torch.cuda.synchronize()
assert rows.value > 148 * 8, rows.value               # the pooled launch alone fills 148 x 8 rows at this knob value
assert rows.value * 2 * c <= ws, (rows.value, ws)
assert bool(torch.isnan(buf[ws:]).all()), "the reduce wrote past the workspace"
got = buf[: rows.value * 2 * c].view(rows.value, 2, c).double().sum(0)
da = g1.double()
r = da[:, : 2 * (h // 2), : 2 * (w // 2)]
for k in range(4):
    r[:, k >> 1::2, k & 1::2] += torch.where(idx == k, gp.double(), 0.0)
da = torch.where(y.double() > 0, da.float().double(), 0.0)
want = torch.stack([da.sum((0, 1, 2)), (da * y.double()).sum((0, 1, 2))])
err = float(((got - want).norm() / want.norm()))
assert err < 1e-5, err
print("REDUCE_OK", rows.value, err)
"""


def test_floor_reduce_fits_its_workspace_at_the_largest_grid():
    """With B200UNET_BWD_BLOCKS_PER_SM=8 (the largest grid the knob allows) the pooled reduce of a 16 x 125 x 125 x 256 map
    already fills 148 x 8 partial rows and the pad strip's launch appends ~500 more: they must stay inside the workspace
    b200unet_bn_bwd_workspace_floats sizes (a NaN guard follows it) and reduce to the fp64 sums. The knob is read once per
    process, hence the subprocess."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, B200UNET_BWD_BLOCKS_PER_SM="8")
    r = subprocess.run([sys.executable, "-c", _REDUCE_AT_THE_GRID_CAP], cwd=root, env=env, capture_output=True, text=True,
                       timeout=300)
    print(r.stdout[-500:])
    assert r.returncode == 0 and "REDUCE_OK" in r.stdout, r.stderr[-3000:]


@pytest.mark.parametrize("n,h,w,cin,cup", [(2, 5, 8, 128, 64), (1, 7, 6, 256, 128), (1, 3, 5, 1024, 512)])
@pytest.mark.parametrize("odd", [(1, 0), (0, 1), (1, 1)], ids=["odd_h", "odd_w", "odd_hw"])
def test_conv_transpose_into_an_odd_canvas(ops, n, h, w, cin, cup, odd):
    """ConvTranspose2d of an h x w map into the upsampled half of a (2h + dh) x (2w + dw) concat buffer filled with a
    sentinel: the 2h x 2w region against the bf16 operands at the one-operator tolerance, the pad strip all zero bits after
    pad_strip_zero, the skip half untouched; backward-data and weight gradient read the region only."""
    hh, ww = 2 * h + odd[0], 2 * w + odd[1]
    g = torch.Generator().manual_seed(hh * ww + cin)
    xv = torch.randn(n, cin, h, w, generator=g).to(BF16).float()
    wv = (torch.randn(cin, cup, 2, 2, generator=g) * (1.0 / cin) ** 0.5).to(BF16).float()
    b = torch.randn(cup, generator=g)
    want = F.conv_transpose2d(xv.double(), wv.double(), b.double(), stride=2).float()
    wf, wd = ops.prep_convt2x2_weight(wv.cuda())
    cv = E.sentinel_like(n * hh * ww * 2 * cup, BF16).view(n, hh, ww, 2 * cup)
    ops.convt2x2(to_nhwc_bf16(xv), wf, b.cuda(), cv[..., cup:])
    ops.pad_strip_zero(cv[..., cup:])
    assert rel_l2(from_nhwc(cv[:, : 2 * h, : 2 * w, cup:]), want) < 1e-2
    strip = _strip_mask(n, hh, ww)
    assert bool((cv[..., cup:].view(torch.int16)[strip] == 0).all()), "pad strip not all zero bits"
    assert bool((cv[..., :cup].view(torch.int16) == E.BF16_SENTINEL).all()), "skip half written"
    # backward: a NaN gradient on the strip must not reach dx or dw
    du = torch.randn(n, cup, 2 * h, 2 * w, generator=g).to(BF16).float()
    dcat = torch.full((n, hh, ww, 2 * cup), float("nan"), dtype=BF16, device="cuda")
    dcat[:, : 2 * h, : 2 * w, cup:] = to_nhwc_bf16(du)
    dx = torch.empty(n, h, w, cin, dtype=BF16, device="cuda")
    ops.convt2x2_dgrad(dcat[..., cup:], wd, dx)
    xr = xv.double().requires_grad_(True)
    wr = wv.double().requires_grad_(True)
    (F.conv_transpose2d(xr, wr, None, stride=2) * du.double()).sum().backward()
    assert rel_l2(from_nhwc(dx), xr.grad.float()) < 1e-2
    dw = torch.empty(cin, cup, 2, 2, device="cuda")
    ops.convt2x2_wgrad(to_nhwc_bf16(xv), dcat[..., cup:], dw)
    assert rel_l2(dw, wr.grad.float()) < 1e-4


@pytest.mark.parametrize("dropout", [False, True])
@pytest.mark.parametrize("hw", [(33, 50), (32, 47), (17, 17)])
def test_convt_bias_gradient_excludes_the_pad_strip(ops, hw, dropout):
    """The engine's ConvTranspose2d bias gradient at an odd level: the sums the up.conv1 backward-data epilogue (or the
    dropout backward with sums=) takes over the whole upsampled half, minus pad_strip_sub_colsum - with a gradient 1000x
    larger on the strip than elsewhere - equals the host sum over the 2h' x 2w' region to 1e-5."""
    h, w = hw
    n, cin, c = 2, 128, 64          # up.conv1 of level 0: concat 128 channels -> 64; its dx upsampled half = 64 channels
    g = _gen(h * w + dropout)
    dy = (torch.randn((n, h, w, c), generator=g, device="cuda")).to(BF16)
    strip = _strip_mask(n, h, w)
    dy[strip] = dy[strip] * 1000   # through the 3x3 taps the strip of dx is large too
    wv = torch.randn(c, cin, 3, 3, generator=torch.Generator().manual_seed(3)) * (1.0 / (9 * cin)) ** 0.5
    _, wd = ops.prep_conv3x3_weight(wv.cuda())
    dcat = torch.empty((n, h, w, cin), dtype=BF16, device="cuda")
    db = torch.empty(cin - c, dtype=F32, device="cuda")
    if not dropout:
        rows = ops.conv3x3_stat_rows(n, h, w, c, cin)
        part = torch.empty(rows * 2 * cin, dtype=F32, device="cuda")
        ops.conv3x3(dy, wd, dcat, part)
        ops.partial_colsum(part, rows, 2 * cin, c, cin - c, db)
    else:
        ops.conv3x3(dy, wd, dcat)
        seed = torch.tensor([1234], dtype=torch.int64, device="cuda")
        ops.dropout_mul(dcat, 7, seed, 0.3, sums=(c, db))
    full = dcat[..., c:].double().sum((0, 1, 2))
    ops.pad_strip_sub_colsum(dcat[..., c:], db)
    want = _region(dcat[..., c:], h, w).double().sum((0, 1, 2))
    assert float((full - want).abs().max()) > 100 * float(want.abs().max()) * 1e-5, "the strip does not weigh in"
    assert rel_l2(db.double(), want) < 1e-5


def test_strip_kernels_at_even_sizes_launch_nothing(ops):
    from unet_torch_b200 import _lib

    x = torch.ones((2, 8, 6, 64), dtype=BF16, device="cuda")
    out = torch.zeros(64, device="cuda")
    before = _lib.query("b200unet_launch_count")
    ops.pad_strip_zero(x)
    ops.pad_strip_sub_colsum(x, out)
    assert _lib.query("b200unet_launch_count") == before
    assert bool((x == 1).all()) and bool((out == 0).all())


# ------------------------------------------------------------------------------------------------ networks
def _train_step_against_oracle(n, h, w, width=64):
    """test_gpu_configs.py::test_training_step_at_config_yml_size_against_oracle, on the tensor-core engine."""
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    torch.manual_seed(1063)
    net = U.UNet(3, 2, width).allow_unaligned_sizes()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(7)
    x = torch.randn(n, 3, h, w, generator=g)
    y = (torch.rand(n, h, w, generator=g) > 0.6).float()
    net = net.cuda().train()
    assert isinstance(net._engine_for(x.cuda()), UNetEngine)
    U.loss.CLASS_NUMBER = 2
    out = net(x.cuda())
    loss = U.calc_loss(out, y.cuda(), loss_type="dice_bce_mc")
    loss.backward()
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    sd_req = dict(sd)
    sd_req.update(params)
    want, _ = O.unet_forward(sd_req, x, training=True)
    want_loss = O.calc_loss(want, y, "dice_bce_mc", 2)
    want_loss.backward()
    el, eloss, eg, _ = host_step(sd, x, y, 2, "dice_bce_mc", emulate=True)
    e, yard = rel_l2(out.detach(), want.detach()), rel_l2(el, want.detach())
    e_loss = abs(float(loss.detach()) - float(want_loss.detach())) / abs(float(want_loss.detach()))
    print(f"{n}x{h}x{w} width {width}: logits rel {e:.3e} (emulation {yard:.3e}), loss rel {e_loss:.3e}")
    assert e <= 1.5 * yard and e_loss < 1e-2
    assert rel_l2(out.detach(), el) <= yard
    grads = dict(net.named_parameters())
    errs = {k: rel_l2(grads[k].grad, p.grad) for k, p in params.items()}
    yards = {k: rel_l2(eg[k], p.grad) for k, p in params.items()}
    vs_emu = {k: (rel_l2(grads[k].grad, eg[k]), cos(grads[k].grad, eg[k])) for k in params}
    print(f"{n}x{h}x{w}: param-grad rel error median {statistics.median(errs.values()):.3e} (emulation "
          f"{statistics.median(yards.values()):.3e}), worst {max(errs.values()):.3e}")
    assert statistics.median(errs.values()) <= 1.5 * statistics.median(yards.values())
    for k in errs:
        assert errs[k] <= 1.5 * yards[k] + 0.02, (k, errs[k], yards[k])
    assert statistics.median(v[0] for v in vs_emu.values()) <= statistics.median(yards.values())
    assert min(v[1] for v in vs_emu.values()) > 0.9
    gn = torch.sqrt(sum(grads[k].grad.double().norm() ** 2 for k in params))
    wn = torch.sqrt(sum(p.grad.double().norm() ** 2 for p in params.values()))
    assert abs(float(gn / wn) - 1) < 0.1


# 16 x 17 runs with 16 images: its bottleneck is 1 x 1, so the batch is all the bottleneck BatchNorm averages over. One image
# leaves it a single value per channel (torch refuses to train that); with two, both the engine's and the emulation's
# gradients are dominated by the 1/sigma of a two-sample variance (about 70 % median error against fp32 either way)
@pytest.mark.parametrize("n,h,w", [(2, 97, 131), (1, 401, 399), (3, 33, 50), (16, 16, 17)])
def test_training_step_against_oracle(n, h, w):
    _train_step_against_oracle(n, h, w)


def test_training_step_width_128_against_oracle():
    _train_step_against_oracle(2, 49, 35, width=128)


def test_dropout_network_against_oracle_with_the_engine_masks():
    """test_gpu_dropout.py::test_network_against_oracle_with_the_engine_masks at an odd size; the ConvTranspose2d bias
    gradients are the sums of the masked 2h' x 2w' region of the concat gradient."""
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    n, h, w = 2, 45, 38
    torch.manual_seed(21)
    net = U.UNet(3, 2, 64, dropout=True, dropout_p=0.3).allow_unaligned_sizes()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().train()
    gen = torch.Generator().manual_seed(22)
    x = torch.randn((n, 3, h, w), generator=gen)
    y = torch.randint(0, 2, (n, h, w), generator=gen).float()
    assert isinstance(net._engine_for(x.cuda()), UNetEngine)
    holders = net._engine.drop
    for m in holders:
        m.p = 0.0
    logits, grads, _, _ = _engine_step(net, x.cuda(), y)
    e_off, g_off = _errors(net, sd, x, y, logits, grads, None)
    for m in holders:
        m.p = 0.3
    logits, grads, (seed_t, ps), trace = _engine_step(net, x.cuda(), y)
    masks = PX.oracle_masks(int(seed_t.item()), n, h, w, 64, ps)
    e_on, g_on = _errors(net, sd, x, y, logits, grads, masks)
    _judge(e_on, g_on, e_off, g_off, f"dropout {(n, 3, h, w)}")
    odd_levels = 0
    for kind, kw in trace:
        if kind == "convt_bwd":
            du, db = kw["du"], kw["db"]
            hh, ww = du.shape[1], du.shape[2]
            odd_levels += bool(hh % 2 or ww % 2)
            assert rel_l2(db, _region(du, hh, ww).double().sum((0, 1, 2))) < 1e-5
    assert odd_levels >= 2


def test_multitask_against_emulation_yardstick():
    import unet_torch_b200 as U

    n, h, w = 2, 37, 52
    torch.manual_seed(8)
    net = U.UNet_multitask(3, 2)
    with pytest.raises(ValueError, match="multiples of 16"):
        net._engine_for(torch.zeros(n, 3, h, w))
    net.allow_unaligned_sizes()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    x = torch.randn(n, 3, h, w, generator=torch.Generator().manual_seed(9))
    net = net.cuda().train()
    o1, o2 = net(x.cuda())
    (o1.square().mean() + o2.sin().mean()).backward()
    p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in sd.items()}
    w1, w2 = cpu_baseline.unet_multitask_forward_torchops(p, x, training=True)
    (w1.square().mean() + w2.sin().mean()).backward()
    pe = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in sd.items()}
    e1, e2 = cpu_baseline.unet_multitask_forward_torchops(pe, x, training=True, emulate_bf16=True)
    (e1.square().mean() + e2.sin().mean()).backward()
    for got, want, emu in ((o1, w1, e1), (o2, w2, e2)):
        err, yard = rel_l2(got.detach(), want.detach()), rel_l2(emu.detach(), want.detach())
        print(f"multitask logits rel {err:.3e} (emulation {yard:.3e})")
        assert err <= 1.5 * yard
    named = dict(net.named_parameters())
    errs = {k: rel_l2(named[k].grad, p[k].grad) for k in named}
    yards = {k: rel_l2(pe[k].grad, p[k].grad) for k in named}
    assert statistics.median(errs.values()) <= 1.5 * statistics.median(yards.values())
    for k in errs:
        assert errs[k] <= 1.5 * yards[k] + 0.02, (k, errs[k], yards[k])


@pytest.mark.parametrize("cls_name", ["UNet", "UNet_multitask"])
def test_cuda_graph_replay_is_bit_identical_to_eager(cls_name):
    """Two FusedSGD steps at an odd size (the second replays the captured graphs): the same bits as eager launches."""
    import unet_torch_b200 as U

    x = torch.randn(2, 3, 41, 30, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    t = torch.rand(2, 2, 41, 30, device="cuda", generator=torch.Generator("cuda").manual_seed(4))

    def run(graphs):
        torch.manual_seed(11)
        net = getattr(U, cls_name)(3, 2).allow_unaligned_sizes().cuda().train().enable_cuda_graphs(graphs)
        opt = U.FusedSGD(net, lr=0.01, momentum=0.9, weight_decay=1e-4)
        outs = []
        for _ in range(3):
            o = net(x)
            o = o if isinstance(o, tuple) else (o,)
            loss = sum(U.calc_loss(torch.relu(oi), t, loss_type="mseMC") for oi in o)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            outs.append((tuple(oi.detach().clone() for oi in o), float(loss)))
            opt.step()
        return net, outs

    net_e, eager = run(False)
    net_g, graph = run(True)
    assert net_g._engine._graphs, "no graph was captured"
    for (o1, l1), (o2, l2) in zip(eager, graph):
        assert l1 == l2 and all(torch.equal(a, b) for a, b in zip(o1, o2))
    for (k, a), (_, b) in zip(net_e.state_dict().items(), net_g.state_dict().items()):
        assert torch.equal(a, b), k


def _trained_buffers(net):
    g = torch.Generator().manual_seed(99)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


def test_eval_heads_logits_and_predict_tiled():
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    torch.manual_seed(5)
    net = U.UNet(3, 5)
    with torch.no_grad():
        _trained_buffers(net)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().eval()
    x = torch.randn(2, 3, 75, 102, generator=torch.Generator().manual_seed(6))
    xc = x.cuda()
    with pytest.raises(ValueError, match="allow_unaligned_sizes"):
        net.predict(xc)
    net.allow_unaligned_sizes()
    assert isinstance(net._engine_for(xc), UNetEngine)
    with torch.no_grad():
        logits = net(xc)
        mask = net.predict(xc)
        binary = net.predict_binary(xc)
        dens, counts = net.predict_density(xc)
    assert torch.equal(mask.long(), U.predict_mask(logits))
    assert torch.equal(binary, (torch.sigmoid(logits)[:, 0] >= 0.5).to(torch.uint8))
    assert np.array_equal(dens.cpu().numpy(), torch.relu(logits).cpu().numpy() / 200)
    assert torch.allclose(counts, dens.double().sum(dim=(2, 3)), rtol=1e-12)
    # eval logits against the fp32 oracle, with the bf16-storage emulation as yardstick
    want, _ = O.unet_forward(sd, x, training=False)
    p = {k: v.clone() for k, v in sd.items()}
    emu = cpu_baseline.unet_forward_torchops(p, x, training=False, emulate_bf16=True)
    err, yard = rel_l2(logits.cpu(), want), rel_l2(emu, want)
    print(f"eval logits rel {err:.3e} (emulation {yard:.3e})")
    assert err <= 1.5 * yard
    # predict_tiled with a crop size that is not a multiple of 16, against the crop-by-crop loop
    one = U.UNet(3, 1).cuda().eval()
    img = torch.randint(0, 256, (250, 330, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    with pytest.raises(ValueError, match="multiple of 16"):
        U.predict_tiled(one, img.numpy(), 200)
    one.allow_unaligned_sizes()
    got = U.predict_tiled(one, img.numpy(), 200, head="sigmoid", max_batch=3)
    assert got.shape == (400, 400)
    xt = O.preprocess_crop(img.numpy(), 200)
    with torch.no_grad():
        want_t = O.tiled_masks(lambda t: one(t.cuda()).cpu(), xt, 200, O.sigmoid_mask)
    agree = float((got.cpu() == want_t).float().mean())
    print(f"predict_tiled(200) vs crop-by-crop loop: agreement {agree:.6f}")
    assert agree > 0.9999
