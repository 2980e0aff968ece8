"""-m gpu: bandwidth kernels (BN statistics / pool / loss / head / first conv) against the oracle on the same inputs. The
BatchNorm+ReLU forward and backward kernels are checked exactly in tests/test_gpu_bn_relu_exact.py."""
import pytest
import torch

from oracle import unet_oracle as O
from gpu_util import BF16, bf16_round, from_nhwc, max_abs, rel_l2, to_nhwc_bf16

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200
    from unet_torch_b200 import ops as _ops

    return _ops


def _bn_setup(c, n, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    y = bf16_round(torch.randn(n, c, h, w, generator=g) * 1.7 + 0.3)
    gamma = torch.rand(c, generator=g) + 0.5
    beta = torch.randn(c, generator=g) * 0.2
    return y, gamma, beta


@pytest.mark.parametrize("c,n,h,w", [(64, 2, 16, 32), (128, 1, 8, 16), (256, 3, 4, 6)])
def test_bn_stats_finalize_and_apply(ops, c, n, h, w):
    y, gamma, beta = _bn_setup(c, n, h, w, 1)
    yd = to_nhwc_bf16(y)
    # statistics through the generic partial-reduction path: one "tile" row per pixel row of the image
    rows = n * h
    part = torch.empty(rows, 2, c, device="cuda")
    yr = yd.float().view(rows, w, c)
    part[:, 0] = yr.sum(1)
    part[:, 1] = (yr * yr).sum(1)
    sums = torch.empty(2 * c, dtype=torch.float64, device="cuda")
    ops.bn_reduce_partials(part.view(-1), rows, c, sums)
    rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    mean, rstd, scale, shift = (torch.empty(c, device="cuda") for _ in range(4))
    ops.bn_finalize(sums, n * h * w, gamma.cuda(), beta.cuda(), 1e-5, 0.1, rm, rv, mean, rstd, scale, shift)
    want, nrm, nrv = O.batchnorm_train(y, gamma, beta, torch.zeros(c), torch.ones(c))
    assert rel_l2(mean, y.mean((0, 2, 3))) < 1e-5
    assert rel_l2(rm, nrm) < 1e-5 and rel_l2(rv, nrv) < 1e-5
    a = torch.empty_like(yd)
    ops.bn_relu_fwd(yd, scale, shift, a)
    assert rel_l2(from_nhwc(a), O.relu(want)) < 4e-3  # bf16 output rounding


def test_channel_sum(ops):
    x = bf16_round(torch.randn(2, 128, 8, 16))
    wide = torch.zeros(2, 8, 16, 256, dtype=BF16, device="cuda")
    wide[..., 128:] = to_nhwc_bf16(x)
    out = torch.empty(128, device="cuda")
    ops.channel_sum(wide[..., 128:], out)
    assert rel_l2(out, x.sum((0, 2, 3))) < 1e-5


@pytest.mark.parametrize("cin", [1, 3])
def test_first_conv_forward_and_wgrad(ops, cin):
    g = torch.Generator().manual_seed(4)
    n, h, w, cout = 2, 16, 24, 64
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, 3, 3, generator=g) * 0.3
    y = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    rows = ops.first_conv_stat_rows(n, h, w)
    st = torch.empty(rows * 2 * cout, device="cuda")
    ops.conv3x3_first(x.cuda(), wt.cuda(), y, st)
    want = O.conv3x3(x, wt)
    assert rel_l2(from_nhwc(y), want) < 4e-3
    s = st.view(rows, 2, cout).sum(0).cpu()
    yb = from_nhwc(y)
    assert rel_l2(s[0], yb.sum((0, 2, 3))) < 1e-4 and rel_l2(s[1], (yb * yb).sum((0, 2, 3))) < 1e-4
    # weight gradient
    dy = bf16_round(torch.randn(n, cout, h, w, generator=g))
    xv = x.clone()
    wv = wt.clone().requires_grad_(True)
    (O.conv3x3(xv, wv) * dy).sum().backward()
    dw = torch.empty(cout, cin, 3, 3, device="cuda")
    ops.conv3x3_first_wgrad(x.cuda(), to_nhwc_bf16(dy), dw)
    assert rel_l2(dw, wv.grad) < 1e-4


@pytest.mark.parametrize("ncls", [2, 5])
def test_head_forward_backward(ops, ncls):
    g = torch.Generator().manual_seed(5)
    n, h, w, cin = 2, 8, 24, 64
    a = bf16_round(torch.randn(n, cin, h, w, generator=g))
    wt = torch.randn(ncls, cin, 1, 1, generator=g) * 0.2
    b = torch.randn(ncls, generator=g)
    ad = to_nhwc_bf16(a)
    z = torch.empty(n, ncls, h, w, device="cuda")
    ops.head_fprop(ad, wt.cuda(), b.cuda(), z)
    av, wv, bv = a.clone().requires_grad_(True), wt.clone().requires_grad_(True), b.clone().requires_grad_(True)
    want = O.conv1x1(av, wv, bv)
    assert rel_l2(z, want) < 1e-5
    dz = torch.randn(n, ncls, h, w, generator=g)
    (want * dz).sum().backward()
    da = torch.empty_like(ad)
    dw, db = torch.empty(ncls, cin, 1, 1, device="cuda"), torch.empty(ncls, device="cuda")
    ops.head_bwd(dz.cuda(), ad, wt.cuda(), da, dw, db)
    assert rel_l2(from_nhwc(da), av.grad) < 4e-3
    assert rel_l2(dw, wv.grad) < 1e-5 and rel_l2(db, bv.grad) < 1e-5


@pytest.mark.parametrize("ncls", [2, 5])
@pytest.mark.parametrize("lt", ["dice_bce_mc", "CE"])
def test_loss_matches_reference_golden(golden, ncls, lt):
    import unet_torch_b200 as U

    g = golden("ref_ops.pt")[f"loss_{lt}_{ncls}"]
    z = g["z"].cuda().requires_grad_(True)
    U.loss.CLASS_NUMBER = ncls
    l = U.calc_loss(z, g["t"].cuda(), loss_type=lt)
    l.backward()
    assert abs(float(l) - float(g["loss"])) < 1e-4 * abs(float(g["loss"]))  # fp32 check tolerance 1e-4
    assert rel_l2(z.grad, g["grad"]) < 1e-4


def test_mse_losses_match_reference_golden(golden):
    import unet_torch_b200 as U

    ops_g = golden("ref_ops.pt")
    g = ops_g["loss_relu_mseMC"]
    o = g["o"].cuda().requires_grad_(True)
    l = U.calc_loss(torch.relu(o), g["t"].cuda(), loss_type="mseMC")
    l.backward()
    assert abs(float(l) - float(g["loss"])) < 1e-5 * abs(float(g["loss"])) and rel_l2(o.grad, g["grad"]) < 1e-5
    o2 = g["o"].cuda().requires_grad_(True)
    l2 = U.relu_mse_loss(o2, g["t"].cuda())
    l2.backward()
    assert abs(float(l2) - float(g["loss"])) < 1e-5 * abs(float(g["loss"])) and rel_l2(o2.grad, g["grad"]) < 1e-5
    g = ops_g["loss_mse"]
    o = g["o"].cuda().requires_grad_(True)
    l = U.calc_loss(o, g["t"].cuda(), loss_type="mse")
    l.backward()
    assert abs(float(l) - float(g["loss"])) < 1e-5 * abs(float(g["loss"])) and rel_l2(o.grad, g["grad"]) < 1e-5


def test_softmax_argmax_bit_exact(golden):
    import unet_torch_b200 as U

    ops_g = golden("ref_ops.pt")
    for key in ("argmax_small_logits", "argmax_ties"):
        got = U.predict_mask(ops_g[key]["z"].cuda())
        assert torch.equal(got.cpu(), ops_g[key]["mask"])
    # larger random case against the oracle restatement
    z = torch.randn(2, 5, 64, 64, generator=torch.Generator().manual_seed(9)) * 0.01
    assert torch.equal(U.predict_mask(z.cuda()).cpu(), O.softmax_argmax(z))


def test_maxpool_alone_matches_reference_semantics(ops, golden):
    """b200unet_maxpool2x2_fwd (inference path): values and window positions against torch's max_pool2d goldens (ties ->
    first, NaN wins, -0.0/+0.0 tie) and against the oracle on a random channel-slice input."""
    g = golden("ref_ops.pt")["pool"]
    x = g["x"]                                      # [2,3,6,8] fp32 with ties / NaN / signed zeros
    n, c, h, w = x.shape
    xp = torch.zeros(n, 8, h, w)
    xp[:, :c] = x
    a = to_nhwc_bf16(bf16_round(xp))
    pooled = torch.empty(n, h // 2, w // 2, 8, dtype=BF16, device="cuda")
    idx = torch.empty(n, h // 2, w // 2, 8, dtype=torch.uint8, device="cuda")
    ops.maxpool2x2(a, pooled, idx)
    want_v, want_i = torch.nn.functional.max_pool2d(bf16_round(xp), 2, return_indices=True)
    got_v = from_nhwc(pooled)
    assert bool(((got_v == want_v) | (got_v.isnan() & want_v.isnan())).all())
    k = idx.permute(0, 3, 1, 2).cpu().long()
    hp = torch.arange(h // 2).view(1, 1, -1, 1)
    wp = torch.arange(w // 2).view(1, 1, 1, -1)
    flat = (2 * hp + k // 2) * w + (2 * wp + k % 2)  # window position -> torch's flat index h * W_in + w
    assert torch.equal(flat, want_i)
    gen = torch.Generator().manual_seed(3)
    big = bf16_round(torch.randn(2, 128, 16, 24, generator=gen))
    canvas = to_nhwc_bf16(big)
    out = torch.empty(2, 8, 12, 64, dtype=BF16, device="cuda")
    ops.maxpool2x2(canvas[..., 64:], out)            # strided channel slice in, contiguous out
    wv, _, _ = O.maxpool2x2(big[:, 64:])
    assert torch.equal(from_nhwc(out), wv)
