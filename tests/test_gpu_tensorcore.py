"""-m gpu: tcgen05 implicit-GEMM kernels (conv3x3 fprop / dgrad / wgrad, ConvTranspose2d fprop / dgrad / wgrad)
against the oracle on identical bf16-rounded inputs. Tolerance: 1e-2 relative (north_star, bf16); observed error
is the bf16 rounding of the output (~2e-3)."""
import pytest
import torch

from oracle import unet_oracle as O
from gpu_util import BF16, bf16_round, from_nhwc, rel_l2, to_nhwc_bf16

pytestmark = pytest.mark.gpu
TOL = 1e-2


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200
    from unet_torch_b200 import ops as _ops

    return _ops


CONV_SHAPES = [
    # n, h, w, cin, cout
    (1, 8, 16, 64, 64),       # exactly one tile
    (2, 16, 32, 64, 64),
    (1, 24, 40, 128, 128),    # ragged tiles (h, w not multiples of 8 / 16)
    (2, 8, 16, 256, 256),
    (1, 16, 16, 128, 64),     # decoder-style Cin > Cout
    (1, 4, 4, 64, 128),       # image smaller than a tile
    # persistent resident-weight kernel (Cin <= 128): several 16x8 tiles per CTA, every (BN, K-block) variant
    (4, 64, 96, 64, 64),      # 192 tiles > 148 CTAs
    (2, 40, 72, 64, 128),     # BN = 128, ragged rows
    (3, 64, 64, 128, 64),     # two K blocks per tile
    (2, 48, 64, 128, 256),    # four channel slices share each pixel tile
    # deep-layer shapes (streaming CTA-pair kernel; B200UNET_PAIR=0 selects igemm): odd tile count, BN = 256 and 128
    (3, 16, 24, 256, 256),
    (1, 32, 40, 512, 128),
    (2, 16, 16, 256, 512),
    (1, 16, 8, 256, 256),     # a single tile: the second CTA of the pair works on an out-of-range tile
    (1, 16, 8, 128, 128),
]


@pytest.mark.parametrize("n,h,w,cin,cout", CONV_SHAPES)
def test_conv3x3_fprop_and_stats(ops, n, h, w, cin, cout):
    g = torch.Generator().manual_seed(11)
    x = bf16_round(torch.randn(n, cin, h, w, generator=g))
    wt = bf16_round(torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    wf, wd = ops.prep_conv3x3_weight(wt.cuda())
    assert torch.equal(wf.float().cpu(), wt.permute(0, 2, 3, 1).contiguous())
    y = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    rows = ops.conv3x3_stat_rows(n, h, w, cin, cout)
    st = torch.zeros(rows * 2 * cout, device="cuda")
    ops.conv3x3(to_nhwc_bf16(x), wf, y, st)
    torch.cuda.synchronize()
    want = O.conv3x3(x, wt)
    assert rel_l2(from_nhwc(y), want) < TOL
    yb = from_nhwc(y)
    s = st.view(rows, 2, cout).sum(0).cpu()
    assert rel_l2(s[0], yb.sum((0, 2, 3))) < 1e-3 + 1e-4
    assert rel_l2(s[1], (yb * yb).sum((0, 2, 3))) < 1e-4


@pytest.mark.parametrize("n,h,w,cin,cout", CONV_SHAPES[:5] + CONV_SHAPES[6:])
def test_conv3x3_dgrad(ops, n, h, w, cin, cout):
    g = torch.Generator().manual_seed(12)
    xv = torch.randn(n, cin, h, w, generator=g).requires_grad_(True)
    wt = bf16_round(torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    dy = bf16_round(torch.randn(n, cout, h, w, generator=g))
    (O.conv3x3(xv, wt) * dy).sum().backward()
    _, wd = ops.prep_conv3x3_weight(wt.cuda())
    dx = torch.empty(n, h, w, cin, dtype=BF16, device="cuda")
    ops.conv3x3(to_nhwc_bf16(dy), wd, dx)
    assert rel_l2(from_nhwc(dx), xv.grad) < TOL


@pytest.mark.parametrize("n,h,w,cin,cout", CONV_SHAPES)
def test_conv3x3_wgrad(ops, n, h, w, cin, cout):
    g = torch.Generator().manual_seed(13)
    x = bf16_round(torch.randn(n, cin, h, w, generator=g))
    wv = torch.zeros(cout, cin, 3, 3, requires_grad=True)
    dy = bf16_round(torch.randn(n, cout, h, w, generator=g))
    (O.conv3x3(x, wv) * dy).sum().backward()
    dw = torch.empty(cout, cin, 3, 3, device="cuda")
    ops.conv3x3_wgrad(to_nhwc_bf16(x), to_nhwc_bf16(dy), dw)
    assert rel_l2(dw, wv.grad) < 1e-4  # fp32 accumulation of exact bf16 products


@pytest.mark.parametrize("n,h,w,cin,cout", [CONV_SHAPES[i] for i in (1, 2, 7, 8, 9, 10, 11, 12)])
@pytest.mark.parametrize("choice", [(-1, -1, -1), (0, 0, 0)])
def test_conv3x3_eval_bn_relu_folded_epilogue(ops, n, h, w, cin, cout, choice):
    """Eval mode: a = bf16(relu(scale * conv(x) + shift)) in the epilogue of every conv kernel (automatic dispatch =
    resident / pair kernels, and the one-tile-per-CTA igemm), against the oracle's conv + eval BatchNorm + ReLU;
    negative scales, a NaN-free zero plateau and a channel-slice destination included."""
    from unet_torch_b200 import _lib

    g = torch.Generator().manual_seed(5)
    x = bf16_round(torch.randn(n, cin, h, w, generator=g))
    wt = bf16_round(torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    gamma, beta = torch.randn(cout, generator=g), torch.randn(cout, generator=g) * 0.3
    rm, rv = torch.randn(cout, generator=g) * 0.2, torch.rand(cout, generator=g) + 0.5
    wf, _ = ops.prep_conv3x3_weight(wt.cuda())
    scale, shift = torch.empty(cout, device="cuda"), torch.empty(cout, device="cuda")
    ops.bn_eval_affine(gamma.cuda(), beta.cuda(), rm.cuda(), rv.cuda(), 1e-5, scale, shift)
    canvas = torch.full((n, h, w, 2 * cout), 7.0, dtype=BF16, device="cuda")
    try:
        _lib.call("b200unet_set_kernel_choice", *choice)
        ops.conv3x3_bn_relu(to_nhwc_bf16(x), wf, scale, shift, canvas[..., cout:])
    finally:
        _lib.call("b200unet_set_kernel_choice", -1, -1, -1)
    want = O.relu(O.batchnorm_eval(O.conv3x3(x, wt), gamma, beta, rm, rv))
    got = from_nhwc(canvas[..., cout:].contiguous())
    assert rel_l2(got, want) < TOL
    assert float(got.min()) == 0.0 and bool((canvas[..., :cout] == 7.0).all())   # ReLU applied; the other slice untouched
    # the unfused pair of launches rounds y to bf16 before the affine: the folded result is at least as close
    y = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    ops.conv3x3(to_nhwc_bf16(x), wf, y)
    a = torch.empty_like(y)
    ops.bn_relu_fwd(y, scale, shift, a)
    assert rel_l2(got, want) <= rel_l2(from_nhwc(a), want) * 1.05 + 1e-6


@pytest.mark.parametrize("cin,cout,hw", [(64, 64, 512), (128, 64, 512), (128, 128, 256), (256, 256, 128), (512, 512, 64),
                                         (1024, 512, 64), (1024, 1024, 32), (256, 128, 256), (64, 128, 256)])
def test_full_size_layers_all_kernel_choices_agree(ops, cin, cout, hw):
    """BASELINE config-2 layer shapes (batch 16): the oracle is too slow here, so the property is that every kernel
    able to run the layer (one-tile-per-CTA igemm, resident, resident pairs, streaming pairs) produces the same
    tensor up to bf16 rounding of differently ordered fp32 sums, and identical BatchNorm statistics to 1e-4."""
    from unet_torch_b200 import _lib

    g = torch.Generator(device="cuda").manual_seed(21)
    x = (torch.randn(16, hw, hw, cin, device="cuda", generator=g) * 0.5).to(BF16)
    w = torch.randn(cout, cin, 3, 3, device="cuda", generator=g) * (2.0 / (9 * cin)) ** 0.5
    wf, _ = ops.prep_conv3x3_weight(w)
    outs = []
    try:
        for choice in ((0, 0, 0), (1, 0, 0), (1, 1, 1), (-1, -1, -1)):
            _lib.call("b200unet_set_kernel_choice", *choice)
            rows = ops.conv3x3_stat_rows(16, hw, hw, cin, cout)
            st = torch.zeros(rows * 2 * cout, device="cuda")
            y = torch.empty(16, hw, hw, cout, dtype=BF16, device="cuda")
            ops.conv3x3(x, wf, y, st)
            outs.append((y.float(), st.view(rows, 2, cout).double().sum(0)))
    finally:
        _lib.call("b200unet_set_kernel_choice", -1, -1, -1)
    y0, s0 = outs[0]
    assert torch.isfinite(y0).all() and float(y0.abs().max()) > 0
    for y, st in outs[1:]:
        assert rel_l2(y, y0) < 2e-3           # both are bf16 roundings of the same fp32 sums, differently ordered
        assert rel_l2(st[1], s0[1]) < 1e-4    # sum of squares
        assert float((st[0] - s0[0]).abs().max()) <= 1e-4 * float(s0[1].sqrt().max()) * (16 * hw * hw) ** 0.5


def test_conv3x3_reads_and_writes_channel_slices(ops):
    """The decoder reads the concat buffer and the encoder writes into it: pitches larger than the channel count."""
    g = torch.Generator().manual_seed(14)
    n, h, w, c = 1, 16, 16, 64
    x = bf16_round(torch.randn(n, c, h, w, generator=g))
    wt = bf16_round(torch.randn(c, c, 3, 3, generator=g) * 0.06)
    wf, _ = ops.prep_conv3x3_weight(wt.cuda())
    xin = torch.full((n, h, w, 3 * c), 7.0, dtype=BF16, device="cuda")
    xin[..., c:2 * c] = to_nhwc_bf16(x)
    yout = torch.zeros(n, h, w, 2 * c, dtype=BF16, device="cuda")
    ops.conv3x3(xin[..., c:2 * c], wf, yout[..., c:])
    assert rel_l2(from_nhwc(yout[..., c:]), O.conv3x3(x, wt)) < TOL
    assert float(yout[..., :c].float().abs().max()) == 0.0


@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 16, 24, 1, 64), (3, 64, 72, 3, 64), (1, 40, 24, 4, 128), (2, 48, 200, 7, 64),
                                            (4, 256, 256, 3, 64)])
def test_first_layer_im2col_gemm_and_wgrad(ops, n, h, w, cin, cout):
    """inc.conv1 (Model.py:111): fp32 NCHW input -> bf16 im2col -> 1x1 tcgen05 GEMM (+ BN statistics), and its wgrad."""
    g = torch.Generator().manual_seed(16)
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5
    col = torch.full((n, h, w, 64), 9.0, dtype=BF16, device="cuda")
    ops.first_im2col(x.cuda(), col)
    # im2col itself is exact: bf16-rounded input taps, zero padding, zero tail columns
    xb = bf16_round(x)
    want_col = torch.nn.functional.unfold(xb, 3, padding=1).view(n, cin * 9, h, w).permute(0, 2, 3, 1)
    assert torch.equal(col[..., : cin * 9].float().cpu(), want_col)
    assert float(col[..., cin * 9:].float().abs().max()) == 0.0
    w1 = ops.prep_first_weight(wt.cuda())
    y = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    rows = ops.conv1x1_c64_stat_rows(n, h, w, cout)
    st = torch.zeros(rows * 2 * cout, device="cuda")
    ops.conv1x1_c64(col, w1, y, st)
    want = O.conv3x3(xb, bf16_round(wt))
    assert rel_l2(from_nhwc(y), want) < TOL
    assert rel_l2(from_nhwc(y), O.conv3x3(x, wt)) < 6e-3  # vs the unrounded fp32 conv: input + weight + output rounding
    yb = from_nhwc(y)
    s = st.view(rows, 2, cout).sum(0).cpu()
    assert rel_l2(s[0], yb.sum((0, 2, 3))) < 1e-3 + 1e-4
    assert rel_l2(s[1], (yb * yb).sum((0, 2, 3))) < 1e-4
    # weight gradient
    dy = bf16_round(torch.randn(n, cout, h, w, generator=g))
    wv = wt.clone().requires_grad_(True)
    (O.conv3x3(xb, wv) * dy).sum().backward()
    dw = torch.empty(cout, cin, 3, 3, device="cuda")
    ops.conv1x1_c64_wgrad(col, to_nhwc_bf16(dy), dw)
    assert rel_l2(dw, wv.grad) < 1e-4
    # ---- the FUSED forms the engine uses: im2col rows built in shared memory inside the GEMM kernels (no `col` in HBM).
    # Same operands, same MMA order -> the very same bits as the materialised path.
    y2 = torch.full((n, h, w, 2 * cout), 5.0, dtype=BF16, device="cuda")
    st2 = torch.zeros(rows * 2 * cout, device="cuda")
    ops.conv3x3_first_tc(x.cuda(), w1, y2[..., cout:], st2)          # into a channel slice, like a concat buffer
    assert torch.equal(y2[..., cout:], y) and bool((y2[..., :cout] == 5.0).all())
    assert torch.equal(st2, st)
    dw2 = torch.empty(cout, cin, 3, 3, device="cuda")
    ops.conv3x3_first_tc_wgrad(x.cuda(), to_nhwc_bf16(dy), dw2)
    assert torch.equal(dw2, dw)
    # eval form: BatchNorm (running statistics) + ReLU folded
    gm, bt = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.2
    rm, rv = torch.randn(cout, generator=g) * 0.2, torch.rand(cout, generator=g) + 0.5
    scale, shift = torch.empty(cout, device="cuda"), torch.empty(cout, device="cuda")
    ops.bn_eval_affine(gm.cuda(), bt.cuda(), rm.cuda(), rv.cuda(), 1e-5, scale, shift)
    a1 = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    a2 = torch.empty(n, h, w, cout, dtype=BF16, device="cuda")
    ops.conv1x1_c64_bn_relu(col, w1, scale, shift, a1)
    ops.conv3x3_first_tc_bn_relu(x.cuda(), w1, scale, shift, a2)
    assert torch.equal(a1, a2)
    assert rel_l2(from_nhwc(a2), O.relu(O.batchnorm_eval(want, gm, bt, rm, rv))) < TOL


UP_SHAPES = [(1, 8, 16, 128, 64), (2, 4, 8, 256, 128), (1, 12, 20, 128, 64),
             # resident-weight variants with several tiles per CTA / the streaming kernel (Cin = 1024)
             (3, 64, 72, 128, 64), (2, 32, 40, 256, 128), (1, 16, 24, 512, 256), (1, 8, 8, 1024, 512)]


@pytest.mark.parametrize("n,h,w,cin,cup", UP_SHAPES)
def test_conv_transpose_fprop_dgrad_wgrad(ops, n, h, w, cin, cup):
    g = torch.Generator().manual_seed(15)
    xv = bf16_round(torch.randn(n, cin, h, w, generator=g)).requires_grad_(True)
    wv = bf16_round(torch.randn(cin, cup, 2, 2, generator=g) * (1.0 / cin) ** 0.5).requires_grad_(True)
    b = torch.randn(cup, generator=g)
    want = O.conv_transpose2x2(xv, wv, b)
    du = bf16_round(torch.randn(want.shape, generator=g))
    (want * du).sum().backward()
    wf, wd = ops.prep_convt2x2_weight(wv.detach().cuda())
    # forward into the right half of a concat buffer
    cat = torch.zeros(n, 2 * h, 2 * w, 2 * cup, dtype=BF16, device="cuda")
    ops.convt2x2(to_nhwc_bf16(xv.detach()), wf, b.cuda(), cat[..., cup:])
    assert rel_l2(from_nhwc(cat[..., cup:]), want) < TOL
    assert float(cat[..., :cup].float().abs().max()) == 0.0
    # backward data / weights from a gradient that also lives in a concat-shaped buffer
    dcat = torch.zeros(n, 2 * h, 2 * w, 2 * cup, dtype=BF16, device="cuda")
    dcat[..., cup:] = to_nhwc_bf16(du)
    dx = torch.empty(n, h, w, cin, dtype=BF16, device="cuda")
    ops.convt2x2_dgrad(dcat[..., cup:], wd, dx)
    assert rel_l2(from_nhwc(dx), xv.grad) < TOL
    dw = torch.empty(cin, cup, 2, 2, device="cuda")
    ops.convt2x2_wgrad(to_nhwc_bf16(xv.detach()), dcat[..., cup:], dw)
    assert rel_l2(dw, wv.grad) < 1e-4


@pytest.mark.parametrize("n,h,w", [(1, 16, 8), (2, 40, 72), (4, 64, 96), (3, 20, 12)])
def test_dgrad_with_fused_batchnorm_backward_reduction(ops, n, h, w):
    """conv3x3_dgrad_bnred (64 -> 64): the backward-data output dx must be the plain kernel's bits, and the partial rows the
    epilogue produces - (sum da, sum da*xhat) with da = dx * [scale*y + shift > 0] of the BatchNorm in front (Model.py:17-18)
    - must reduce to what the host computes from the very same dx and y; ragged tiles (20 x 12) included."""
    g = torch.Generator().manual_seed(31)
    c = 64
    dy = to_nhwc_bf16(torch.randn(n, c, h, w, generator=g))
    wt = torch.randn(c, c, 3, 3, generator=g) * (2.0 / (9 * c)) ** 0.5
    _, wd = ops.prep_conv3x3_weight(wt.cuda())
    y_bn = to_nhwc_bf16(torch.randn(n, c, h, w, generator=g) * 1.5 + 0.3)
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.3
    yf = y_bn.float().cpu()
    mean, var = yf.mean((0, 1, 2)), yf.var((0, 1, 2), unbiased=False)
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    scale, shift = gamma * rstd, beta - mean * gamma * rstd
    dev = lambda t: t.float().cuda().contiguous()  # noqa: E731
    dx_plain = torch.empty(n, h, w, c, dtype=BF16, device="cuda")
    ops.conv3x3(dy, wd, dx_plain)
    dx = torch.empty(n, h, w, c, dtype=BF16, device="cuda")
    sc_d, sh_d, mean_d, rstd_d = dev(scale), dev(shift), dev(mean), dev(rstd)
    pre = ops.conv3x3_dgrad_bnred(dy, wd, dx, y_bn, sc_d, sh_d, mean_d, rstd_d)
    assert pre is not None, "the 64 -> 64 backward-data launch has a fused form"
    partial, rows = pre
    assert torch.equal(dx, dx_plain)
    sums = torch.empty(2 * c, dtype=torch.float64, device="cuda")
    ops.bn_reduce_partials(partial, rows, c, sums)
    dxf = dx.float().cpu().double()
    da = dxf * ((scale.double() * yf.double() + shift.double()) > 0)
    xhat = (yf.double() - mean.double()) * rstd.double()
    want = torch.cat([da.sum((0, 1, 2)), (da * xhat).sum((0, 1, 2))])
    err = float((sums.cpu() - want).abs().max() / want.abs().max())
    assert err < 1e-4, err
    # and the two-pass path gives the same sums
    ws = torch.empty(int(__import__("unet_torch_b200")._lib.query("b200unet_bn_bwd_workspace_floats", n, h, w, c)), device="cuda")
    sums2 = torch.empty(2 * c, dtype=torch.float64, device="cuda")
    import unet_torch_b200

    unet_torch_b200._lib.call("b200unet_bn_relu_bwd_reduce", dx.data_ptr(), c, None, None, y_bn.data_ptr(), c, sc_d.data_ptr(),
                              sh_d.data_ptr(), mean_d.data_ptr(), rstd_d.data_ptr(), ws.data_ptr(), sums2.data_ptr(), n,
                              h, w, c, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert float((sums - sums2).abs().max() / want.abs().max()) < 1e-5
    # shapes without a fused form report it instead of guessing
    assert ops.conv3x3_dgrad_bnred(to_nhwc_bf16(torch.zeros(1, 256, 16, 16)), ops.prep_conv3x3_weight(torch.zeros(256, 256, 3, 3).cuda())[1],
                                   torch.empty(1, 16, 16, 256, dtype=BF16, device="cuda"), to_nhwc_bf16(torch.zeros(1, 256, 16, 16)),
                                   *(torch.zeros(256, device="cuda") for _ in range(4))) is None
