"""-m gpu: the BatchNorm finalisation kernels against fp64, at the edges they are written for.

Every training BatchNorm ends in bn_reduce_finalize (or bn_reduce_partials + bn_finalize under SyncBN): fp32 statistics rows
[rows][2][C] -> fp64 sums -> mean, rstd, scale, shift, running buffers and num_batches_tracked. The attention gates' rows
are pre-reduced by fold_rows; eval mode uses bn_eval_affine / bn_eval_stats; the ConvTranspose2d bias gradient and the dropout
sums use partial_colsum. The reference is the same fp32 inputs summed in fp64 on the host followed by torch's formulas in
fp64, so the bounds are a few fp32 ulps of the quantity (or, for fp32 accumulations, the rounding-error bound of the sum)."""
import math

import numpy as np
import pytest
import torch

from gpu_util import BF16

pytestmark = pytest.mark.gpu

U24 = 2.0 ** -24  # fp32 unit roundoff: one correctly rounded fp32 result is within U24 * |value|


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200  # noqa: F401
    from unet_torch_b200 import ops as _ops

    return _ops


def f32(v):
    return float(np.float32(v))


def assert_ulps(got, want, k, mag=None, what=""):
    """|got - want| <= k * U24 * mag elementwise (mag defaults to |want|), got fp32, want fp64."""
    got = got.detach().double().cpu()
    want = want.double().cpu()
    mag = want.abs() if mag is None else mag.double().cpu()
    err = (got - want).abs()
    bound = k * U24 * mag + 1e-300
    bad = ~(err <= bound)
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} of {bad.numel()} outside {k} ulps, worst at "
                                 f"{int((err / bound).argmax())}: got {got.flatten()[(err / bound).argmax()]:.9g} "
                                 f"want {want.flatten()[(err / bound).argmax()]:.9g}")


def stat_rows(rows, c, k, seed):
    """Statistics rows of `rows` tiles of k pixels each: [rows][2][C] fp32 (sum y, sum y^2 of fp32 y). Channel 0 is the constant
    0.75 (variance exactly 0); channel 1 the constant 1 + 2^-12, whose fp32 square rounds down, so that E[y^2] - E[y]^2 is
    -2^-24 in fp64 and the kernel's clamp to 0 is what keeps rstd finite."""
    g = torch.Generator().manual_seed(seed)
    mu = torch.rand(c, generator=g) * 4 - 2
    sigma = torch.rand(c, generator=g) * 3 + 0.1
    y = mu + sigma * torch.randn(rows, k, c, generator=g)
    y[..., 0] = 0.75
    if c > 1:
        y[..., 1] = 1.0 + 2.0 ** -12
    return torch.stack([y.sum(1), (y * y).sum(1)], 1).contiguous()


def reference(part, count, gamma, beta, eps):
    """torch's BatchNorm2d training formulas in fp64 on fp64 sums of the fp32 rows."""
    s = part.double().sum(0)
    m = s[0] / count
    var = (s[1] / count - m * m).clamp_min(0.0)
    rstd = 1.0 / torch.sqrt(var + f32(eps))
    scale = gamma.double() * rstd
    shift = beta.double() - m * scale
    unbiased = var * count / (count - 1) if count > 1 else var
    return m, var, rstd, scale, shift, unbiased


def check_finalize_outputs(out, ref, gamma, beta, what):
    mean, rstd, scale, shift = (t.cpu() for t in out)
    m, var, r_rstd, r_scale, r_shift, _ = ref
    assert_ulps(mean, m, 2, what=what + " mean")
    assert_ulps(rstd, r_rstd, 2, what=what + " rstd")
    assert_ulps(scale, r_scale, 3, what=what + " scale")
    # shift = beta - mean*scale in fp32 from the rounded mean and scale: bound scaled by the magnitudes of both terms
    assert_ulps(shift, r_shift, 6, mag=beta.double().abs() + (m * r_scale).abs(), what=what + " shift")


@pytest.mark.parametrize("c", [1, 16, 32, 33, 64, 96, 1024])
@pytest.mark.parametrize("rows", [1, 31, 32, 33, 4096])
def test_bn_reduce_finalize_against_fp64(ops, c, rows):
    dev = "cuda"
    g = torch.Generator().manual_seed(1000 * c + rows)
    gamma = torch.rand(c, generator=g) * 2 - 0.5
    beta = torch.randn(c, generator=g)
    rm0 = torch.randn(c, generator=g) * 3
    rv0 = torch.rand(c, generator=g) * 5 + 0.01
    eps = 1e-5
    for k in (1, 3):  # pixels per row: count = rows * k, so rows = 1, k = 1 is count == 1 (no unbiased correction)
        part = stat_rows(rows, c, k, seed=c * 7 + rows * 13 + k)
        count = rows * k
        ref = reference(part, count, gamma, beta, eps)
        m, var, r_rstd, _, _, unbiased = ref
        assert float(var[0]) == 0.0 and (c == 1 or float(var[1]) == 0.0)
        pd = part.to(dev).view(-1)
        gd, bd = gamma.to(dev), beta.to(dev)
        first = None
        for mom in (0.0, 0.1, 0.3, 1.0):
            for tracked in (True, False):
                rm, rv = rm0.to(dev), rv0.to(dev)
                nbt = torch.tensor(7, dtype=torch.int64, device=dev) if tracked else None
                out = [torch.full((c,), float("nan"), device=dev) for _ in range(4)]
                ops.bn_reduce_finalize(pd, rows, count, gd, bd, eps, mom, rm if tracked else None, rv if tracked else None,
                                       nbt, *out)
                # the data-parallel fallback reduces in the same fixed fp64 order: bit-identical
                sums = torch.empty(2 * c, dtype=torch.float64, device=dev)
                ops.bn_reduce_partials(pd, rows, c, sums)
                rm2, rv2 = rm0.to(dev), rv0.to(dev)
                out2 = [torch.full((c,), float("nan"), device=dev) for _ in range(4)]
                ops.bn_finalize(sums, count, gd, bd, eps, mom, rm2 if tracked else None, rv2 if tracked else None, *out2)
                torch.cuda.synchronize()
                what = f"C={c} rows={rows} count={count} momentum={mom} tracked={tracked}"
                for a, b in zip(out, out2):
                    assert torch.equal(a, b), what
                assert torch.equal(rm, rm2) and torch.equal(rv, rv2), what
                if first is None:
                    first = [t.clone() for t in out]
                    check_finalize_outputs(out, ref, gamma, beta, what)
                    # constant channels: rstd = 1/sqrt(eps) exactly as the kernel rounds it, never NaN
                    assert float(out[1][0]) == f32(1.0 / math.sqrt(f32(eps))), what
                    if c > 1:
                        assert float(out[1][1]) == f32(1.0 / math.sqrt(f32(eps))), what
                else:  # momentum and running buffers do not touch the batch statistics
                    for a, b in zip(out, first):
                        assert torch.equal(a, b), what
                if not tracked:
                    assert torch.equal(rm, rm0.to(dev)) and torch.equal(rv, rv0.to(dev)), what
                    continue
                assert int(nbt) == 8, what
                rm_c, rv_c = rm.cpu(), rv.cpu()
                if mom == 0.0:
                    assert torch.equal(rm_c, rm0) and torch.equal(rv_c, rv0), what
                    continue
                if mom == 1.0:  # (1-1)*rm + 1*mean is exact in fp32
                    assert torch.equal(rm_c, out[0].cpu()), what
                    assert_ulps(rv_c, unbiased, 2, what=what + " running_var")
                    continue
                mf = f32(mom)
                a_m, b_m = (1 - mf) * rm0.double(), mf * m
                assert_ulps(rm_c, a_m + b_m, 5, mag=a_m.abs() + b_m.abs(), what=what + " running_mean")
                a_v, b_v = (1 - mf) * rv0.double(), mf * unbiased
                assert_ulps(rv_c, a_v + b_v, 5, mag=a_v.abs() + b_v.abs(), what=what + " running_var")


def test_num_batches_tracked_once_per_launch(ops):
    """32 blocks (C = 1024) finalise together; the counter advances by exactly one per launch."""
    dev = "cuda"
    c, rows = 1024, 33
    part = stat_rows(rows, c, 2, seed=3).to(dev).view(-1)
    gamma, beta = torch.ones(c, device=dev), torch.zeros(c, device=dev)
    rm, rv = torch.zeros(c, device=dev), torch.ones(c, device=dev)
    nbt = torch.tensor(0, dtype=torch.int64, device=dev)
    out = [torch.empty(c, device=dev) for _ in range(4)]
    for i in range(1, 6):
        ops.bn_reduce_finalize(part, rows, 2 * rows, gamma, beta, 1e-5, 0.1, rm, rv, nbt, *out)
        assert int(nbt) == i


def folded_reference(part, out_rows):
    """fp64 residue-class sums: out[b] = sum of the rows r = b (mod out_rows), and the same sums of |x| for the error bound."""
    rows, ncols = part.shape
    q = (rows + out_rows - 1) // out_rows
    pad = torch.zeros(q * out_rows, ncols, dtype=torch.float64, device=part.device)
    pad[:rows] = part.double()
    pv = pad.view(q, out_rows, ncols)
    return pv.sum(0), pv.abs().sum(0), q


def fold_chain(q, ncols):
    """Longest chain of fp32 additions behind one folded value: a lane's share of the q rows, then the lane fold."""
    lanes = 256 // min(ncols, 256)
    return (q + lanes - 1) // lanes + lanes


@pytest.mark.parametrize("rows", [4097, 10000, 131072])
@pytest.mark.parametrize("ncols", [2, 4, 64, 128, 256, 512, 1024])
def test_fold_rows_against_fp64(ops, rows, ncols):
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(rows + ncols)
    part = torch.randn(rows, ncols, device=dev, generator=gen) + 0.5
    assert rows > ops.FOLD_ROWS_ABOVE
    out, out_rows = ops.fold_rows(part.view(-1), rows, ncols)
    assert out_rows == ops.FOLD_ROWS_TO == 296
    want, mag, q = folded_reference(part, out_rows)
    # first-order bound of fp32 recursive summation: (additions in the chain) * u * sum |x|, plus the final rounding
    bound = fold_chain(q, ncols) * U24 * mag + U24 * want.abs()
    err = (out.view(out_rows, ncols).double() - want).abs()
    assert bool((err <= bound).all()), float((err / bound).max())


def test_fold_then_finalize_at_gate_shapes(ops):
    """The BatchNorms of UNet_attention(3, 2)'s four gates - W_q / W_x (C = C_hidden = 32 ... 256) and psi (C = 1) - with the
    row count of a 16 x 512 x 512 map (one statistics row per 8x16 tile, as the GEMM epilogues emit them): fold_rows ->
    bn_reduce_finalize against fp64 over the unfolded rows. The bound carries the fold's fp32 accumulation error through the
    mean and the variance."""
    import unet_torch_b200 as U

    dev = "cuda"
    net = U.UNet_attention(3, 2)
    widths = sorted({m.num_features for a in net._attention_gates() for m in (a.W_q[1], a.W_x[1], a.psi[1])})
    assert widths == [1, 32, 64, 128, 256]
    rows, k = 16 * (512 // 8) * (512 // 16), 4
    assert rows > ops.FOLD_ROWS_ABOVE
    for c in widths:
        gen = torch.Generator(device=dev).manual_seed(c)
        mu = torch.rand(c, device=dev, generator=gen) * 2 - 1
        sigma = torch.rand(c, device=dev, generator=gen) * 1.5 + 0.5
        y = mu + sigma * torch.randn(rows, k, c, device=dev, generator=gen)
        part = torch.stack([y.sum(1), (y * y).sum(1)], 1).contiguous()
        del y
        gamma = torch.rand(c, device=dev, generator=gen) + 0.5
        beta = torch.randn(c, device=dev, generator=gen)
        folded, frows = ops.fold_rows(part.view(-1), rows, 2 * c)
        assert frows == ops.FOLD_ROWS_TO
        out = [torch.empty(c, device=dev) for _ in range(4)]
        ops.bn_reduce_finalize(folded, frows, rows * k, gamma, beta, 1e-5, 0.1, None, None, None, *out)
        count = rows * k
        m, var, r_rstd, r_scale, _, _ = reference(part.cpu(), count, gamma.cpu(), beta.cpu(), 1e-5)
        _, mag, q = folded_reference(part.view(rows, 2 * c), frows)
        fold_err = fold_chain(q, 2 * c) * U24 * mag.sum(0).cpu() / count  # bound on the error of E[y] and E[y^2]
        e1, e2 = fold_err[:c], fold_err[c:]
        mean_bound = e1 + 2 * U24 * m.abs()
        var_bound = e2 + 2 * m.abs() * e1 + e1 * e1
        got_m, got_r, got_s = (t.cpu().double() for t in out[:3])
        assert bool(((got_m - m).abs() <= mean_bound).all()), f"C={c} mean"
        rstd_bound = r_rstd * (0.5 * var_bound / (var + f32(1e-5)) + 2 * U24)
        assert bool(((got_r - r_rstd).abs() <= rstd_bound).all()), f"C={c} rstd"
        scale_bound = gamma.cpu().double() * rstd_bound + 3 * U24 * r_scale.abs()
        assert bool(((got_s - r_scale).abs() <= scale_bound).all()), f"C={c} scale"


@pytest.mark.parametrize("eps", [1e-5, 1e-3])
def test_bn_eval_affine_and_stats_against_fp64(ops, eps):
    dev = "cuda"
    c = 300  # not a multiple of the 128-thread block
    g = torch.Generator().manual_seed(11)
    gamma = torch.randn(c, generator=g)
    beta = torch.randn(c, generator=g)
    rm = torch.randn(c, generator=g) * 4
    rv = torch.rand(c, generator=g) * 3
    rv[:20] = 0.0                                              # variance near 0: eps decides rstd
    rv[20:40] = torch.rand(20, generator=g) * 1e-6
    rv[40:60] = torch.rand(20, generator=g) * 1e6 + 1e4       # large: eps below one ulp of rv
    rstd = 1.0 / torch.sqrt(rv.double() + f32(eps))
    scale_w = gamma.double() * rstd
    shift_w = beta.double() - rm.double() * scale_w
    scale = torch.full((c,), float("nan"), device=dev)
    shift = torch.full((c,), float("nan"), device=dev)
    ops.bn_eval_affine(gamma.to(dev), beta.to(dev), rm.to(dev), rv.to(dev), eps, scale, shift)
    # fp32: rv + eps, sqrt, reciprocal, times gamma - each correctly rounded
    assert_ulps(scale.cpu(), scale_w, 4, what="scale")
    assert_ulps(shift.cpu(), shift_w, 6, mag=beta.double().abs() + (rm.double() * scale_w).abs(), what="shift")
    mean = torch.full((c,), float("nan"), device=dev)
    rs = torch.full((c,), float("nan"), device=dev)
    ops.bn_eval_stats(rm.to(dev), rv.to(dev), eps, mean, rs)
    assert torch.equal(mean.cpu(), rm)
    assert_ulps(rs.cpu(), rstd, 3, what="rstd")
    with pytest.raises(RuntimeError, match="running statistics"):
        ops.bn_eval_affine(gamma.to(dev), beta.to(dev), None, None, eps, scale, shift)
    with pytest.raises(RuntimeError, match="running statistics"):
        ops.bn_eval_stats(None, None, eps, mean, rs)


@pytest.mark.parametrize("rows", [1, 7, 8, 9, 1000])
@pytest.mark.parametrize("n", [1, 31, 33, 64])
def test_partial_colsum_against_fp64(ops, rows, n):
    """Columns [col_lo, col_lo + n) of [rows][row_pitch] rows; every other column is NaN, so reading one shows up, and the
    output tensor continues past n with a sentinel that must survive."""
    dev = "cuda"
    col_lo, row_pitch = 5, n + 12
    g = torch.Generator().manual_seed(rows * 100 + n)
    part = torch.full((rows, row_pitch), float("nan"))
    part[:, col_lo:col_lo + n] = torch.randn(rows, n, generator=g) * 10 + 3
    out = torch.full((n + 8,), -7.0, device=dev)
    ops.partial_colsum(part.to(dev).view(-1), rows, row_pitch, col_lo, n, out[:n])
    sel = part[:, col_lo:col_lo + n].double()
    want = sel.sum(0)
    # fp64 accumulation, one fp32 rounding at the end
    bound = U24 * want.abs() + rows * 2.0 ** -52 * sel.abs().sum(0)
    assert bool(((out[:n].cpu().double() - want).abs() <= bound).all())
    assert bool((out[n:].cpu() == -7.0).all())


@pytest.mark.parametrize("c", [64, 2048])
def test_channel_sum_of_a_channel_slice(ops, c):
    dev = "cuda"
    n, h, w = 2, 64, 32
    g = torch.Generator().manual_seed(c)
    wide = torch.full((n, h, w, c + 64), float("nan")).to(BF16)
    x = (torch.randn(n, h, w, c, generator=g) + 0.5).to(BF16)
    wide[..., 64:] = x
    out = torch.full((c,), float("nan"), device=dev)
    ops.channel_sum(wide.to(dev)[..., 64:], out)
    xs = x.double().view(-1, c)
    want, mag = xs.sum(0), xs.abs().sum(0)
    # per-thread fp32 sums, an fp32 block reduction over the 256 / (C/8) threads of a channel group, fp64 across blocks
    pixels = n * h * w
    total = pixels * (c // 8)
    blocks = min((total + 255) // 256, 148 * 8)
    chain = (total + blocks * 256 - 1) // (blocks * 256) + max(256 // (c // 8), 1)
    bound = chain * U24 * mag + U24 * want.abs()
    assert bool(((out.cpu().double() - want).abs() <= bound).all())
