"""Exact-arithmetic checks of the tensor-core convolution kernels: operand generators, fp64 references, sentinel canvases and
a launch recorder (tests/test_gpu_conv_exact.py; the checker itself is validated on the CPU in tests/test_host_logic.py).

Why the comparisons can be exact: with small-integer operands every product is an integer and every partial sum is an
integer below 2^16, so an fp32 accumulator holds the exact value whatever the order of summation, the K split or the MMA
shape. A bf16 output then equals bf16_rne(exact) bit for bit, and an fp32 output (weight gradients, statistics rows) equals
the exact value outright.

Regimes (both seeded; `check_regime` asserts the invariant of each on the host, in fp64, before a case is used):
- sparse: ternary x at a density of min(0.3, 128 / K), ternary w. Every output satisfies |y| <= 256, so it is exact in bf16,
  and the BatchNorm sums Sum(y) and Sum(y^2) per channel stay below 2^24: exact in an fp32 row.
- dense: integers in [-m, m] at a density of min(1, 576 / K), with m the largest value for which the expected Sum|x*w| of an
  output stays at 0.35 * 2^16. Most outputs exceed 256, so the bf16 rounding of the epilogue (and its ties) is exercised:
  at least 30 % of the outputs must be changed by it.
K is the number of products per output element (9 * Cin for a 3x3 conv, Cin for a 1x1 conv, the pixel count for a weight
gradient)."""
import re

import torch
import torch.nn.functional as F

BF16 = torch.bfloat16
F64 = torch.float64
SPARSE, DENSE = "sparse", "dense"
ABS_LIMIT = 2 ** 16          # Sum|x*w| per output element, both regimes
SUM_LIMIT = 2 ** 24          # Sum|y| and Sum(y^2) per channel, sparse regime
MIN_ROUNDED = 0.30           # dense regime: share of the outputs the bf16 rounding changes
DENSE_K = 576                # the dense regime keeps K * density at this (9 * 64: one 64-channel 3x3 conv)
BF16_SENTINEL = 0x7FAB       # a quiet-NaN payload no kernel produces
F32_SENTINEL = 0x7FABCDEF


# --------------------------------------------------------------------------------------------- operands
def density(regime, k):
    return min(0.3, 128.0 / k) if regime == SPARSE else min(1.0, DENSE_K / k)


def dense_m(k):
    """Largest m with K_eff * E|v|^2 <= 0.35 * 2^16 for v uniform on [-m, m] (E|v| = m(m+1)/(2m+1)), capped at 128 so that
    every operand is exact in bf16. Below K = 256 a sum of K terms does not concentrate near its mean: there m also keeps the
    worst case K * m^2 below 2^16."""
    keff = k * density(DENSE, k)
    m = 1
    while m < 128 and keff * ((m + 1) * (m + 2) / (2 * m + 3)) ** 2 <= 0.35 * ABS_LIMIT:
        m += 1
    while k < 256 and m > 1 and k * m * m >= ABS_LIMIT:
        m -= 1
    return m


def operand(shape, regime, k, gen, sparse_input=True):
    """Integer-valued fp64 tensor. sparse_input: the operand that carries the density (the activations); the weight-like
    operand is dense."""
    m = 1 if regime == SPARSE else dense_m(k)
    v = torch.randint(-m, m + 1, shape, generator=gen).to(F64)
    d = density(regime, k) if sparse_input else 1.0
    if d < 1.0:
        v = v * (torch.rand(shape, generator=gen) < d)
    return v


def check_regime(regime, y, y_abs, channel_dim=1, rounded_out=True):
    """y: the exact fp64 result; y_abs: the same operation on |operands| (Sum|x*w| per element). Raises if the case breaks
    its regime's invariant: the exactness argument would not hold, so the case must not be used."""
    peak = float(y_abs.max()) if y_abs.numel() else 0.0
    assert peak < ABS_LIMIT, f"{regime}: Sum|x*w| reaches {peak:.0f} >= 2^16"
    if regime == SPARSE:
        assert torch.equal(bf16_rne(y), y), "sparse: an output is not exact in bf16"
        if rounded_out:
            dims = [d for d in range(y.dim()) if d != channel_dim % y.dim()]
            s1, s2 = y.abs().sum(dims), (y * y).sum(dims)
            assert float(s1.max()) < SUM_LIMIT and float(s2.max()) < SUM_LIMIT, "sparse: channel sums reach 2^24"
    elif rounded_out:
        share = float((bf16_rne(y) != y).double().mean())
        assert share >= MIN_ROUNDED, f"dense: only {share:.1%} of the outputs are rounded (needs {MIN_ROUNDED:.0%})"


def bf16_rne(t):
    """Round to bf16, nearest-even, returned in t's dtype. From fp64 through fp32: exact for values below 2^24."""
    return t.to(torch.float32).to(BF16).to(t.dtype)


def bf16_rz(t):
    """Round toward zero to bf16 (the defect the tests must notice): drop the low 16 bits of the fp32 value."""
    u = t.to(torch.float32).view(torch.int32) & ~0xFFFF
    return u.view(torch.float32).to(t.dtype)


# --------------------------------------------------------------------------------------------- fp64 references (NCHW)
# Plain fp64 GEMM-style convolutions: cuDNN is switched off, because its FFT / Winograd algorithms would round the integer
# partial sums that make these references exact.
def _exact(fn):
    def wrapped(*args, **kw):
        with torch.backends.cudnn.flags(enabled=False):
            return fn(*args, **kw)

    wrapped.__name__, wrapped.__doc__ = fn.__name__, fn.__doc__
    return wrapped


@_exact
def conv3x3(x, w):
    """fp64 conv3x3, padding 1. x [N,C,H,W], w [K,C,3,3]."""
    return F.conv2d(x.to(F64), w.to(F64), padding=1)


@_exact
def conv3x3_dgrad(dy, w):
    """Gradient at the input of conv3x3(x, w) for the output gradient dy [N,K,H,W]."""
    return F.conv_transpose2d(dy.to(F64), w.to(F64), padding=1)


@_exact
def conv3x3_wgrad(x, dy):
    """Sum over pixels of dy (x) the 3x3 neighbourhood of x: [K,C,3,3]."""
    x, dy = x.to(F64), dy.to(F64)
    n, c, h, w = x.shape
    cols = F.unfold(x, 3, padding=1).view(n, c * 9, h * w)
    return torch.einsum("nkp,nqp->kq", dy.reshape(n, dy.shape[1], h * w), cols).view(dy.shape[1], c, 3, 3)


def bn_relu_eval(y, scale, shift):
    """max(scale * y + shift, 0) per channel (dim 1)."""
    return torch.clamp_min(y * scale.to(F64).view(1, -1, 1, 1) + shift.to(F64).view(1, -1, 1, 1), 0.0)


def bn_backward_sums(g, y, scale, shift, mean, rstd):
    """The first pass of BatchNorm+ReLU backward: (Sum da, Sum da * xhat) per channel, da = g * [scale * y + shift > 0],
    xhat = (y - mean) * rstd."""
    sh = (1, -1, 1, 1)
    g, y = g.to(F64), y.to(F64)
    da = g * ((scale.to(F64).view(sh) * y + shift.to(F64).view(sh)) > 0)
    xhat = (y - mean.to(F64).view(sh)) * rstd.to(F64).view(sh)
    return da.sum((0, 2, 3)), (da * xhat).sum((0, 2, 3))


@_exact
def convt2x2(x, w, bias=None):
    """ConvTranspose2d(kernel 2, stride 2). x [N,Cin,H,W], w [Cin,Cup,2,2]."""
    return F.conv_transpose2d(x.to(F64), w.to(F64), None if bias is None else bias.to(F64), stride=2)


@_exact
def convt2x2_dgrad(du, w):
    """Gradient at the input of convt2x2 for du [N,Cup,2H,2W]: a stride-2 2x2 convolution."""
    return F.conv2d(du.to(F64), w.to(F64), stride=2)


@_exact
def convt2x2_wgrad(x, du):
    """[Cin,Cup,2,2]: dW[c,d,i,j] = Sum x[n,c,h,w] du[n,d,2h+i,2w+j]."""
    x, du = x.to(F64), du.to(F64)
    n, c, h, w = x.shape
    d = du.view(n, du.shape[1], h, 2, w, 2)
    return torch.einsum("nchw,ndhiwj->cdij", x, d)


@_exact
def conv1x1(x, w, bias=None):
    """x [N,Cin,H,W], w [Cout,Cin]."""
    y = torch.einsum("nchw,kc->nkhw", x.to(F64), w.to(F64))
    return y if bias is None else y + bias.to(F64).view(1, -1, 1, 1)


@_exact
def conv1x1_wgrad(x, dy):
    """[Cout,Cin] = Sum over pixels dy (x) x."""
    return torch.einsum("nchw,nkhw->kc", x.to(F64), dy.to(F64))


def channel_sums(y):
    """(Sum y, Sum y^2) per channel of an NCHW tensor, fp64."""
    y = y.to(F64)
    return y.sum((0, 2, 3)), (y * y).sum((0, 2, 3))


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def nchw(t):
    return t.permute(0, 3, 1, 2)


# --------------------------------------------------------------------------------------------- comparison
RES_TILE = (16, 8)     # conv3_res / conv3_res2 / conv3_pair output tile (rows, columns)
IGEMM_TILE = (8, 16)   # igemm / wgrad pixel tile


def _tile(h, w, H, W, tile):
    th, tw = tile
    tiles_w = (W + tw - 1) // tw
    return (h // th) * tiles_w + (w // tw)


def assert_exact(got, want, what="output", limit=6):
    """Element-for-element equality with torch.equal semantics (-0.0 == 0.0; NaN never equal). 4-d tensors are NHWC
    activations: a mismatch report names (n, h, w, c) and the (image, tile) it falls in under both tile geometries."""
    got, want = got.to(F64).cpu(), want.to(F64).cpu()
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} != {tuple(want.shape)}"
    bad = ~(got == want)
    nbad = int(bad.sum())
    if nbad == 0:
        return
    idx = bad.nonzero()[:limit].tolist()
    lines = []
    for i in idx:
        g, v = float(got[tuple(i)]), float(want[tuple(i)])
        if got.dim() == 4:
            n, h, w, c = i
            _, H, W, _ = got.shape
            lines.append(f"  (n={n}, h={h}, w={w}, c={c}): got {g!r}, want {v!r}; image {n}, 16x8 tile "
                         f"{_tile(h, w, H, W, RES_TILE)}, 8x16 tile {_tile(h, w, H, W, IGEMM_TILE)}")
        else:
            lines.append(f"  {tuple(i)}: got {g!r}, want {v!r}")
    raise AssertionError(f"{what}: {nbad} of {got.numel()} elements differ\n" + "\n".join(lines))


def rel_l2(got, want):
    got, want = got.to(F64).cpu(), want.to(F64).cpu()
    return float((got - want).norm() / max(float(want.norm()), 1e-300))


# --------------------------------------------------------------------------------------------- sentinel canvases
GUARD_C = 8  # channels of sentinel on each side of a slice (16 bytes: keeps the slice's TMA base aligned)


def bf16_canvas(n, h, w, c, device="cuda"):
    """[n + 1, h, w, c + 2 * GUARD_C] bf16 filled with the sentinel NaN; returns (canvas, target slice [n, h, w, c])."""
    canvas = torch.full((n + 1, h, w, c + 2 * GUARD_C), BF16_SENTINEL, dtype=torch.int16, device=device).view(BF16)
    return canvas, canvas[:n, :, :, GUARD_C:GUARD_C + c]


def input_canvas(x_nhwc, device="cuda"):
    """An NHWC input as the channel slice of a sentinel canvas with a guard image: a read outside the slice or past the last
    image brings a NaN into the output."""
    n, h, w, c = x_nhwc.shape
    canvas, sl = bf16_canvas(n, h, w, c, device)
    sl.copy_(x_nhwc.to(device=device, dtype=BF16))
    return canvas, sl


def f32_sentinel(numel, device="cuda"):
    return torch.full((numel,), F32_SENTINEL, dtype=torch.int32, device=device).view(torch.float32)


def stats_buffer(rows, c, device="cuda"):
    """[rows + 1][2][c] fp32 sentinel NaN: one guard row after the rows the kernel must write."""
    return f32_sentinel((rows + 1) * 2 * c, device)


def assert_canvas_intact(canvas, n, c, what="output"):
    """Everything outside canvas[:n, ..., GUARD_C:GUARD_C + c] is still the sentinel, bit for bit; the target is finite."""
    bits = canvas.view(torch.int16)
    keep = torch.ones(bits.shape, dtype=torch.bool, device=bits.device)
    keep[:n, :, :, GUARD_C:GUARD_C + c] = False
    changed = int((bits[keep] != BF16_SENTINEL).sum())
    assert changed == 0, f"{what}: {changed} elements outside the target were written"
    target = canvas[:n, :, :, GUARD_C:GUARD_C + c].float()
    nonfinite = int((~torch.isfinite(target)).sum())
    assert nonfinite == 0, f"{what}: {nonfinite} target elements are not finite (unwritten, or a NaN read from outside the input)"


def assert_stats_rows(buf, rows, c, what="statistics"):
    """Rows [0, rows) of a [rows + 1][2][c] buffer are finite; the guard row is still the sentinel."""
    v = buf.view(rows + 1, 2 * c)
    bad = (~torch.isfinite(v[:rows])).any(1).nonzero().flatten().tolist()
    assert not bad, f"{what}: rows {bad[:8]} of {rows} hold non-finite values (left unwritten?)"
    assert bool((v[rows].view(torch.int32) == F32_SENTINEL).all()), f"{what}: the guard row after row {rows} was written"


# --------------------------------------------------------------------------------------------- launch recorder
_KERNEL = re.compile(r"(\w+)(<[^()]*>)?\(")


def kernel_name(profiler_name):
    """'void (anonymous namespace)::conv3_pair_kernel<256, 2, 6, 1>((anonymous namespace)::PairArgs)' ->
    'conv3_pair_kernel<256, 2, 6, 1>'."""
    m = _KERNEL.match(re.sub(r"^(void )?(\(anonymous namespace\)::)?", "", profiler_name))
    return (m.group(1) + (m.group(2) or "")) if m else profiler_name


def launched_kernels(fn):
    """Runs fn under torch.profiler (CUDA activity) and returns the names of the kernels it launched, in launch order, as
    `kernel_name` spells them."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memset", "Memcpy"))]
    evs.sort(key=lambda e: e.time_range.start)
    return [kernel_name(e.name) for e in evs]
