"""Exact-arithmetic checks of the bandwidth kernels in csrc/elementwise.cu (BatchNorm-apply + ReLU, 2x2 max pool, the two
BatchNorm+ReLU backward passes, channel-slice copy / add): an exact emulation of fp32 fmaf, fp64 references, error bounds,
sentinel buffers and the launch-grid formulas (tests/test_gpu_bn_relu_exact.py; the checker itself is validated on the CPU
in tests/test_host_logic.py).

What the kernels compute (y, g1, g_pool bf16; scale, shift, gamma, mean, rstd fp32; f32() / bf16() round to nearest even):
- forward: a = bf16(max(fmaf(sc, y, sh), 0)); pooled = the first maximum of the four bf16 values of a 2x2 window in row-major
  order, pool_idx its position 0..3. maxpool2x2 applies the same rule to a stored bf16 tensor, and a NaN wins.
- backward: da = f32(g1 + [k == idx] g_pool), zero where !(fmaf(sc, y, sh) > 0) (the fp32 pre-activation, not the stored a).
  The reduce pass gives dbeta = Sum da and dgamma = rstd (Sum da y - mean Sum da); the apply pass
  dy = bf16(fmaf(k1, da, fmaf(k2, y, k3))) with k1 = f32(g r), k2 = f32(-g r^2 sdx), k3 = f32(-g r sda + g r^2 m sdx) from
  sda = sums[c] / count, sdx = sums[C + c] / count (k3 is evaluated in fp64 on the device, where nvcc may contract it).
- nhwc_add: bf16(f32(a) + f32(b)); nhwc_copy: a bit copy.

Which results are exact: everything in the forward (fmaf is emulated exactly, below), the ReLU mask, the pooled values and
positions, nhwc_copy / nhwc_add, and dy of a frozen BatchNorm (zero sums: dy = bf16(f32(k1 da))). dgamma / dbeta are exact
in the sparse regime of the tests (integer partial sums below 2^24, power-of-two rstd); otherwise they and dy are held to the
bounds of `sum_bounds` and `dy_bound`.

The references run with torch in float64 on the tensors' own device: full-size activations are too large for a CPU
reference inside the suite's time budget."""
import math

import torch

import conv_check as C

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
BF16_SENTINEL, F32_SENTINEL, U8_SENTINEL = C.BF16_SENTINEL, C.F32_SENTINEL, 0xAB
GUARD = 1024            # sentinel elements after a contiguous output
U = 2.0 ** -24          # unit roundoff of fp32

# ------------------------------------------------------------------------------------------------ launch grids
# Restated from csrc/elementwise.cu so that a test case can be placed on a grid-stride edge and the bounds can count the
# terms one thread sums. They hold for the default grid only: B200UNET_FWD_BLOCKS_PER_SM / B200UNET_BWD_BLOCKS_PER_SM change
# the caps and B200UNET_EW_REV the traversal order.
GRID_ENV = ("B200UNET_EW_REV", "B200UNET_FWD_BLOCKS_PER_SM", "B200UNET_BWD_BLOCKS_PER_SM")
EW_THREADS = 256            # EW_THREADS
EW_MAX_BLOCKS = 148 * 8     # EW_MAX_BLOCKS (ew_blocks) = the forward cap of 8 blocks per SM (b200unet_bn_relu_fwd)
BWD_MAX_BLOCKS = 148 * 2    # bwd_blocks(): 2 resident blocks per SM
UNROLL = {False: 4, True: 1}  # items in flight per thread (U) of bn_relu_fwd_kernel / bn_bwd_*_kernel: plain / pooled


def work_items(n, h, w, c, pool):
    """Grid-stride items of the BN kernels: one 8-channel group of one pixel, or of one 2x2 window when pooled."""
    return (n * (h // 2) * (w // 2) if pool else n * h * w) * (c // 8)


def ew_blocks(items):
    return max(1, min(-(-items // EW_THREADS), EW_MAX_BLOCKS))


def grid(kind, items):
    """(blocks, stride) of a launch over `items` work items. kind: 'fwd' (bn_relu_fwd), 'bwd' (both backward passes) or
    'ew' (maxpool2x2, nhwc_copy, nhwc_add)."""
    b = ew_blocks(items)
    if kind == "bwd":
        b = min(b, BWD_MAX_BLOCKS)
    return b, b * EW_THREADS


def items_per_thread(kind, items):
    return -(-items // grid(kind, items)[1])


def terms_per_thread(n, h, w, c, pool):
    """The most pixels whose da one backward thread sums in fp32 (the k of gamma_k)."""
    return items_per_thread("bwd", work_items(n, h, w, c, pool)) * (4 if pool else 1)


def gamma_k(k):
    return k * U / (1.0 - k * U)


# ------------------------------------------------------------------------------------------------ exact fmaf
def fmaf(a, b, c):
    """fp32 fmaf(a, b, c), emulated exactly in fp64, for fp32 a, b, c whose product is exact in fp64 (fp32 x bf16: 32
    significant bits, fp32 x fp32: 48). Returns (result, midpoint): the result as fp64 holding the fp32 value, and the mask
    of the elements that went through the double-rounding branch.

    p = a b is exact and s = p + c rounds once in fp64. Rounding s to fp32 is then correct unless s landed exactly on the
    midpoint between two fp32 values while p + c did not (a double rounding): those elements are detected and resolved by
    the TwoSum error term e (p + c == s + e exactly) - toward its sign, and ties-to-even when it is zero."""
    a, b, c = a.to(F64), b.to(F64), c.to(F64)
    p = a * b
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.to(F32)
    r64 = r.to(F64)
    inf = torch.full_like(r, math.inf)
    nb = torch.nextafter(r, torch.where(s > r64, inf, -inf))     # the other fp32 neighbour of s
    mid = (s != r64) & ((r64 + nb.to(F64)) * 0.5 == s) & (e != 0)
    fixed = torch.where(e > 0, torch.maximum(r, nb), torch.minimum(r, nb))
    return torch.where(mid, fixed, r).to(F64), mid


# a * b = 2^30 + rho (rho = +-1) with a < 2^24 and b < 256 odd: products of an fp32 and a bf16 significand that put the sum
# s = K 2^-23 + a b 2^-54 (K a 24-bit integer) exactly on an fp32 midpoint in fp64, while the exact sum is off it by rho 2^-54
# (below half an fp64 ulp of s, so the fp64 addition rounds it away).
MIDPOINT_PRODUCTS = ((16519105, 65, 1), (5237765, 205, 1), (13944699, 77, -1), (11545611, 93, -1), (10845877, 99, -1),
                     (7110873, 151, -1), (4948119, 217, -1), (4648233, 231, -1))


def midpoint_case(i, hi_bits, j):
    """(sc, y, sh) as Python floats with fmaf(sc, y, sh) on the double-rounding branch, and the branch visible after the
    bf16 rounding of the forward: K's low 17 bits make the two candidate fp32 results round to different bf16 values
    (rho = +1: K even at a bf16 tie that rounds down; rho = -1: K odd just below a tie that rounds up). hi_bits: 0..63 picks
    the rest of K, j a power-of-two scale of the whole case."""
    a, b, rho = MIDPOINT_PRODUCTS[i % len(MIDPOINT_PRODUCTS)]
    k = (1 << 23) | (hi_bits << 17) | (0x08000 if rho > 0 else 0x17FFF)
    return math.ldexp(a, j - 47), math.ldexp(b, -7), math.ldexp(k, j - 23)


def plant_midpoints(scale, shift, y, gen, channels=8, share=0.5):
    """Overwrites scale / shift of the first `channels` channels with `midpoint_case`s and sets a share of those channels'
    y (NHWC, last dim) to the case's y, so that real kernel inputs go through the double-rounding branch."""
    for c in range(channels):
        sc, yv, sh = midpoint_case(c, int(torch.randint(0, 64, (1,), generator=gen)), int(torch.randint(-3, 4, (1,), generator=gen)))
        scale[c], shift[c] = sc, sh
        pick = torch.rand(y.shape[:-1], generator=gen, device="cpu").to(y.device) < share
        y[..., c][pick] = yv


# ------------------------------------------------------------------------------------------------ references
def to_bf16(x):
    """bf16 RNE of fp64 values that are exact fp32 values (a single rounding)."""
    return x.to(F32).to(BF16)


def bn_relu_fwd(y, scale, shift):
    """(a bf16, pre-activation fp64 = f32(fmaf(sc, y, sh)), midpoint mask) over NHWC y."""
    pre, mid = fmaf(scale, y, shift)
    return to_bf16(torch.clamp_min(pre, 0.0)), pre, mid


WINDOW = ((0, 0), (0, 1), (1, 0), (1, 1))   # position k of a 2x2 window: (row, column) = (k >> 1, k & 1)


def maxpool2x2(a):
    """(pooled, idx uint8) of NHWC bf16 a: the first maximum in row-major window order; a NaN wins (the last one)."""
    v = [a[:, dh::2, dw::2].float() for dh, dw in WINDOW]
    best, idx = v[0], torch.zeros(v[0].shape, dtype=torch.uint8, device=a.device)
    for k in (1, 2, 3):
        take = (v[k] > best) | torch.isnan(v[k])
        best = torch.where(take, v[k], best)
        idx = torch.where(take, torch.full_like(idx, k), idx)
    return best.to(BF16), idx


def unpool(g_pool, idx, h, w):
    """g_pool scattered to the window positions idx: [N, H, W, C] fp64."""
    n, _, _, c = g_pool.shape
    out = torch.zeros((n, h, w, c), dtype=F64, device=g_pool.device)
    gp = g_pool.to(F64)
    for k, (dh, dw) in enumerate(WINDOW):
        out[:, dh::2, dw::2] = torch.where(idx == k, gp, 0.0)
    return out


def bwd_da(y, g1, g_pool, idx, scale, shift):
    """da (fp64 holding fp32 values): f32(g1 + [k == idx] g_pool), zero where !(fmaf(sc, y, sh) > 0)."""
    pre, _ = fmaf(scale, y, shift)
    g = torch.zeros(y.shape, dtype=F64, device=y.device) if g1 is None else g1.to(F64)
    if g_pool is not None:
        g = (g + unpool(g_pool, idx, y.shape[1], y.shape[2])).to(F32).to(F64)
    return torch.where(pre > 0, g, 0.0)


def bwd_sums(da, y):
    """Per channel: Sum da, Sum da y, Sum |da|, Sum |da y| (fp64; add chunks together)."""
    dims = tuple(range(da.dim() - 1))
    dy = da * y.to(F64)
    return torch.stack([da.sum(dims), dy.sum(dims), da.abs().sum(dims), dy.abs().sum(dims)])


def param_grads(sums, mean, rstd):
    """(dgamma, dbeta) in fp64 from the exact sums: rstd (Sum da y - mean Sum da), Sum da."""
    s1, s2 = sums[0], sums[1]
    return rstd.to(F64) * (s2 - mean.to(F64) * s1), s1


def sum_bounds(sums, mean, rstd, k):
    """Bounds on |dgamma - exact| and |dbeta - exact| for the reduce pass: each thread sums at most k terms per channel in
    fp32 (gamma_k), every block partial is rounded to fp32 (2^-23 of Sum_blocks |partial| <= (1 + gamma_k) Sum |term|), and
    the result once more (2^-24). The fp64 stages in between are below 2^-50 relative and covered by the slack of 2^-23."""
    s1, s2, a1, a2 = sums
    m, r = mean.to(F64).abs(), rstd.to(F64)
    gk = gamma_k(k)
    ag = r * (a2 + m * a1)
    dgamma, dbeta = param_grads(sums, mean, rstd)
    bg = gk * ag + 2.0 ** -23 * (1 + gk) * ag + U * dgamma.abs()
    bb = gk * a1 + 2.0 ** -23 * (1 + gk) * a1 + U * dbeta.abs()
    return bg, bb


def ulp_bf16(x):
    """ulp of bf16 at |x| (fp64 tensor); 0 at 0."""
    _, e = torch.frexp(x.abs())
    return torch.where(x != 0, torch.ldexp(torch.ones_like(x), (e - 8).clamp_min(-133)), 0.0)


def dy_ref(da, y, gamma, mean, rstd, sums, count):
    """(dy exact in fp64 for the device's k1..k3 formula with exact sums, |k1 da| + |k2 y| + |k3| for the bound).
    sums: fp64 [2, C] (Sum da, Sum da xhat) as the apply pass receives them."""
    g, r, m = gamma.to(F64), rstd.to(F64), mean.to(F64)
    sda, sdx = sums[0] / count, sums[1] / count
    k1, k2, k3 = g * r, -g * r * r * sdx, -g * r * sda + g * r * r * m * sdx
    y = y.to(F64)
    return k1 * da + (k2 * y + k3), (k1 * da).abs() + (k2 * y).abs() + k3.abs()


def dy_bound(ref, mag, y, gamma, mean, rstd, count, bg=None, bb=None):
    """|dy - ref| bound: 1/2 ulp_bf16 of the output, 4 fp32 roundings of the terms (k1, k2, k3 and the two fmaf), and, when the
    sums are the device's own rather than exact, their error bounds bg / bb (on Sum da xhat and Sum da) carried through
    k2 and k3: |g r| bb / count + |g| r^2 |y - m| bg / (r count)."""
    e = 4 * U * mag
    if bg is not None:
        g, r = gamma.to(F64).abs(), rstd.to(F64)
        e = e + g * r * bb / count + g * r * (y.to(F64) - mean.to(F64)).abs() * bg / count
    return 0.5 * ulp_bf16(ref.abs() + e) + e


# ------------------------------------------------------------------------------------------------ comparisons
def assert_equal(got, want, what, limit=6):
    """Value equality on the device (-0.0 == 0.0; NaN equals NaN). Reports the first mismatches with their NHWC index."""
    g, w = got.to(F64), want.to(F64)
    bad = ~((g == w) | (torch.isnan(g) & torch.isnan(w)))
    nbad = int(bad.sum())
    if nbad:
        idx = bad.nonzero()[:limit]
        lines = [f"  {tuple(i.tolist())}: got {float(g[tuple(i)])!r}, want {float(w[tuple(i)])!r}" for i in idx]
        raise AssertionError(f"{what}: {nbad} of {got.numel()} elements differ\n" + "\n".join(lines))


def assert_within(got, want, bound, what, limit=6):
    """|got - want| <= bound element by element; returns the worst |got - want| / bound (0 where both are 0)."""
    err = (got.to(F64) - want).abs()
    bad = ~(err <= bound)
    nbad = int(bad.sum())
    if nbad:
        idx = bad.nonzero()[:limit]
        lines = [f"  {tuple(i.tolist())}: got {float(got[tuple(i)])!r}, want {float(want[tuple(i)])!r}, bound "
                 f"{float(bound[tuple(i)]):.3e}" for i in idx]
        raise AssertionError(f"{what}: {nbad} of {got.numel()} elements outside the bound\n" + "\n".join(lines))
    ratio = torch.where(err > 0, err / bound, 0.0)
    return float(ratio.max()) if ratio.numel() else 0.0


# ------------------------------------------------------------------------------------------------ sentinel buffers
def sentinel_like(numel, dtype, device="cuda"):
    if dtype == BF16:
        return torch.full((numel,), BF16_SENTINEL, dtype=torch.int16, device=device).view(BF16)
    if dtype == F32:
        return torch.full((numel,), F32_SENTINEL, dtype=torch.int32, device=device).view(F32)
    return torch.full((numel,), U8_SENTINEL, dtype=torch.uint8, device=device)


def guarded(shape, dtype, device="cuda"):
    """(buffer, view): a contiguous tensor of `shape` at the start of a sentinel buffer with GUARD more elements after it."""
    numel = math.prod(shape)
    buf = sentinel_like(numel + GUARD, dtype, device)
    return buf, buf[:numel].view(shape)


def _bits(t):
    return t.view({BF16: torch.int16, F32: torch.int32, torch.uint8: torch.uint8}[t.dtype])


def _sentinel_bits(dtype):
    return {BF16: BF16_SENTINEL, F32: F32_SENTINEL, torch.uint8: U8_SENTINEL}[dtype]


def assert_guard(buf, numel, what):
    """The elements after the first `numel` are still the sentinel; none of the first `numel` is (every one written)."""
    s = _sentinel_bits(buf.dtype)
    bits = _bits(buf)
    over = int((bits[numel:] != s).sum())
    assert over == 0, f"{what}: {over} elements written past the end"
    if buf.dtype != torch.uint8:  # a position byte can legitimately hold any value 0..3, but never 0xAB
        unwritten = int((bits[:numel] == s).sum())
    else:
        unwritten = int((bits[:numel] > 3).sum())
    assert unwritten == 0, f"{what}: {unwritten} elements left unwritten"


def canvas2(n, h, w, c, device="cuda"):
    """A concat-style [n, h, w, 2c] bf16 sentinel buffer and its left half (pixel pitch 2c)."""
    cv = sentinel_like(n * h * w * 2 * c, BF16, device).view(n, h, w, 2 * c)
    return cv, cv[..., :c]


def assert_right_half(cv, what):
    """The right half of a canvas2 buffer is still the sentinel, and its left half holds no sentinel (all written)."""
    c = cv.shape[-1] // 2
    bits = _bits(cv)
    changed = int((bits[..., c:] != BF16_SENTINEL).sum())
    assert changed == 0, f"{what}: {changed} elements of the other half were written"
    unwritten = int((bits[..., :c] == BF16_SENTINEL).sum())
    assert unwritten == 0, f"{what}: {unwritten} target elements left unwritten"
