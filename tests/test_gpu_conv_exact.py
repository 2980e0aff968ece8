"""-m gpu: every tensor-core convolution instantiation, forced one at a time, bit-exact against an fp64 reference.

Operands are small integers (tests/conv_check.py), so each kernel's fp32 accumulator holds the exact value and every bf16
output must equal bf16_rne(exact) bit for bit; weight gradients and statistics must equal the exact value. Each case of the
table names the instantiation it expects; `launched_kernels` asserts that exactly that one ran. Inputs are channel slices
of NaN canvases with a NaN guard image; outputs and statistics rows go to sentinel canvases that must stay intact outside
the target. The 3x3 shapes cover a one-pixel image, images smaller than a tile with W % 8 != 0, a single tile (the second
CTA of a pair gets the out-of-range tile), an odd tile count, ragged tiles in both geometries, a deep persistent schedule
(depth derived from conv3x3_stat_rows and asserted) and more than one channel slice (ntiles_n > 1).

The table's kernels are exactly the tensor-core instantiations compiled into libb200unet.so (checked against the library's
machine code). The module skips when B200UNET_NO_WGRAD_SWAP or B200UNET_NO_BNRED is set: both are read once per process
and change which kernel a case runs, so the expected kernels would be wrong."""
import collections
import math
import os
import re
import shutil
import subprocess
import zlib
from dataclasses import dataclass, field

import pytest
import torch

import conv_check as C

pytestmark = pytest.mark.gpu

_ENV = [v for v in ("B200UNET_NO_WGRAD_SWAP", "B200UNET_NO_BNRED") if v in os.environ]
if _ENV:
    pytest.skip(f"{', '.join(_ENV)} set: the kernel choice it controls is fixed per process, the expected kernels would be wrong",
                allow_module_level=True)

TC_FAMILIES = ("conv3_res_kernel", "conv3_res2_kernel", "conv3_pair_kernel", "igemm_kernel", "wgrad_kernel", "wgrad_swap_kernel",
               "wgrad_swap3_kernel")
RES, RES2, PAIR, IGEMM = (1, 0, 0), (1, 1, 0), (0, 0, 1), (0, 0, 0)   # b200unet_set_kernel_choice(resident, pairs, streaming)
MIN_DEPTH = 5


@dataclass
class Case:
    id: str
    op: str
    kernel: str
    choice: tuple
    nhw: tuple
    cin: int
    cout: int
    regime: str = C.SPARSE
    extra: dict = field(default_factory=dict)


def _res(bn, kb, na, ob, taps, kind=0, cin=0, bnred=False):
    return f"conv3_res_kernel<{bn}, {kb}, {na}, {ob}, {taps}, {kind}, {cin}, {'true' if bnred else 'false'}>"


SHAPES = [(1, 1, 1), (1, 3, 5), (2, 4, 3), (1, 16, 8), (3, 16, 24), (2, 20, 12)]
DEEP = (4, 160, 160)
# (kernel, choice, Cin, Cout, (Cin, Cout) with more than one channel slice, persistent)
CONV3 = [
    (_res(64, 1, 4, 2, 9), RES, 64, 64, (64, 192), True),
    (_res(128, 1, 2, 1, 9), RES, 64, 128, (64, 256), True),
    (_res(64, 2, 2, 2, 9), RES, 128, 64, (128, 192), True),
    ("conv3_res2_kernel<64, 1, 4, 2>", RES2, 64, 64, (64, 192), True),
    ("conv3_res2_kernel<128, 1, 3, 2>", RES2, 64, 128, (64, 256), True),
    ("conv3_res2_kernel<64, 2, 4, 2>", RES2, 128, 64, (128, 192), True),
    ("conv3_res2_kernel<128, 2, 2, 1>", RES2, 128, 128, (128, 256), True),
    ("conv3_pair_kernel<256, 2, 6, 1>", PAIR, 256, 256, (256, 512), True),
    ("conv3_pair_kernel<128, 3, 8, 2>", PAIR, 256, 128, (384, 384), True),
    ("igemm_kernel<0, 128, 2, 4>", IGEMM, 64, 128, (192, 256), False),   # Cin = 192: only igemm takes it
    ("igemm_kernel<0, 64, 3, 6>", IGEMM, 64, 64, (64, 192), False),
]


def _short(kernel):
    return kernel.replace("_kernel", "").replace(" ", "")


def _cases():
    out = []
    for kern, choice, cin, cout, (cin2, cout2), persistent in CONV3:
        k = _short(kern)
        for s in SHAPES + [DEEP]:
            out.append(Case(f"fprop-{k}-{'x'.join(map(str, s))}", "conv3", kern, choice, s, cin, cout,
                            extra={"deep": persistent and s == DEEP}))
        for s in ((3, 16, 24), DEEP):
            out.append(Case(f"fprop-dense-{k}-{'x'.join(map(str, s))}", "conv3", kern, choice, s, cin, cout, C.DENSE,
                            extra={"deep": persistent and s == DEEP}))
        out.append(Case(f"fprop-slices-{k}-{cin2}to{cout2}", "conv3", kern, choice, (3, 16, 24), cin2, cout2))
        out.append(Case(f"dgrad-{k}", "conv3_dgrad", kern, choice, (2, 20, 12), cin, cout))
        out.append(Case(f"dgrad-dense-{k}", "conv3_dgrad", kern, choice, (1, 3, 5), cin, cout, C.DENSE))
        out.append(Case(f"eval-dense-{k}", "conv3_eval", kern, choice, (2, 20, 12), cin, cout, C.DENSE))
    bnred = _res(64, 1, 3, 2, 9, bnred=True)
    for s in ((1, 3, 5), (3, 16, 24), (2, 20, 12), DEEP):
        out.append(Case(f"bnred-{'x'.join(map(str, s))}", "bnred", bnred, RES, s, 64, 64, extra={"deep": s == DEEP}))
    # ConvTranspose2d(2, 2): fprop resident (RES_UP = 1), dgrad resident (RES_GATHER = 2), igemm MODE_UP = 1 / MODE_GATHER4 = 2
    up = [(_res(256, 2, 4, 1, 1, 1), RES, 128), (_res(128, 4, 4, 1, 1, 1), RES, 256), (_res(128, 8, 3, 1, 1, 1), RES, 512),
          ("igemm_kernel<1, 256, 3, 4>", RES, 1024), ("igemm_kernel<1, 256, 3, 4>", IGEMM, 128)]
    for kern, choice, cin in up:
        for s, regime in (((1, 1, 1), C.SPARSE), ((2, 5, 9), C.SPARSE), ((3, 20, 12), C.DENSE)):
            out.append(Case(f"convt-{regime}-{_short(kern)}-cin{cin}-{'x'.join(map(str, s))}", "convt", kern, choice, s, cin,
                            cin // 2, regime))
    for s in ((1, 3, 5), (3, 20, 12)):
        out.append(Case(f"convt-stats-cin256-{'x'.join(map(str, s))}", "convt_stats", "igemm_kernel<1, 256, 3, 4>", RES, s, 256,
                        128))
    # (kernel, choice, Cin, Cup); Cin = 192 is not a multiple of 128, so igemm takes 64 columns per tile
    gather = [(_res(128, 4, 4, 1, 1, 2), RES, 128, 64), (_res(128, 8, 3, 1, 1, 2), RES, 256, 128),
              ("igemm_kernel<2, 128, 2, 4>", RES, 512, 256), ("igemm_kernel<2, 128, 2, 4>", IGEMM, 128, 64),
              ("igemm_kernel<2, 64, 3, 6>", RES, 192, 64)]
    for kern, choice, cin, cup in gather:
        cups = "" if cup == cin // 2 else f"-cup{cup}"
        for s, regime in (((1, 1, 1), C.SPARSE), ((2, 5, 9), C.SPARSE), ((3, 20, 12), C.DENSE)):
            out.append(Case(f"convt-dgrad-{regime}-{_short(kern)}-cin{cin}{cups}-{'x'.join(map(str, s))}", "convt_dgrad", kern,
                            choice, s, cin, cup, regime))
    # 1x1 convolutions: igemm MODE_UP with bias + statistics, the resident K = 64 kernel (TAPS = 1) with and without statistics
    for kern, cout in (("igemm_kernel<1, 128, 2, 4>", 128), ("igemm_kernel<1, 64, 3, 6>", 64)):
        for s, regime in (((2, 5, 9), C.SPARSE), ((3, 20, 12), C.SPARSE), ((2, 20, 12), C.DENSE)):
            out.append(Case(f"conv1x1-{regime}-{_short(kern)}-{'x'.join(map(str, s))}", "conv1x1", kern, RES, s, 128, cout,
                            regime))
    c64 = _res(64, 1, 4, 2, 1)
    for s, regime in (((1, 3, 5), C.SPARSE), ((3, 20, 12), C.DENSE), ((4, 100, 60), C.SPARSE)):
        out.append(Case(f"conv1x1-c64-{regime}-{'x'.join(map(str, s))}", "conv1x1_c64", c64, RES, s, 64, 128, regime))
        out.append(Case(f"conv1x1-c64-stats-{regime}-{'x'.join(map(str, s))}", "conv1x1_c64_stats", c64, RES, s, 64, 64, regime))
    # first layer (RES_FIRST = 3, CIN 1..7): fused im2col from the fp32 NCHW input
    for cin in range(1, 8):
        kern = _res(64, 1, 4, 2, 1, 3, cin)
        out.append(Case(f"first-cin{cin}", "first", kern, RES, (2, 20, 12), cin, 64))
        out.append(Case(f"first-dense-cin{cin}", "first", kern, RES, (3, 37, 29), cin, 64, C.DENSE))
    out.append(Case("first-eval-dense-cin3", "first_eval", _res(64, 1, 4, 2, 1, 3, 3), RES, (2, 20, 12), 3, 64, C.DENSE))
    # weight gradients (KIND_CONV3 = 0, KIND_UP = 1, KIND_PLAIN = 2, KIND_FIRST = 3): 91 pixel tiles, split unevenly
    wg = (1, 100, 100)
    for kern, cin, cout in (("wgrad_kernel<0, 128, 0>", 128, 128), ("wgrad_kernel<0, 64, 0>", 64, 128),
                            ("wgrad_swap_kernel<2>", 128, 64), ("wgrad_swap3_kernel", 64, 64)):
        for regime in (C.SPARSE, C.DENSE):
            out.append(Case(f"wgrad3-{regime}-{_short(kern)}-{cin}to{cout}", "wgrad3", kern, RES, wg, cin, cout, regime))
    out.append(Case("wgrad3-small-wgrad_swap3", "wgrad3", "wgrad_swap3_kernel", RES, (2, 4, 3), 64, 64))
    for regime in (C.SPARSE, C.DENSE):
        out.append(Case(f"wgrad-up-{regime}", "wgrad_up", "wgrad_kernel<1, 64, 0>", RES, wg, 128, 64, regime))
        out.append(Case(f"wgrad-1x1-{regime}", "wgrad_1x1", "wgrad_kernel<2, 64, 0>", RES, wg, 64, 128, regime))
    for cin in range(1, 8):
        out.append(Case(f"wgrad-first-cin{cin}", "wgrad_first", f"wgrad_kernel<3, 64, {cin}>", RES, wg, cin, 64,
                        C.DENSE if cin % 2 else C.SPARSE))
    return out


CASES = _cases()
RAN = collections.defaultdict(list)       # kernel -> ids of the cases that launched it
CASES_RUN = set()
DEPTH = {}                                # kernel -> deepest schedule reached (tiles or tile pairs per persistent CTA)


@pytest.fixture(scope="module")
def ops():
    import unet_torch_b200  # noqa: F401
    from unet_torch_b200 import ops as _ops

    return _ops


@pytest.fixture
def kernel_choice():
    """Forces b200unet_set_kernel_choice for the test; automatic dispatch is restored afterwards."""
    from unet_torch_b200 import _lib

    try:
        yield lambda choice: _lib.call("b200unet_set_kernel_choice", *choice)
    finally:
        _lib.call("b200unet_set_kernel_choice", -1, -1, -1)


def _launch(case, fn):
    names = [n for n in C.launched_kernels(fn) if n.split("<")[0] in TC_FAMILIES]
    CASES_RUN.add(case.id)
    for name in names:
        RAN[name].append(case.id)
    assert names == [case.kernel], f"{case.id}: expected one launch of {case.kernel}, the profiler saw {names}"


def _gen(case):
    return torch.Generator().manual_seed(zlib.crc32(case.id.encode()))


def _dev(t):
    return t.cuda()


def _scale_shift(gen, c, y):
    """Dyadic per-channel scale (+-k/4) and shift (multiples of 1/2 around the outputs' magnitude): the folded affine is exact in
    fp32, so the only rounding is the final bf16 one."""
    sc = torch.randint(1, 9, (c,), generator=gen).to(C.F64) / 4 * (torch.randint(0, 2, (c,), generator=gen) * 2 - 1)
    mag = int(y.abs().mean()) + 1
    sh = torch.randint(-mag, mag + 1, (c,), generator=gen).to(C.F64) / 2
    return sc, sh


def _reduced(ops, st, rows, c):
    sums = torch.empty(2 * c, dtype=torch.float64, device="cuda")
    ops.bn_reduce_partials(st, rows, c, sums)
    return sums.cpu()


def _depth(case, ops, n, h, w, cin, cout):
    """Tiles (conv3_res) or tile pairs (pair kernels) per persistent CTA, from the statistics-row count (= CTAs per slice)."""
    rows = ops.conv3x3_stat_rows(n, h, w, cin, cout)
    tiles = n * math.ceil(h / 16) * math.ceil(w / 8)
    paired = case.kernel.startswith(("conv3_res2", "conv3_pair"))
    workers = rows // 2 if paired else rows
    return math.ceil(math.ceil(tiles / 2) / workers) if paired else math.ceil(tiles / workers)


def run_conv3(case, ops, dgrad=False, evaluate=False):
    n, h, w = case.nhw
    gen = _gen(case)
    cin, cout = case.cin, case.cout
    k = 9 * cin
    x = C.operand((n, cin, h, w), case.regime, k, gen)
    if dgrad:   # the kernel's (Cin, Cout) are the forward conv's (Cout, Cin): wd is the rotated operand of w [Cin_k, Cout_k]
        wt = C.operand((cin, cout, 3, 3), case.regime, k, gen, sparse_input=False)
        _, wop = ops.prep_conv3x3_weight(_dev(wt.float()))
        y = C.conv3x3_dgrad(_dev(x), _dev(wt)).cpu()
        y_abs = C.conv3x3_dgrad(_dev(x.abs()), _dev(wt.abs())).cpu()
    else:
        wt = C.operand((cout, cin, 3, 3), case.regime, k, gen, sparse_input=False)
        wop, _ = ops.prep_conv3x3_weight(_dev(wt.float()), want_dgrad=False)
        y = C.conv3x3(_dev(x), _dev(wt)).cpu()
        y_abs = C.conv3x3(_dev(x.abs()), _dev(wt.abs())).cpu()
    C.check_regime(case.regime, y, y_abs)
    _, xs = C.input_canvas(C.nhwc(x))
    ycan, ys = C.bf16_canvas(n, h, w, cout)
    if case.extra.get("deep"):
        d = _depth(case, ops, n, h, w, cin, cout)
        assert d >= MIN_DEPTH, f"{case.id}: the schedule is only {d} deep"
        DEPTH[case.kernel] = max(DEPTH.get(case.kernel, 0), d)
    if evaluate:
        sc, sh = _scale_shift(gen, cout, y)
        scd, shd = _dev(sc.float()), _dev(sh.float())
        _launch(case, lambda: ops.conv3x3_bn_relu(xs, wop, scd, shd, ys))
        want = C.bf16_rne(C.bn_relu_eval(y, sc, sh))
    elif dgrad:
        _launch(case, lambda: ops.conv3x3(xs, wop, ys))
        want = C.bf16_rne(y)
    else:
        rows = ops.conv3x3_stat_rows(n, h, w, cin, cout)
        st = C.stats_buffer(rows, cout)
        _launch(case, lambda: ops.conv3x3(xs, wop, ys, st))
        torch.cuda.synchronize()
        C.assert_stats_rows(st, rows, cout)
        if case.regime == C.SPARSE:
            s1, s2 = C.channel_sums(y)
            C.assert_exact(_reduced(ops, st, rows, cout), torch.cat([s1, s2]), "statistics (sum y, sum y^2)")
        want = C.bf16_rne(y)
    torch.cuda.synchronize()
    C.assert_canvas_intact(ycan, n, cout)
    C.assert_exact(ys.cpu(), C.nhwc(want), case.id)


def run_bnred(case, ops):
    from unet_torch_b200 import _lib

    n, h, w = case.nhw
    c = 64
    gen = _gen(case)
    dy = C.operand((n, c, h, w), case.regime, 9 * c, gen)
    wt = C.operand((c, c, 3, 3), case.regime, 9 * c, gen, sparse_input=False)
    _, wd = ops.prep_conv3x3_weight(_dev(wt.float()))
    dx = C.conv3x3_dgrad(_dev(dy), _dev(wt)).cpu()
    C.check_regime(case.regime, dx, C.conv3x3_dgrad(_dev(dy.abs()), _dev(wt.abs())).cpu())
    y_bn = torch.randint(-6, 7, (n, c, h, w), generator=gen).to(C.F64)       # the consumer BatchNorm's input
    sc, sh = _scale_shift(gen, c, y_bn)
    mean = torch.randint(-8, 9, (c,), generator=gen).to(C.F64) / 8
    rstd = 2.0 ** torch.randint(-2, 2, (c,), generator=gen).to(C.F64)
    _, dys = C.input_canvas(C.nhwc(dy))
    _, ybs = C.input_canvas(C.nhwc(y_bn))
    dxcan, dxs = C.bf16_canvas(n, h, w, c)
    rows = _lib.query("b200unet_conv3x3_dgrad_bnred_rows", n, h, w, c, c)
    assert rows == ops.conv3x3_stat_rows(n, h, w, c, c) > 0
    if case.extra.get("deep"):
        d = _depth(case, ops, n, h, w, c, c)
        assert d >= MIN_DEPTH, f"{case.id}: the schedule is only {d} deep"
        DEPTH[case.kernel] = max(DEPTH.get(case.kernel, 0), d)
    st = C.stats_buffer(rows, c)
    aff = [_dev(t.float()) for t in (sc, sh, mean, rstd)]
    stream = torch.cuda.current_stream().cuda_stream
    _launch(case, lambda: _lib.call("b200unet_conv3x3_igemm_bnred", dys.data_ptr(), dys.stride(2), wd.data_ptr(), dxs.data_ptr(),
                                    dxs.stride(2), ybs.data_ptr(), ybs.stride(2), *(t.data_ptr() for t in aff), st.data_ptr(),
                                    n, h, w, c, c, stream))
    torch.cuda.synchronize()
    C.assert_canvas_intact(dxcan, n, c, "dx")
    C.assert_exact(dxs.cpu(), C.nhwc(C.bf16_rne(dx)), "dx")
    C.assert_stats_rows(st, rows, c, "backward partial rows")
    s1, s2 = C.bn_backward_sums(dx, y_bn, sc, sh, mean, rstd)
    C.assert_exact(_reduced(ops, st, rows, c), torch.cat([s1, s2]), "(sum da, sum da * xhat)")


def run_convt(case, ops, stats=False):
    n, h, w = case.nhw
    cin, cup = case.cin, case.cout
    gen = _gen(case)
    x = C.operand((n, cin, h, w), case.regime, cin, gen)
    wt = C.operand((cin, cup, 2, 2), case.regime, cin, gen, sparse_input=False)
    bias = torch.randint(-4, 5, (cup,), generator=gen).to(C.F64)
    y = C.convt2x2(_dev(x), _dev(wt), _dev(bias)).cpu()
    C.check_regime(case.regime, y, C.convt2x2(_dev(x.abs()), _dev(wt.abs()), _dev(bias.abs())).cpu())
    wf, _ = ops.prep_convt2x2_weight(_dev(wt.float()))
    _, xs = C.input_canvas(C.nhwc(x))
    ycan, ys = C.bf16_canvas(n, 2 * h, 2 * w, cup)
    bd = _dev(bias.float())
    if stats:
        rows = ops.convt2x2_stat_rows(n, h, w)
        st = C.stats_buffer(rows, cup)
        _launch(case, lambda: ops.convt2x2_stats(xs, wf, bd, ys, st, cup))
        torch.cuda.synchronize()
        C.assert_stats_rows(st, rows, cup)
        s1, s2 = C.channel_sums(y)
        C.assert_exact(_reduced(ops, st, rows, cup), torch.cat([s1, s2]), "statistics (sum y, sum y^2)")
    else:
        _launch(case, lambda: ops.convt2x2(xs, wf, bd, ys))
    torch.cuda.synchronize()
    C.assert_canvas_intact(ycan, n, cup)
    C.assert_exact(ys.cpu(), C.nhwc(C.bf16_rne(y)), case.id)


def run_convt_dgrad(case, ops):
    n, h, w = case.nhw
    cin, cup = case.cin, case.cout
    gen = _gen(case)
    du = C.operand((n, cup, 2 * h, 2 * w), case.regime, 4 * cup, gen)
    wt = C.operand((cin, cup, 2, 2), case.regime, 4 * cup, gen, sparse_input=False)
    dx = C.convt2x2_dgrad(_dev(du), _dev(wt)).cpu()
    C.check_regime(case.regime, dx, C.convt2x2_dgrad(_dev(du.abs()), _dev(wt.abs())).cpu())
    _, wd = ops.prep_convt2x2_weight(_dev(wt.float()))
    _, dus = C.input_canvas(C.nhwc(du))
    dxcan, dxs = C.bf16_canvas(n, h, w, cin)
    _launch(case, lambda: ops.convt2x2_dgrad(dus, wd, dxs))
    torch.cuda.synchronize()
    C.assert_canvas_intact(dxcan, n, cin)
    C.assert_exact(dxs.cpu(), C.nhwc(C.bf16_rne(dx)), case.id)


def run_conv1x1(case, ops, bias=True, stats=True, c64_entry=False):
    n, h, w = case.nhw
    cin, cout = case.cin, case.cout
    gen = _gen(case)
    x = C.operand((n, cin, h, w), case.regime, cin, gen)
    wt = C.operand((cout, cin), case.regime, cin, gen, sparse_input=False)
    b = torch.randint(-4, 5, (cout,), generator=gen).to(C.F64) if bias else None
    y = C.conv1x1(_dev(x), _dev(wt), None if b is None else _dev(b)).cpu()
    C.check_regime(case.regime, y, C.conv1x1(_dev(x.abs()), _dev(wt.abs()), None if b is None else _dev(b.abs())).cpu())
    _, xs = C.input_canvas(C.nhwc(x))
    ycan, ys = C.bf16_canvas(n, h, w, cout)
    wop = _dev(wt.to(C.BF16)).contiguous()
    st, rows = None, 0
    if stats:
        rows = ops.conv1x1_c64_stat_rows(n, h, w, cout) if c64_entry else ops.conv1x1_stat_rows(n, h, w)
        st = C.stats_buffer(rows, cout)
    if c64_entry:
        _launch(case, lambda: ops.conv1x1_c64(xs, wop, ys, st))
    else:
        bd = None if b is None else _dev(b.float())
        _launch(case, lambda: ops.conv1x1(xs, wop, bd, ys, st))
    torch.cuda.synchronize()
    if stats:
        C.assert_stats_rows(st, rows, cout)
        if case.regime == C.SPARSE:
            s1, s2 = C.channel_sums(y)
            C.assert_exact(_reduced(ops, st, rows, cout), torch.cat([s1, s2]), "statistics (sum y, sum y^2)")
    C.assert_canvas_intact(ycan, n, cout)
    C.assert_exact(ys.cpu(), C.nhwc(C.bf16_rne(y)), case.id)


def _nchw_with_guard(x):
    """fp32 NCHW input followed by one NaN image (the first layer reads a contiguous NCHW tensor, not a channel slice)."""
    buf = torch.full((x.shape[0] + 1, *x.shape[1:]), float("nan"), device="cuda")
    buf[: x.shape[0]] = _dev(x.float())
    return buf[: x.shape[0]]


def run_first(case, ops, evaluate=False):
    n, h, w = case.nhw
    cin, cout = case.cin, case.cout
    gen = _gen(case)
    x = C.operand((n, cin, h, w), case.regime, 9 * cin, gen)
    wt = C.operand((cout, cin, 3, 3), case.regime, 9 * cin, gen, sparse_input=False)
    y = C.conv3x3(_dev(x), _dev(wt)).cpu()
    C.check_regime(case.regime, y, C.conv3x3(_dev(x.abs()), _dev(wt.abs())).cpu())
    w1 = ops.prep_first_weight(_dev(wt.float()))
    xin = _nchw_with_guard(x)
    ycan, ys = C.bf16_canvas(n, h, w, cout)
    if evaluate:
        sc, sh = _scale_shift(gen, cout, y)
        scd, shd = _dev(sc.float()), _dev(sh.float())
        _launch(case, lambda: ops.conv3x3_first_tc_bn_relu(xin, w1, scd, shd, ys))
        want = C.bf16_rne(C.bn_relu_eval(y, sc, sh))
    else:
        rows = ops.conv1x1_c64_stat_rows(n, h, w, cout)
        st = C.stats_buffer(rows, cout)
        _launch(case, lambda: ops.conv3x3_first_tc(xin, w1, ys, st))
        torch.cuda.synchronize()
        C.assert_stats_rows(st, rows, cout)
        if case.regime == C.SPARSE:
            s1, s2 = C.channel_sums(y)
            C.assert_exact(_reduced(ops, st, rows, cout), torch.cat([s1, s2]), "statistics (sum y, sum y^2)")
        want = C.bf16_rne(y)
    torch.cuda.synchronize()
    C.assert_canvas_intact(ycan, n, cout)
    C.assert_exact(ys.cpu(), C.nhwc(want), case.id)


def _assert_uneven_split(case, ws_floats, per_split, tiles):
    z = ws_floats // per_split
    assert ws_floats == z * per_split and z > 1 and tiles % z != 0, f"{case.id}: {tiles} pixel tiles in {z} splits"


def run_wgrad(case, ops):
    from unet_torch_b200 import _lib

    n, h, w = case.nhw
    cin, cout = case.cin, case.cout
    gen = _gen(case)
    kind = case.op
    tiles = n * math.ceil(h / 8) * math.ceil(w / 16)
    if kind == "wgrad_up":
        k = n * h * w
        x = C.operand((n, cin, h, w), case.regime, k, gen)
        dy = C.operand((n, cout, 2 * h, 2 * w), case.regime, k, gen, sparse_input=False)
        want = C.convt2x2_wgrad(_dev(x), _dev(dy)).cpu()
        want_abs = C.convt2x2_wgrad(_dev(x.abs()), _dev(dy.abs())).cpu()
    else:
        k = n * h * w
        x = C.operand((n, cin, h, w), case.regime, k, gen)
        dy = C.operand((n, cout, h, w), case.regime, k, gen, sparse_input=False)
        ref = C.conv1x1_wgrad if kind == "wgrad_1x1" else C.conv3x3_wgrad
        want = ref(_dev(x), _dev(dy)).cpu()
        want_abs = ref(_dev(x.abs()), _dev(dy.abs())).cpu()
    C.check_regime(case.regime, want, want_abs, rounded_out=False)
    _, dys = C.input_canvas(C.nhwc(dy))
    dw = C.f32_sentinel(want.numel()).view(want.shape)
    if kind == "wgrad_first":
        xin = _nchw_with_guard(x)
        ws = _lib.query("b200unet_conv3x3_first_tc_wgrad_workspace_floats", n, h, w, cout)
        _assert_uneven_split(case, ws, cout * 64, tiles)
        _launch(case, lambda: ops.conv3x3_first_tc_wgrad(xin, dys, dw))
    else:
        _, xs = C.input_canvas(C.nhwc(x))
        if kind == "wgrad3":
            ws = _lib.query("b200unet_conv3x3_wgrad_workspace_floats", n, h, w, cin, cout)
            if h * w > 100:
                _assert_uneven_split(case, ws, cout * 9 * cin, tiles)
            _launch(case, lambda: ops.conv3x3_wgrad(xs, dys, dw))
        elif kind == "wgrad_up":
            ws = _lib.query("b200unet_convt2x2_wgrad_workspace_floats", n, h, w, cin, cout)
            _assert_uneven_split(case, ws, cin * 4 * cout, tiles)
            _launch(case, lambda: ops.convt2x2_wgrad(xs, dys, dw))
        else:
            ws = _lib.query("b200unet_conv1x1_wgrad_workspace_floats", n, h, w, cin, cout)
            _assert_uneven_split(case, ws, cout * cin, tiles)
            _launch(case, lambda: ops.conv1x1_wgrad(xs, dys, dw))
    torch.cuda.synchronize()
    C.assert_exact(dw.cpu(), want, case.id)


RUNNERS = {
    "conv3": run_conv3,
    "conv3_dgrad": lambda c, o: run_conv3(c, o, dgrad=True),
    "conv3_eval": lambda c, o: run_conv3(c, o, evaluate=True),
    "bnred": run_bnred,
    "convt": run_convt,
    "convt_stats": lambda c, o: run_convt(c, o, stats=True),
    "convt_dgrad": run_convt_dgrad,
    "conv1x1": run_conv1x1,
    "conv1x1_c64": lambda c, o: run_conv1x1(c, o, bias=False, stats=False),
    "conv1x1_c64_stats": lambda c, o: run_conv1x1(c, o, bias=False, stats=True, c64_entry=True),
    "first": run_first,
    "first_eval": lambda c, o: run_first(c, o, evaluate=True),
    "wgrad3": run_wgrad,
    "wgrad_up": run_wgrad,
    "wgrad_1x1": run_wgrad,
    "wgrad_first": run_wgrad,
}


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_exact(ops, kernel_choice, case):
    kernel_choice(case.choice)
    RUNNERS[case.op](case, ops)


def _cuda_tool(name):
    for cand in (shutil.which(name), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)):
        if cand and os.path.exists(cand):
            return cand
    return None


def _profiler_spelling(demangled):
    """'void <unnamed>::conv3_res_kernel<(int)64, ..., (bool)1>(<unnamed>::ResArgs)' -> 'conv3_res_kernel<64, ..., true>'."""
    s = re.sub(r"\(bool\)([01])", lambda m: "true" if m.group(1) == "1" else "false", demangled)
    s = re.sub(r"\(int\)(-?\d+)", r"\1", s)
    return C.kernel_name(s.replace("<unnamed>::", ""))


def test_library_instantiations_are_the_table():
    """Every tensor-core instantiation compiled into libb200unet.so has a case in the table, and every kernel the table names
    is compiled: a new instantiation without a case fails here."""
    from unet_torch_b200 import _lib

    cuobjdump, cufilt = _cuda_tool("cuobjdump"), _cuda_tool("cu++filt")
    if cuobjdump is None or cufilt is None:
        pytest.skip("cuobjdump / cu++filt not found")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = re.findall(r"Function : (\S+)", sass)
    demangled = subprocess.run([cufilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(demangled) == len(mangled)
    built = {n for n in map(_profiler_spelling, demangled) if n.split("<")[0] in TC_FAMILIES}
    table = {c.kernel for c in CASES}
    assert built == table, f"compiled without a case: {sorted(built - table)}; in the table but not compiled: {sorted(table - built)}"


def test_every_instantiation_in_the_table_ran():
    """Last in the module: the kernels launched across the table are exactly the table's instantiations."""
    if len(CASES_RUN) < len(CASES):
        pytest.skip(f"only {len(CASES_RUN)} of {len(CASES)} cases ran (a selection, or failures): run the whole module")
    want = {c.kernel for c in CASES}
    for kern in sorted(want):
        print(f"{kern}: {len(RAN[kern])} cases, deepest schedule {DEPTH.get(kern, '-')}; e.g. {RAN[kern][:3]}")
    assert set(RAN) == want
