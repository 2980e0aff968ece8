"""-m gpu: UNet(dropout=True) on the tensor-core engine (csrc/dropout.cu, DESIGN.md §4).

* the dropout kernel bit for bit against oracle/philox.py: channel slices of sentinel canvases, ragged pixel counts, slices
  starting at e % 4 != 0, p from 0.1 to 1, and the per-channel sums of the ConvTranspose2d bias gradient against fp64;
* mask statistics over >= 10^7 elements;
* the network against the fp64 oracle fed with the engine's own masks, judged against the same engine's dropout-off error;
  every traced dropout operator against the host mask bit for bit;
* nothing changes where dropout does nothing (eval, p = 0); reproducibility under torch.manual_seed; CUDA-graph replays draw
  new masks; the config-2 full-size step keeps its gradient invariants and trains.
"""
import numpy as np
import pytest
import torch

import conv_check as C
from gpu_util import rel_l2
from oracle import philox as PX
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
SEED = 0x0123456789ABCDEF


def _seed(v=SEED):
    return torch.tensor([v], dtype=torch.int64, device="cuda")


def _host_dropout(before, seed, site, p, c_site=None, c_lo=0):
    """What the kernel must write for `before` (NHWC, channels [c_lo, c_lo + C) of a site with c_site channels)."""
    n, h, w, c = before.shape
    keep = torch.from_numpy(PX.keep_mask(seed, site, (n, h, w, c if c_site is None else c_site), p, c_lo, c))
    _, scale = PX.threshold_scale(p)
    out = (before.float().cpu() * np.float32(scale)).to(BF16)
    return torch.where(keep, out, torch.zeros((), dtype=BF16))


def _bits(t):
    return t.contiguous().view(torch.int16).cpu()


# (n, h, w, c_site, c_lo, nc, site, sum_lo or None)
KERNEL_CASES = [
    (2, 7, 9, 64, 0, 64, 0, None),          # ragged pixel count, whole site
    (2, 16, 16, 128, 0, 128, 4, 64),        # a concat site: both halves, sums over the upsampled half
    (1, 5, 13, 200, 40, 96, 6, 8),          # channel slice in the middle of a wider site
    (3, 3, 11, 26, 2, 16, 3, 0),            # e % 4 != 0 at slice starts (C_site = 26, c_lo = 2)
    (1, 9, 7, 2048, 0, 2048, 7, 1024),      # 256 groups per pixel: one pixel per block row
    (1, 3, 5, 4096, 1024, 3072, 5, None),   # more groups than threads: each thread loops over groups
]


@pytest.mark.parametrize("p", [0.1, 0.3, 0.5, 0.999, 1.0])
@pytest.mark.parametrize("case", KERNEL_CASES, ids=[f"{c[0]}x{c[1]}x{c[2]}_site{c[6]}_C{c[3]}_lo{c[4]}_n{c[5]}" for c in KERNEL_CASES])
def test_kernel_bit_exact(case, p):
    from unet_torch_b200 import ops

    n, h, w, c_site, c_lo, nc, site, sum_lo = case
    gen = torch.Generator().manual_seed(n * 10007 + c_site + 97 * site)
    x = torch.randn(n, h, w, nc, generator=gen).to(BF16)
    canvas, sl = C.input_canvas(x)
    sums = None
    if sum_lo is not None:
        out = C.f32_sentinel(nc - sum_lo + 1)
        sums = (sum_lo, out[: nc - sum_lo])
    ops.dropout_mul(sl, site, _seed(), p, c_site=c_site, c_lo=c_lo, sums=sums)
    torch.cuda.synchronize()
    C.assert_canvas_intact(canvas, n, nc, "dropout_mul")
    want = _host_dropout(x, SEED, site, p, c_site, c_lo)
    assert torch.equal(_bits(sl), _bits(want)), f"{int((_bits(sl) != _bits(want)).sum())} elements differ"
    if sums is not None:
        ref = want[..., sum_lo:].double().sum((0, 1, 2))
        mag = want[..., sum_lo:].double().abs().sum((0, 1, 2))
        got = sums[1].double().cpu()
        assert bool(((got - ref).abs() <= 1e-5 * mag + 1e-6).all()), float((got - ref).abs().max())
        assert int(out[-1:].view(torch.int32).item()) == C.F32_SENTINEL   # nothing past the sum range


def test_mask_statistics():
    from unet_torch_b200 import ops

    shape = (4, 64, 64, 640)              # 10.5 M elements
    p = 0.3
    ones = torch.ones(shape, dtype=BF16, device="cuda")
    masks = {}
    for site, seed in ((2, SEED), (3, SEED), (2, SEED + 1)):
        t = ones.clone()
        ops.dropout_mul(t, site, _seed(seed), p)
        masks[(site, seed)] = (t != 0).double()
    m = masks[(2, SEED)]
    n = m.numel()
    frac = float(m.mean())
    assert abs(frac - (1 - p)) < 5 * (p * (1 - p) / n) ** 0.5, frac

    def corr(a, b):
        a, b = a.flatten() - a.mean(), b.flatten() - b.mean()
        return float((a * b).sum() / (a.norm() * b.norm()))

    for name, a, b in (("channel", m[..., :-1], m[..., 1:]), ("pixel", m[:, :, :-1], m[:, :, 1:]),
                       ("row", m[:, :-1], m[:, 1:])):
        rho = corr(a, b)
        assert abs(rho) < 5 / a.numel() ** 0.5, (name, rho)
    for other in ((3, SEED), (2, SEED + 1)):
        agree = float((masks[other] == m).double().mean())
        want = p * p + (1 - p) * (1 - p)    # independent masks agree this often
        assert abs(agree - want) < 1e-3, (other, agree)
        assert abs(corr(masks[other], m)) < 5 / n ** 0.5


# ------------------------------------------------------------------------------------------------ network vs oracle
def _oracle_run(sd, x, y, masks):
    sd64 = {k: (v.double().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.double()
                if v.is_floating_point() else v) for k, v in sd.items()}
    logits, _ = O.unet_forward(sd64, x.double(), training=True, dropout_masks=masks)
    O.calc_loss(logits, y.double(), "dice_bce_mc", 2).backward()
    return logits.detach(), {k: v.grad for k, v in sd64.items() if isinstance(v, torch.Tensor) and v.requires_grad}


def _errors(net, sd, x, y, logits, grads, masks):
    """(logits error, {param: gradient error}) of one engine step against the fp64 oracle with the same masks."""
    want, want_grads = _oracle_run(sd, x, y, masks)
    return rel_l2(logits, want), {k: rel_l2(grads[k], want_grads[k]) for k in want_grads}


def _engine_step(net, x, y):
    """Forward + backward through the engine (the loss gradient from the fp64 loss at the device logits)."""
    eng = net._engine_for(x)
    eng.trace = []
    logits, saved = eng.forward(x, training=True, save=True)
    lg = logits.detach().cpu().double().requires_grad_(True)
    O.calc_loss(lg, y.double(), "dice_bce_mc", 2).backward()
    g = eng.backward(saved, lg.grad.float().cuda())
    trace, eng.trace = eng.trace, None
    named = dict(net.named_parameters())
    return logits, {k: g[p] for k, p in named.items()}, saved.drop, trace


def _judge(e_on, g_on, e_off, g_off, what):
    med_on, med_off = float(np.median(list(g_on.values()))), float(np.median(list(g_off.values())))
    worst = max(g_on, key=lambda k: g_on[k] / (1.5 * g_off[k] + 0.02))
    print(f"{what}: logits {e_on:.2e} (off {e_off:.2e}), median gradient {med_on:.2e} (off {med_off:.2e}), "
          f"tightest {worst} {g_on[worst]:.2e} (off {g_off[worst]:.2e})")
    assert e_on <= 1.5 * e_off
    assert med_on <= 1.5 * med_off
    for k in g_on:
        assert g_on[k] <= 1.5 * g_off[k] + 0.02, (k, g_on[k], g_off[k])


def _check_trace(trace, seed):
    ops = [kw for kind, kw in trace if kind == "dropout"]
    for kw in ops:
        want = _host_dropout(kw["before"], seed, kw["site"], kw["p"])
        assert torch.equal(_bits(kw["after"]), _bits(want)), (kw["site"], kw["backward"])
    return ops


@pytest.mark.parametrize("shape", [(2, 3, 64, 64), (1, 3, 48, 80)])
def test_network_against_oracle_with_the_engine_masks(shape):
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    n, _, h, w = shape
    torch.manual_seed(21)
    net = U.UNet(3, 2, 64, dropout=True, dropout_p=0.3)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().train()
    gen = torch.Generator().manual_seed(22)
    x = torch.randn(shape, generator=gen)
    y = torch.randint(0, 2, (n, h, w), generator=gen).float()
    assert isinstance(net._engine_for(x.cuda()), UNetEngine)
    holders = net._engine.drop
    # dropout off: the same engine, weights and input, every site at p = 0 (the dropout-off code path)
    for m in holders:
        m.p = 0.0
    logits, grads, drop, trace = _engine_step(net, x.cuda(), y)
    assert drop == (None, (0.0,) * 8) and not any(kind == "dropout" for kind, _ in trace)
    e_off, g_off = _errors(net, sd, x, y, logits, grads, None)
    for m in holders:
        m.p = 0.3
    logits, grads, (seed_t, ps), trace = _engine_step(net, x.cuda(), y)
    seed = int(seed_t.item())
    masks = PX.oracle_masks(seed, n, h, w, 64, ps)
    e_on, g_on = _errors(net, sd, x, y, logits, grads, masks)
    _judge(e_on, g_on, e_off, g_off, f"dropout {shape}")
    ops = _check_trace(trace, seed)
    assert sorted((kw["site"], kw["backward"]) for kw in ops) == sorted((s, b) for s in range(8) for b in (False, True))
    # the ConvTranspose2d bias gradient is the sum of the masked upsampled half of the concat gradient
    for kw in ops:
        if kw["backward"] and kw["site"] >= 4:
            up = getattr(net, f"up{kw['site'] - 3}").up
            c = up.bias.numel()
            ref = kw["after"][..., c:].double().sum((0, 1, 2)).cpu()
            assert rel_l2(grads[[k for k, p in net.named_parameters() if p is up.bias][0]], ref) < 1e-5


def _pair(width=64, p=0.5, seed=31):
    """A dropout network and a dropout=False network with the same weights (maxpool_conv.2 <-> maxpool_conv.1)."""
    import unet_torch_b200 as U

    torch.manual_seed(seed)
    a = U.UNet(3, 2, width, dropout=True, dropout_p=p)
    b = U.UNet(3, 2, width)
    b.load_state_dict({k.replace("maxpool_conv.2", "maxpool_conv.1"): v for k, v in a.state_dict().items()})
    return a.cuda(), b.cuda()


def _grads(net):
    return {k.replace("maxpool_conv.2", "maxpool_conv.1"): p.grad.clone() for k, p in net.named_parameters()}


def test_no_change_where_dropout_does_nothing():
    import unet_torch_b200 as U

    a, b = _pair()
    x = torch.randn(2, 3, 64, 96, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    y = (torch.rand(2, 64, 96, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)) > 0.5).float()
    with torch.no_grad():
        assert torch.equal(a.eval()(x), b.eval()(x))
    for m in a._engine.drop:
        m.p = 0.0
    a.train(), b.train()
    U.loss.CLASS_NUMBER = 2
    outs = []
    for net in (a, b):
        out = net(x)
        U.calc_loss(out, y, loss_type="dice_bce_mc").backward()
        outs.append((out.detach(), _grads(net)))
    assert torch.equal(outs[0][0], outs[1][0])
    for k, g in outs[1][1].items():
        assert torch.equal(outs[0][1][k], g), k


def test_reproducible_and_graph_replays_draw_new_masks():
    import unet_torch_b200 as U

    U.loss.CLASS_NUMBER = 2
    net, _ = _pair(p=0.3)
    sd = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(1, 3, 64, 64, generator=gen)
    y = torch.randint(0, 2, (1, 64, 64), generator=gen).float()
    xc, yc = x.cuda(), y.cuda()

    def step():
        net.zero_grad(set_to_none=True)
        out = net(xc)
        U.calc_loss(out, yc, loss_type="dice_bce_mc").backward()
        return out.detach().clone(), {k: p.grad.clone() for k, p in net.named_parameters()}

    runs = []
    for _ in range(2):
        torch.manual_seed(77)
        runs.append(step())
    assert torch.equal(runs[0][0], runs[1][0])
    assert all(torch.equal(runs[0][1][k], runs[1][1][k]) for k in runs[0][1])
    # dropout-off error of this engine at this size (the yardstick of every replay below)
    holders = net._engine.drop
    for m in holders:
        m.p = 0.0
    logits, grads, _, _ = _engine_step(net, xc, y)
    e_off, g_off = _errors(net, sd, x, y, logits, grads, None)
    for m in holders:
        m.p = 0.3
    net.enable_cuda_graphs(True)
    step()                                   # eager warm-up of this shape
    seeds = []
    for i in range(3):                       # capture + replay, then two replays
        logits, grads = step()
        st = next(iter(net._engine._graphs.values()))
        seed_t, ps = st.saved.drop
        seeds.append(int(seed_t.item()))
        e_on, g_on = _errors(net, sd, x, y, logits, grads, PX.oracle_masks(seeds[-1], 1, 64, 64, 64, ps))
        _judge(e_on, g_on, e_off, g_off, f"graph replay {i}")
    assert len(set(seeds)) == 3, seeds
    net.enable_cuda_graphs(False)


def test_config2_full_size_with_dropout():
    """16 x 3 x 512^2, p = 0.5: the gradient invariants of the dropout-off config-2 test (train-mode BatchNorm after every 3x3
    conv -> <dL/dW, W> = 0; softmax losses -> sum(d outc.bias) = 0), a bit-reproducible step under torch.manual_seed, and
    FusedSGD steps that lower the loss."""
    import unet_torch_b200 as U

    torch.manual_seed(35)
    net = U.UNet(3, 2, dropout=True, dropout_p=0.5).cuda().train()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    U.loss.CLASS_NUMBER = 2
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(16, 3, 512, 512, device="cuda", generator=g)
    f = torch.nn.functional.interpolate(torch.randn(16, 1, 32, 32, device="cuda", generator=g), size=(512, 512), mode="bilinear")
    y = (f[:, 0] > 0.2).float()

    def step():
        net.load_state_dict(sd)
        net.zero_grad(set_to_none=True)
        torch.manual_seed(5)
        out = net(x)
        loss = U.calc_loss(out, y, loss_type="dice_bce_mc")
        loss.backward()
        return float(loss.detach()), {k: p.grad.detach().clone() for k, p in net.named_parameters()}

    l1, g1 = step()
    l2, g2 = step()
    assert l1 == l2 and all(torch.equal(g1[k], g2[k]) for k in g1)
    params = dict(net.named_parameters())
    cos = {}
    for k, gr in g1.items():
        assert torch.isfinite(gr).all(), k
        if gr.dim() == 4 and gr.shape[-1] == 3:
            w = params[k].detach().double()
            cos[k] = float((gr.double() * w).sum() / (gr.double().norm() * w.norm() + 1e-300))
    assert len(cos) == 18
    worst_k = max(cos, key=lambda k: abs(cos[k]))
    db = g1["outc.conv.bias"].double()
    print(f"config2 dropout 0.5: loss {l1:.5f}, worst |cos(dW, W)| {abs(cos[worst_k]):.2e} ({worst_k}), "
          f"sum(d bias) / |d bias| = {float(db.sum() / db.norm()):.2e}")
    assert abs(cos[worst_k]) < 1e-2
    assert abs(float(db.sum())) < 1e-3 * float(db.norm())
    # a few FusedSGD steps on this batch lower the loss (each with its own masks)
    net.load_state_dict(sd)
    opt = U.FusedSGD(net, lr=0.01, momentum=0.9)
    losses = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    print(f"config2 dropout 0.5 FusedSGD losses {losses}")
    assert np.mean(losses[-2:]) < losses[0]
