"""-m gpu: BatchNorm module semantics of both engines over several training steps, against torch's recurrence.

Arm A sets momentum = 1.0 on every BatchNorm, so its buffers after step k are exactly that step's batch mean and unbiased
variance ((1-1)*rv + 1*v is exact in fp32). Arm B is the same network (same seed, same weights) with momentum m. Both run
K steps on the same inputs without an optimizer step, so they see identical batch statistics - their logits must be
bit-identical (the reductions are deterministic) - and every BatchNorm of arm B must follow torch's update
    running_k = (1 - f_k) * running_{k-1} + f_k * batch_k,   f_k = m, or 1 / num_batches_tracked for momentum=None,
computed here in fp32 from arm A's per-step values. Covers the attention gates' BatchNorms (psi: C = 1), CUDA-graph replay
(the cumulative factor changes at every replay), track_running_stats=False and a non-default eps."""
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

K = 4
SHAPE = (2, 3, 32, 48)
U24 = 2.0 ** -24


def make_net(cls_name, seed, check_mode=False, graphs=False):
    import unet_torch_b200 as U

    torch.manual_seed(seed)
    net = getattr(U, cls_name)(3, 2).cuda().train()
    if check_mode:
        net.set_check_mode(True)
    if graphs:
        net.enable_cuda_graphs(True)
    return net


def bns(net):
    return [(k, m) for k, m in net.named_modules() if isinstance(m, nn.BatchNorm2d)]


def step(net, x, t):
    out = net(x)
    outs = out if isinstance(out, tuple) else (out,)
    sum((o * t).mean() for o in outs).backward()
    return tuple(o.detach().clone() for o in outs)


def inputs(k):
    g = torch.Generator().manual_seed(100 + k)
    x = torch.randn(*SHAPE, generator=g).cuda()
    t = torch.randn(SHAPE[0], 2, SHAPE[2], SHAPE[3], generator=g).cuda()
    return x, t


ENGINES = [("UNet", False, False), ("UNet", False, True), ("UNet_attention", False, False), ("UNet_attention", False, True),
           ("UNet_multitask", False, False), ("UNet_multitask", False, True),
           # the fp32 generic engine (check mode) has no CUDA-graph path; UNet_multitask has no check mode
           ("UNet", True, False), ("UNet_attention", True, False)]


def engine_id(e):
    return f"{e[0]}-{'generic' if e[1] else 'tc'}{'-graphs' if e[2] else ''}"


@pytest.mark.parametrize("momentum", [0.1, 0.3, None], ids=["m0.1", "m0.3", "cumulative"])
@pytest.mark.parametrize("engine", ENGINES, ids=engine_id)
def test_running_statistics_follow_torch_recurrence(engine, momentum):
    cls_name, check_mode, graphs = engine
    arm_a = make_net(cls_name, 3, check_mode, graphs)
    arm_b = make_net(cls_name, 3, check_mode, graphs)
    g = torch.Generator().manual_seed(4)
    bn_a, bn_b = bns(arm_a), bns(arm_b)
    assert len(bn_a) == len(bn_b) > 0
    if cls_name == "UNet_attention":
        assert any(m.num_features == 1 for _, m in bn_a)
    with torch.no_grad():
        for (_, a), (_, b) in zip(bn_a, bn_b):
            a.momentum, b.momentum = 1.0, momentum
            rm, rv = torch.randn(a.num_features, generator=g), torch.rand(a.num_features, generator=g) + 0.5
            for m in (a, b):
                m.running_mean.copy_(rm)
                m.running_var.copy_(rv)
    for k in range(1, K + 1):
        prev = [(m.running_mean.clone(), m.running_var.clone()) for _, m in bn_b]
        x, t = inputs(k)
        out_a, out_b = step(arm_a, x, t), step(arm_b, x, t)
        torch.cuda.synchronize()
        for oa, ob in zip(out_a, out_b):
            assert torch.equal(oa, ob), f"step {k}: the two arms' logits differ (batch statistics are not reproducible)"
        f = 1.0 / k if momentum is None else momentum
        f32 = torch.tensor(f, dtype=torch.float32)
        for ((name, a), (_, b)), (rm0, rv0) in zip(zip(bn_a, bn_b), prev):
            for got, batch, old, what in ((b.running_mean, a.running_mean, rm0, "running_mean"),
                                          (b.running_var, a.running_var, rv0, "running_var")):
                t1, t2 = (1 - f32) * old, f32 * batch
                want = t1 + t2
                if momentum is None and k == 1:  # torch's factor is 1: the batch value itself
                    assert torch.equal(got, batch), f"step {k} {name}.{what}: {got[:4].tolist()} vs {batch[:4].tolist()}"
                # both sides round each product and the sum once (the device may fuse one into an fma, or lerp)
                bound = 6 * U24 * (t1.abs() + t2.abs()) + 1e-30
                err = (got - want).abs()
                assert bool((err <= bound).all()), (f"step {k} {name}.{what}: worst {float((err / bound).max()):.3g} x bound; "
                                                    f"got {got[:4].tolist()} want {want[:4].tolist()}")
    for (name, a), (_, b) in zip(bn_a, bn_b):
        assert int(a.num_batches_tracked) == K and int(b.num_batches_tracked) == K, name


def untrack(net):
    for _, m in bns(net):
        m.track_running_stats = False
        m.running_mean = None
        m.running_var = None
        m.num_batches_tracked = None


@pytest.mark.parametrize("engine", [("UNet", False, False), ("UNet_attention", False, False), ("UNet_multitask", False, False),
                                    ("UNet", True, False), ("UNet_attention", True, False)], ids=engine_id)
def test_untracked_batchnorm_trains_identically_and_refuses_eval(engine):
    cls_name, check_mode, _ = engine
    tracked = make_net(cls_name, 5, check_mode)
    free = make_net(cls_name, 5, check_mode)
    untrack(free)
    assert not any("running" in k or "num_batches" in k for k in free.state_dict())
    for k in (1, 2):
        x, t = inputs(k)
        out_t, out_f = step(tracked, x, t), step(free, x, t)
        for a, b in zip(out_t, out_f):
            assert torch.equal(a, b)
        for (n, pa), (_, pb) in zip(tracked.named_parameters(), free.named_parameters()):
            assert torch.equal(pa.grad, pb.grad), n
    free.eval()
    with pytest.raises(RuntimeError, match="track_running_stats=False"):
        with torch.no_grad():
            free(inputs(3)[0])


def test_eps_reaches_training_and_eval_statistics(monkeypatch):
    """eps = 1e-3 on every BatchNorm. Training (tensor-core engine): the traced rstd of each conv BatchNorm is
    1/sqrt(var + 1e-3) over the stored pre-BatchNorm map. Eval (both engines): every scale bn_eval_affine produces is
    gamma / sqrt(running_var + 1e-3), with running variances small enough that eps matters."""
    from unet_torch_b200 import ops

    eps = 1e-3
    net = make_net("UNet", 6)
    for _, m in bns(net):
        m.eps = eps
    eng = net._get_engine()
    eng.trace = []
    x, t = inputs(1)
    step(net, x * 0.05, t)   # a small input: the first BatchNorm's variance is comparable to eps
    torch.cuda.synchronize()
    trace, eng.trace = eng.trace, None
    n_checked = 0
    for kind, r in trace:
        if kind != "conv_bn_relu":
            continue
        y = r["y"].float().permute(0, 3, 1, 2).cpu().double()
        mean, var = y.mean((0, 2, 3)), y.var((0, 2, 3), unbiased=False)
        rstd = 1.0 / torch.sqrt(var + eps)
        assert torch.allclose(r["mean"].double().cpu(), mean, rtol=1e-4, atol=1e-6)
        assert torch.allclose(r["rstd"].double().cpu(), rstd, rtol=1e-4)
        n_checked += 1
    assert n_checked == 18

    calls = []
    real = ops.bn_eval_affine

    def recording(gamma, beta, rm, rv, e, scale, shift):
        real(gamma, beta, rm, rv, e, scale, shift)
        calls.append((gamma.data_ptr(), gamma.detach().clone(), rv.clone(), e, scale.clone()))

    monkeypatch.setattr(ops, "bn_eval_affine", recording)
    g = torch.Generator().manual_seed(7)
    for cls_name, check_mode in (("UNet", False), ("UNet", True), ("UNet_attention", False), ("UNet_attention", True)):
        net = make_net(cls_name, 6, check_mode)
        with torch.no_grad():
            for _, m in bns(net):
                m.eps = eps
                m.running_var.copy_(torch.rand(m.num_features, generator=g) * 2e-3)
        net.eval()
        calls.clear()
        with torch.no_grad():
            net(x)
        torch.cuda.synchronize()
        assert {c[0] for c in calls} == {m.weight.data_ptr() for _, m in bns(net)}, cls_name
        for _, gamma, rv, e, scale in calls:
            assert e == eps
            want = gamma.double().cpu() / torch.sqrt(rv.double().cpu() + torch.tensor(eps, dtype=torch.float32).double())
            err = (scale.double().cpu() - want).abs()
            assert bool((err <= 4 * U24 * want.abs()).all()), cls_name
