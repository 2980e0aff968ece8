"""-m gpu: networks with more than eight classes (up to 256) on the tensor-core engine, and the fused CE/Dice loss and
softmax -> argmax at any class count.

kernels   the many-class OutConv forward / backward against fp64 on the host, bit-for-bit against the per-class-count head
          at <= 8 classes; the fused mask / density / sigmoid heads against the two-kernel path; CE + softmax-Dice forward and
          backward against the fp64 oracle; softmax_argmax against oracle.softmax_argmax.
networks  a UNet(3, 21) training step against the bf16-storage emulation on the host; eager vs CUDA-graph replay; FusedAdam;
          UNet_multitask / UNet_attention with 12 classes; the predict* heads; the generic engine with 12 classes.
"""
import statistics

import numpy as np
import pytest
import torch

from gpu_util import cos, host_step, rel_l2, to_nhwc_bf16
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu


def _many(name, *args):
    from unet_torch_b200 import _lib

    _lib.call(name, *args, torch.cuda.current_stream().cuda_stream)


def _head_inputs(ncls, n, h, w, cin, seed):
    g = torch.Generator().manual_seed(seed)
    a = to_nhwc_bf16(torch.randn(n, cin, h, w, generator=g))
    wt = (torch.randn(ncls, cin, 1, 1, generator=g) * 0.2).cuda()
    b = (torch.randn(ncls, generator=g) * 0.1).cuda()
    return a, wt, b


def _many_fprop(a, wt, b):
    n, h, w, cin = a.shape
    ncls = wt.shape[0]
    z = torch.empty((n, ncls, h, w), dtype=torch.float32, device="cuda")
    _many("b200unet_head_many_fprop", a.data_ptr(), a.stride(2), wt.data_ptr(), b.data_ptr(), z.data_ptr(), n, h, w, cin, ncls)
    return z


def _many_bwd(dz, a, wt):
    from unet_torch_b200 import _lib

    n, h, w, cin = a.shape
    ncls = wt.shape[0]
    da = torch.empty_like(a)
    dw = torch.empty((ncls, cin), dtype=torch.float32, device="cuda")
    db = torch.empty((ncls,), dtype=torch.float32, device="cuda")
    ws = torch.empty(_lib.query("b200unet_head_many_bwd_workspace_floats", n, h, w, cin, ncls), dtype=torch.float32, device="cuda")
    _many("b200unet_head_many_bwd", dz.data_ptr(), a.data_ptr(), a.stride(2), wt.data_ptr(), da.data_ptr(), da.stride(2),
          ws.data_ptr(), dw.data_ptr(), db.data_ptr(), n, h, w, cin, ncls)
    return da, dw, db


@pytest.mark.parametrize("ncls,cin,n,h,w", [(1, 64, 2, 24, 40), (8, 64, 2, 24, 40), (9, 64, 2, 24, 40), (21, 64, 2, 64, 96),
                                            (64, 64, 1, 48, 40), (256, 64, 1, 32, 48), (21, 128, 2, 32, 40),
                                            (256, 128, 1, 16, 24), (5, 128, 1, 16, 24)])
def test_head_many_forward_backward_against_fp64(ncls, cin, n, h, w):
    from unet_torch_b200 import ops

    a, wt, b = _head_inputs(ncls, n, h, w, cin, ncls * 31 + cin)
    z = _many_fprop(a, wt, b)
    a64 = a.double().cpu()
    w64 = wt.view(ncls, cin).double().cpu()
    ref = torch.einsum("nhwc,jc->njhw", a64, w64) + b.double().cpu().view(1, ncls, 1, 1)
    assert rel_l2(z, ref) < 1e-6, rel_l2(z, ref)
    if ncls <= 8:  # same fmaf chain as the per-class-count head: identical bits
        z8 = torch.empty_like(z)
        ops.head_fprop(a, wt, b, z8)
        assert torch.equal(z.view(torch.int32), z8.view(torch.int32))
    g = torch.Generator().manual_seed(ncls + 7)
    dz = torch.randn(n, ncls, h, w, generator=g).cuda()
    da, dw, db = _many_bwd(dz, a, wt)
    dz64 = dz.double().cpu()
    dw_ref = torch.einsum("njhw,nhwc->jc", dz64, a64)
    db_ref = dz64.sum(dim=(0, 2, 3))
    assert rel_l2(dw, dw_ref) < 1e-5 and rel_l2(db, db_ref) < 1e-5, (rel_l2(dw, dw_ref), rel_l2(db, db_ref))
    da_ref = torch.einsum("njhw,jc->nhwc", dz64, w64)
    err = (da.double().cpu() - da_ref).abs()
    # one bf16 rounding of an fp32 sum: half an ulp of bf16 (2^-9 relative) plus the fp32 summation error
    assert bool((err <= 2.0 ** -8 * da_ref.abs() + 1e-5 * float(da_ref.abs().max())).all()), float(err.max())
    if ncls <= 8:  # the fixed-count backward sums the classes in the same order: the same da
        da8, dw8, db8 = torch.empty_like(a), torch.empty_like(dw).view(ncls, cin, 1, 1), torch.empty_like(db)
        ops.head_bwd(dz, a, wt, da8, dw8, db8)
        assert torch.equal(da, da8)
        assert rel_l2(dw, dw8.view(ncls, cin)) < 1e-6 and rel_l2(db, db8) < 1e-6


def _same_bits(a, b):
    return bool(((a == b) | (a.isnan() & b.isnan())).all())


@pytest.mark.parametrize("ncls,cin,n,h,w", [(9, 64, 2, 64, 96), (21, 64, 3, 32, 80), (256, 64, 1, 48, 48),
                                            (256, 128, 1, 32, 32), (12, 128, 2, 16, 48)])
def test_fused_many_heads_equal_the_two_kernel_path(ncls, cin, n, h, w):
    from unet_torch_b200 import ops

    a, wt, b = _head_inputs(ncls, n, h, w, cin, ncls * 3 + n)
    wt[1] = wt[0]  # an exact tie between classes 0 and 1 wherever they win: the first must be reported
    b[1] = b[0]
    a[0, 0, 3, 5] = float("nan")  # a NaN row: every logit NaN -> class 0, NaN maps
    a[-1, h - 1, w - 1, 0] = float("nan")
    logits = torch.empty((n, ncls, h, w), dtype=torch.float32, device="cuda")
    ops.head_fprop(a, wt, b, logits)
    mask = ops.head_mask(a, wt, b)
    assert mask.dtype == torch.uint8 and mask.shape == (n, h, w)
    assert torch.equal(mask.long(), ops.softmax_argmax(logits))
    assert not bool((mask == 1).any()) and int(mask[0, 0, 3]) == 0 and int(mask[-1, h - 1, w - 1]) == 0
    assert len(torch.unique(mask)) >= min(ncls - 1, 8)
    dens, counts = ops.head_density(a, wt, b, 200.0)
    want, want_counts = O.density_maps(logits.cpu(), 200.0)
    assert _same_bits(dens.cpu(), want) and bool(dens[0, :, 0, 3].isnan().all())
    fin = torch.isfinite(want_counts)
    assert torch.equal(fin, torch.isfinite(counts.cpu()))
    assert torch.allclose(counts.cpu()[fin], want_counts[fin], rtol=1e-12, atol=1e-12)
    relu_only, none = ops.head_density(a, wt, b, 1.0, with_counts=False)
    assert none is None and _same_bits(relu_only.cpu(), torch.relu(logits.cpu()))
    sm = ops.head_sigmoid_mask(a, wt, b, 0.5)
    assert torch.equal(sm, (torch.sigmoid(logits)[:, 0] >= 0.5).to(torch.uint8))
    assert torch.equal(sm.cpu(), O.sigmoid_mask(logits.cpu()))


def _oracle_loss_grad(z, y, loss_type, ncls):
    z64 = z.double().cpu().requires_grad_(True)
    loss = O.calc_loss(z64, y.double().cpu(), loss_type, ncls)
    loss.backward()
    return float(loss), z64.grad


@pytest.mark.parametrize("ncls,n,h,w", [(9, 2, 32, 48), (21, 2, 17, 23), (21, 3, 40, 40), (256, 1, 20, 20), (256, 2, 7, 9)])
@pytest.mark.parametrize("loss_type", ["dice_bce_mc", "CE"])
def test_ce_dice_many_classes_against_fp64_oracle(ncls, n, h, w, loss_type):
    import unet_torch_b200 as U

    g = torch.Generator().manual_seed(ncls * 100 + h)
    z = (torch.randn(n, ncls, h, w, generator=g) * 3).cuda().requires_grad_(True)
    y = torch.randint(0, ncls, (n, h, w), generator=g).float().cuda()
    U.loss.CLASS_NUMBER = ncls
    loss = U.calc_loss(z, y, loss_type=loss_type)
    loss.backward()
    want, dwant = _oracle_loss_grad(z.detach(), y, loss_type, ncls)
    assert abs(float(loss) - want) <= 1e-5 * abs(want), (float(loss), want)
    assert rel_l2(z.grad, dwant) < 1e-5, rel_l2(z.grad, dwant)
    # deterministic: the per-class sums are reduced in a fixed order
    z2 = z.detach().clone().requires_grad_(True)
    loss2 = U.calc_loss(z2, y, loss_type=loss_type)
    loss2.backward()
    assert float(loss2) == float(loss) and torch.equal(z2.grad, z.grad)
    if loss_type == "dice_bce_mc":
        d = U.DiceLoss(ncls)(z.detach(), y, softmax=True)
        dref = float(O.dice_softmax(z.detach().double().cpu(), y.double().cpu(), ncls))
        assert abs(float(d) - dref) <= 1e-5 * abs(dref) + 1e-7


@pytest.mark.parametrize("ncls", [9, 21, 256])
def test_out_of_range_labels_set_the_flag(ncls):
    import unet_torch_b200 as U

    z = torch.randn(2, ncls, 16, 20, device="cuda")
    for bad in (ncls, -1, ncls + 0.5):
        y = torch.randint(0, ncls, (2, 16, 20), device="cuda").float()
        y[1, 7, 3] = bad
        with pytest.raises(IndexError):
            U.loss.ce_dice_loss(z, y, check_labels=True)
    U.loss._pending.clear()
    y = torch.randint(0, ncls, (2, 16, 20), device="cuda").float()
    U.loss.ce_dice_loss(z, y, check_labels=True)
    y[0, 0, 0] = ncls
    U.calc_loss(z, y, loss_type="CE")
    with pytest.raises(IndexError):
        U.loss.check_pending_label_errors(wait=True)


@pytest.mark.parametrize("ncls,n,h,w", [(9, 2, 64, 64), (21, 2, 33, 47), (256, 1, 40, 40)])
def test_softmax_argmax_any_class_count_matches_the_oracle(ncls, n, h, w):
    from unet_torch_b200 import ops

    g = torch.Generator().manual_seed(ncls)
    z = torch.randn(n, ncls, h, w, generator=g) * 2
    z[:, 2] = z[:, 1]  # exact ties: the first maximum wins
    z[0, :, 0, 0] = float("nan")
    z[-1, 3, 1, 1] = float("nan")
    got = ops.softmax_argmax(z.cuda()).cpu()
    want = O.softmax_argmax(z)
    p = torch.softmax(z, dim=1)
    top2 = p.nan_to_num(-1.0).topk(2, dim=1).values
    near = (top2[:, 0] - top2[:, 1]) <= (torch.nextafter(top2[:, 0], torch.full_like(top2[:, 0], 2.0)) - top2[:, 0])
    differ = got != want
    print(f"softmax_argmax C={ncls}: {int(near.sum())} pixels with the top two probabilities within 1 ulp, "
          f"{int(differ.sum())} differ from the oracle")
    assert not bool((differ & ~near).any())
    assert int(got[0, 0, 0]) == 0 and int(got[-1, 1, 1]) == 0 and not bool((got == 2).any())


def _step_inputs(n, h, w, ncls, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 3, h, w, generator=g)
    y = torch.randint(0, ncls, (n, h, w), generator=g).float()
    return x, y


def test_unet_21_classes_training_step_against_the_emulation():
    """One training step of UNet(3, 21) against the same torch CPU ops in fp64 (truth) and with only the engine's bf16
    storage points inserted (emulation): the engine is no further from the truth than the emulation, and close to it."""
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    ncls = 21
    torch.manual_seed(3)
    net = U.UNet(3, ncls)
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().train()
    x, y = _step_inputs(2, 64, 96, ncls, 4)
    assert isinstance(net._engine_for(x.cuda()), UNetEngine)
    U.loss.CLASS_NUMBER = ncls
    out = net(x.cuda())
    loss = U.calc_loss(out, y.cuda(), loss_type="dice_bce_mc")
    loss.backward()
    torch.cuda.synchronize()
    tl, tloss, tg, _ = host_step(sd0, x, y, ncls, "dice_bce_mc", dtype=torch.float64)
    el, eloss, eg, _ = host_step(sd0, x, y, ncls, "dice_bce_mc", emulate=True)
    grads = {k: p.grad for k, p in net.named_parameters()}
    e_logits, y_logits = rel_l2(out.detach(), tl), rel_l2(el, tl)
    errs = {k: rel_l2(grads[k], tg[k]) for k in tg}
    yard = {k: rel_l2(eg[k], tg[k]) for k in tg}
    med, med_yard = statistics.median(errs.values()), statistics.median(yard.values())
    rows = {k: (rel_l2(grads[k], eg[k]), cos(grads[k], eg[k])) for k in eg}
    print(f"UNet(3, 21): logits rel {e_logits:.3e} (emulation {y_logits:.3e}), loss {float(loss):.6f} vs {tloss:.6f} "
          f"(emulation {eloss:.6f}); grads median rel {med:.3e} (emulation {med_yard:.3e}); vs the emulation: median "
          f"{statistics.median(r[0] for r in rows.values()):.3e}, min cos {min(r[1] for r in rows.values()):.4f}")
    assert e_logits <= 1.5 * y_logits and abs(float(loss) - tloss) < 1e-2 * abs(tloss)
    assert med <= 1.5 * med_yard
    assert rel_l2(out.detach(), el) <= y_logits
    assert statistics.median(r[0] for r in rows.values()) <= med_yard and min(r[1] for r in rows.values()) > 0.9
    # head parameters: the many-class backward against the truth
    assert rel_l2(grads["outc.conv.weight"], tg["outc.conv.weight"]) <= 1.5 * yard["outc.conv.weight"] + 1e-3
    assert rel_l2(grads["outc.conv.bias"], tg["outc.conv.bias"]) <= 1.5 * yard["outc.conv.bias"] + 1e-3


def test_graph_replay_equals_eager_and_fused_optimizers_train():
    import unet_torch_b200 as U

    ncls = 21
    U.loss.CLASS_NUMBER = ncls
    x, y = (t.cuda() for t in _step_inputs(2, 64, 48, ncls, 8))
    states = []
    for graphs in (False, True):
        torch.manual_seed(9)
        net = U.UNet(3, ncls).cuda().train().enable_cuda_graphs(graphs)
        opt = U.FusedSGD(net, lr=0.05, momentum=0.9, weight_decay=1e-4)
        rec = []
        for _ in range(3):
            out = net(x)
            loss = U.calc_loss(out, y, loss_type="dice_bce_mc")
            opt.zero_grad(set_to_none=True)
            loss.backward()
            rec.append((out.detach().clone(), float(loss), net.outc.conv.weight.grad.clone(), net.outc.conv.bias.grad.clone()))
            opt.step()
        states.append((net, rec))
    (ne, re), (ng, rg) = states
    assert ng._engine._graphs, "no graph was captured"
    for (o1, l1, g1, b1), (o2, l2, g2, b2) in zip(re, rg):
        assert torch.equal(o1, o2) and l1 == l2 and torch.equal(g1, g2) and torch.equal(b1, b2)
    for (k, a), (_, b) in zip(ne.state_dict().items(), ng.state_dict().items()):
        assert torch.equal(a, b), k
    assert re[-1][1] < re[0][1]
    torch.manual_seed(9)
    net = U.UNet(3, ncls).cuda().train()
    opt = U.FusedAdam(net, lr=1e-3)
    losses = []
    for _ in range(4):
        loss = U.calc_loss(net(x), y, loss_type="dice_bce_mc")
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print("FusedAdam, 21 classes:", losses)
    assert losses[-1] < losses[0]


def test_multitask_and_attention_with_12_classes_train_on_the_tensor_core_engine():
    import unet_torch_b200 as U
    from unet_torch_b200.model import UNetEngine

    ncls = 12
    U.loss.CLASS_NUMBER = ncls
    g = torch.Generator().manual_seed(12)
    x = torch.randn(2, 3, 64, 64, generator=g).cuda()
    t1, t2 = torch.rand(2, ncls, 64, 64, generator=g).cuda(), torch.rand(2, ncls, 64, 64, generator=g).cuda()
    y = torch.randint(0, ncls, (2, 64, 64), generator=g).float().cuda()
    torch.manual_seed(1)
    mt = U.UNet_multitask(3, ncls).cuda().train()
    assert isinstance(mt._engine_for(x), UNetEngine)
    opt = U.FusedSGD(mt, lr=0.05, momentum=0.9)
    losses = []
    for _ in range(4):
        o1, o2 = mt(x)
        assert o1.shape == (2, ncls, 64, 64)
        loss = U.calc_loss(torch.relu(o1), t1, loss_type="mseMC") + U.calc_loss(torch.relu(o2), t2, loss_type="mseMC")
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print("UNet_multitask(3, 12) mseMC:", losses)
    assert losses[-1] < losses[0]
    torch.manual_seed(2)
    at = U.UNet_attention(3, ncls).cuda().train()
    assert isinstance(at._engine_for(x), UNetEngine)
    opt = U.FusedSGD(at, lr=0.05, momentum=0.9)
    losses = []
    for _ in range(4):
        loss = U.calc_loss(at(x), y, loss_type="dice_bce_mc")
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print("UNet_attention(3, 12) dice_bce_mc:", losses)
    assert losses[-1] < losses[0]


def test_predict_heads_with_21_classes_equal_the_unfused_path():
    import unet_torch_b200 as U

    torch.manual_seed(5)
    net = U.UNet(3, 21).cuda().eval()
    x = torch.randn(2, 3, 64, 96, device="cuda")
    with torch.no_grad():
        logits = net(x)
        mask = net.predict(x)
        dens, counts = net.predict_density(x)
    assert torch.equal(mask.long(), U.predict_mask(logits))
    assert torch.equal(net.predict_binary(x), (torch.sigmoid(logits)[:, 0] >= 0.5).to(torch.uint8))
    assert np.array_equal(dens.cpu().numpy(), torch.relu(logits).cpu().numpy() / 200)
    assert torch.allclose(counts, dens.double().sum(dim=(2, 3)), rtol=1e-12)
    # tiled inference (test.py:420-447) with the fused many-class mask head against the crop-by-crop loop
    img = torch.randint(0, 256, (100, 150, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    got = U.predict_tiled(net, img.numpy(), 64, head="mask", max_batch=4)
    with torch.no_grad():
        want = O.tiled_masks(lambda t: net(t.cuda()).cpu(), O.preprocess_crop(img.numpy(), 64), 64, O.mask_uint8)
    assert got.shape == (128, 192) and float((got.cpu() == want).float().mean()) > 0.9999


def test_generic_engine_trains_12_classes_against_the_fp64_oracle():
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine

    ncls = 12
    torch.manual_seed(4)
    net = U.UNet(3, ncls, 64)
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().train().set_check_mode(True)
    x, y = _step_inputs(2, 32, 48, ncls, 5)
    assert isinstance(net._engine_for(x.cuda()), GenericEngine)
    U.loss.CLASS_NUMBER = ncls
    out = net(x.cuda())
    loss = U.calc_loss(out, y.cuda(), loss_type="dice_bce_mc")
    loss.backward()
    tl, tloss, tg, _ = host_step(sd0, x, y, ncls, "dice_bce_mc", dtype=torch.float64)
    e_logits, e_loss = rel_l2(out.detach(), tl), abs(float(loss) - tloss) / abs(tloss)
    errs = {k: rel_l2(p.grad, tg[k]) for k, p in net.named_parameters()}
    print(f"generic engine, 12 classes: logits rel {e_logits:.2e}, loss rel {e_loss:.2e}, worst grad rel {max(errs.values()):.2e}")
    assert e_logits < 1e-4 and e_loss < 1e-4
    assert max(errs.values()) < 5e-2  # fp32 against fp64, as tests/test_gpu_generic.py judges check mode
