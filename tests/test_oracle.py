"""CPU: the oracle (oracle/unet_oracle.py) against the golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py), and - when the reference modules are staged (oracle/build_ref.py) - against the live reference."""
import os
import sys

import pytest
import torch

from oracle import ref_loader
from oracle import unet_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.mark.parametrize("case", ["w4_c1_k2_dicebce", "w4_c3_k5_dicebce", "w4_c3_k3_ce", "w4_c3_k2_msemc"])
def test_small_net_forward_backward_matches_reference(golden, case):
    g = golden("ref_small_nets.pt")[case]
    ch, ncls, width, n, h, w, seed = g["cfg"]
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd0"].items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    sd_req = dict(sd)
    sd_req.update(params)
    logits, new_buf = O.unet_forward(sd_req, g["x"].double(), training=True)
    pred = O.relu(logits) if g["loss_type"].startswith("mse") else logits
    loss = O.calc_loss(pred, g["y"].double(), g["loss_type"], ncls)
    loss.backward()
    # fp64 oracle vs fp64 reference: tight; vs the fp32 reference: fp32 round-off
    assert rel(logits, g["logits64"]) < 2e-6
    assert abs(float(loss) - float(g["loss64"])) < 1e-9 * max(1.0, abs(float(g["loss64"])))
    assert rel(logits, g["logits"]) < 1e-4
    for k, p in params.items():
        assert rel(p.grad, g["grads64"][k]) < 1e-5, k
    for k, v in g["buffers1"].items():
        if "num_batches" in k:
            assert int(new_buf[k]) == int(v)
        else:
            assert rel(new_buf[k], v) < 1e-5, k
    # eval mode uses the updated running statistics
    sd_eval = dict(sd)
    sd_eval.update({k: v.double() if v.is_floating_point() else v for k, v in g["buffers1"].items()})
    le, _ = O.unet_forward(sd_eval, g["x"].double(), training=False)
    assert rel(le, g["logits_eval"]) < 1e-4


def test_pool_semantics(golden):
    ops = golden("ref_ops.pt")
    for key in ("pool", "pool_odd"):
        v, pos, idx = O.maxpool2x2(ops[key]["x"])
        assert torch.equal(idx, ops[key]["idx"])
        assert torch.equal(torch.nan_to_num(v, nan=7.0), torch.nan_to_num(ops[key]["out"], nan=7.0))


def test_softmax_argmax_semantics(golden):
    ops = golden("ref_ops.pt")
    for key in ("argmax_small_logits", "argmax_ties"):
        assert torch.equal(O.softmax_argmax(ops[key]["z"]), ops[key]["mask"])


@pytest.mark.parametrize("ncls", [2, 5])
@pytest.mark.parametrize("lt", ["dice_bce_mc", "CE"])
def test_loss_closed_form(golden, ncls, lt):
    g = golden("ref_ops.pt")[f"loss_{lt}_{ncls}"]
    z = g["z"].clone().requires_grad_(True)
    l = O.calc_loss(z, g["t"], lt, ncls)
    (gr,) = torch.autograd.grad(l, z)
    assert abs(float(l) - float(g["loss"])) < 2e-6
    assert rel(gr, g["grad"]) < 1e-5


def test_mse_losses(golden):
    ops = golden("ref_ops.pt")
    g = ops["loss_relu_mseMC"]
    o = g["o"].clone().requires_grad_(True)
    l = O.calc_loss(O.relu(o), g["t"], "mseMC")
    (gr,) = torch.autograd.grad(l, o)
    assert abs(float(l) - float(g["loss"])) < 1e-6 and rel(gr, g["grad"]) < 1e-6
    g = ops["loss_mse"]
    o = g["o"].clone().requires_grad_(True)
    l = O.calc_loss(o, g["t"], "mse")
    (gr,) = torch.autograd.grad(l, o)
    assert abs(float(l) - float(g["loss"])) < 1e-6 and rel(gr, g["grad"]) < 1e-6


@pytest.mark.skipif(not ref_loader.available(), reason="reference modules not staged (python oracle/build_ref.py)")
def test_live_reference_agrees():
    ref, _ = ref_loader.load()
    torch.manual_seed(3)
    net = ref.UNet(2, 3, 4).double()
    x = torch.randn(2, 2, 32, 32, dtype=torch.float64)
    net.train()
    want = net(x)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    # the training forward above already updated the running stats; recompute from the pre-update buffers
    for k in sd:
        if k.endswith("running_mean"):
            sd[k] = torch.zeros_like(sd[k])
        if k.endswith("running_var"):
            sd[k] = torch.ones_like(sd[k])
    got, _ = O.unet_forward(sd, x, training=True)
    assert rel(got, want) < 1e-10


@pytest.mark.skipif(not ref_loader.available(), reason="reference modules not staged (python oracle/build_ref.py)")
@pytest.mark.parametrize("h,w,dropout", [(37, 45, False), (32, 32, True), (50, 35, True)])
def test_live_reference_odd_sizes_and_dropout(h, w, dropout):
    """Pins the oracle's floor-mode pooling, the F.pad branch (Model.py:69-73) and the dropout placement
    (Model.py:34-39, 81-82) to the unmodified reference: same seed -> same masks (CPU generator, same draw order)."""
    import torch.nn.functional as F

    ref, _ = ref_loader.load()
    torch.manual_seed(4)
    net = ref.UNet(3, 2, 4, dropout=dropout, dropout_p=0.3).double()
    x = torch.randn(2, 3, h, w, dtype=torch.float64)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net.train()
    torch.manual_seed(77)
    want = net(x)
    masks = None
    if dropout:
        torch.manual_seed(77)
        masks = {name: F.dropout(torch.ones(shape, dtype=torch.float64), 0.3, True)
                 for name, shape in O.dropout_mask_shapes(2, h, w, 4)}
    got, _ = O.unet_forward(sd, x, training=True, dropout_masks=masks)
    assert got.shape == want.shape == (2, 2, h, w)
    assert rel(got, want) < 1e-10


def test_cpu_baseline_port_matches_oracle():
    """bench.py's CPU baseline issues the torch library ops the reference calls; it must agree with the oracle."""
    from oracle import cpu_baseline as CB

    sd = CB.init_state(3, 2, width=4, seed=5)
    x = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(6))
    a = CB.unet_forward_torchops({k: v.clone() for k, v in sd.items()}, x, True)
    b, _ = O.unet_forward(sd, x, True)
    assert rel(a, b) < 1e-5


def test_preprocess_restatement_matches_reference_golden(golden):
    """oracle.preprocess against the outputs of the reference's own `preprocess` (oracle/make_golden_edge.py)."""
    import numpy as np

    g = golden("ref_edge.pt")
    assert len(g) >= 8
    with np.errstate(all="ignore"):
        for name, c in g.items():
            if name.startswith("crop_"):   # preprocessCrop of test.py: pad with 255 to a multiple of the crop size first
                got = O.preprocess_crop(c["img"].numpy(), c["crop"])
                assert tuple(got.shape[2:]) == c["label_shape"] and torch.equal(got, c["out"]), name
                continue
            got = O.preprocess(c["img"].numpy())
            assert got.shape == c["out"].shape and got.dtype == torch.float32, name
            same = (got == c["out"]) | (got.isnan() & c["out"].isnan())
            assert bool(same.all()), name
    assert bool(g["bgr_constant_channel"]["out"].isnan().any())  # std = 0 channel: the reference yields nan


def test_inference_epilogue_restatements():
    z = torch.randn(2, 5, 8, 8, generator=torch.Generator().manual_seed(3))
    assert torch.equal(O.mask_uint8(z).long(), torch.argmax(torch.softmax(z, 1), 1))
    assert torch.equal(O.sigmoid_mask(z), (torch.sigmoid(z)[:, 0] >= 0.5).to(torch.uint8))
    tiny = torch.tensor([-1e-9, -3e-8, -2e-7, -4e-7, 0.0, 1e-9]).reshape(1, 1, 1, 6)  # fp32 rounding decides around z = 0-
    assert torch.equal(O.sigmoid_mask(tiny), (torch.sigmoid(tiny)[:, 0] >= 0.5).to(torch.uint8))
    d, cnt = O.density_maps(z, 200.0)
    assert torch.equal(d, torch.relu(z) / 200) and torch.allclose(cnt, d.double().sum((2, 3)))


@pytest.mark.parametrize("case", ["w4_sum", "w4_uncertainty"])
def test_multitask_restatement_matches_reference_golden(golden, case):
    """oracle.unet_multitask_forward (+ relu/mseMC, MultitaskUncertaintyLoss) against the reference's UNet_multitask."""
    g = golden("ref_multitask.pt")[case]
    ch, ncls, width, n, h, w, seed = g["cfg"]
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd0"].items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    sd_req = dict(sd)
    sd_req.update(params)
    (o1, o2), new_buf = O.unet_multitask_forward(sd_req, g["x"].double(), training=True)
    l1 = O.calc_loss(O.relu(o1), g["t1"].double(), "mseMC", ncls)
    l2 = O.calc_loss(O.relu(o2), g["t2"].double(), "mseMC", ncls)
    if g["combine"] == "sum":
        loss = l1 + l2
    else:
        lv = [torch.tensor([0.3], dtype=torch.float64), torch.tensor([-0.2], dtype=torch.float64)]
        loss = O.multitask_uncertainty_loss([l1, l2], lv, [True, True]).reshape(())
    loss.backward()
    assert rel(o1, g["o1_64"]) < 2e-6 and rel(o2, g["o2_64"]) < 2e-6
    assert abs(float(loss) - float(g["loss64"])) < 1e-9 * max(1.0, abs(float(g["loss64"])))
    assert rel(o1, g["o1"]) < 1e-4 and rel(o2, g["o2"]) < 1e-4
    for k, p in params.items():
        assert rel(p.grad, g["grads64"][k]) < 1e-5, k
    for k, v in g["buffers1"].items():
        if "num_batches" in k:
            assert int(new_buf[k]) == int(v)
        else:
            assert rel(new_buf[k], v) < 1e-5, k


def test_bf16_storage_emulation_reproduces_the_references_own_bf16_error(golden):
    """`cpu_baseline.unet_forward_torchops(emulate_bf16=True)` is the yardstick AND the composition checker of the -m gpu
    end-to-end tests. It is pinned two ways: with the flag off it equals the oracle (test_cpu_baseline_port_matches_oracle);
    with the flag on, its error against the reference's fp64 run must look like the reference's OWN error under
    torch.autocast(bfloat16) (tests/golden/ref_bf16_yardstick.pt, oracle/make_golden_yardstick.py): logits within 10 %,
    median parameter-gradient error within 10 %, no parameter above 2 x (measured 0.99-1.02 median, <= 1.74 worst)."""
    import statistics
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gpu_util import host_step, rel_l2

    import unet_torch_b200 as U

    full = golden("ref_full_nets.pt")
    yard_all = golden("ref_bf16_yardstick.pt")
    for case in ("w64_c3_k2_dicebce", "w64_c3_k2_msemc"):
        g, yard = full[case], yard_all[case]["bf16_autocast"]
        ch, ncls, width, n, h, w, seed = g["cfg"]
        torch.manual_seed(seed)
        sd0 = {k: v.clone() for k, v in U.UNet(ch, ncls, width).state_dict().items()}
        el, eloss, eg, _ = host_step(sd0, g["x"], g["y"], ncls, g["loss_type"], relu=g["loss_type"].startswith("mse"), emulate=True)
        e_logits = rel_l2(el, g["logits64"])
        errs = {k: rel_l2(eg[k], gs) for k, gs in g["grad_small64"].items()}
        errs.update({k: rel_l2(eg[k].flatten()[::997], gs) for k, gs in g["grad_sample64"].items()})
        med, med_yard = statistics.median(errs.values()), statistics.median(yard["grads"].values())
        assert abs(e_logits / yard["logits"] - 1) < 0.1, (case, e_logits, yard["logits"])
        assert abs(med / med_yard - 1) < 0.1, (case, med, med_yard)
        assert all(errs[k] <= 2.0 * yard["grads"][k] + 0.02 for k in errs)
        assert abs(eloss - float(g["loss64"])) / abs(float(g["loss64"])) < 1e-2


def test_staged_reference_copy_is_the_reference_byte_for_byte():
    """oracle/_ref (git-ignored) must be the unmodified reference files: the staged files still have the hashes that
    oracle/build_ref.py recorded (and checked against the source) when it copied them."""
    import hashlib
    import json

    d = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(d, "MANIFEST.json")):
        pytest.skip("oracle/_ref not staged (python oracle/build_ref.py)")
    for name, digest in json.load(open(os.path.join(d, "MANIFEST.json")))["files"].items():
        assert hashlib.sha256(open(os.path.join(d, name), "rb").read()).hexdigest() == digest, name
    RefModel, ref_loss = ref_loader.load()
    assert RefModel.UNet(1, 2, 4).state_dict().keys() and callable(ref_loss.calc_loss)


@pytest.mark.parametrize("case", ["w4_c3_k2_dicebce", "w4_c1_k3_msemc"])
def test_attention_restatement_matches_reference_golden(golden, case):
    """unet_oracle.unet_attention_forward / attention_block against the unmodified reference's UNet_attention
    (Model.py:257-391): logits, loss, every parameter gradient, BatchNorm buffers (incl. the gates' three BatchNorms per
    level), eval logits."""
    g = golden("ref_attention.pt")[case]
    ch, ncls, width, n, h, w, seed = g["cfg"]
    sd = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else
              (v.double() if v.is_floating_point() else v)) for k, v in g["sd0"].items()}
    out, nb = O.unet_attention_forward(sd, g["x"].double(), training=True)
    pred = torch.relu(out) if g["loss_type"].startswith("mse") else out
    loss = O.calc_loss(pred, g["y"].double(), g["loss_type"], ncls)
    loss.backward()
    # fp64 oracle vs fp64 reference: tight; vs the fp32 reference: fp32 round-off
    assert rel(out.detach(), g["logits64"]) < 2e-6 and rel(out.detach(), g["logits"]) < 1e-4
    assert abs(float(loss) - float(g["loss64"])) < 1e-9 * max(1.0, abs(float(g["loss64"])))
    # biases in front of a BatchNorm (W_q / W_x / psi conv, the gate's ConvTranspose2d) have an exactly-zero gradient:
    # errors are measured against max(|reference gradient|, 1e-6 x the largest gradient norm of the net)
    floor = 1e-6 * max(float(gr.double().norm()) for gr in g["grads64"].values())
    for k, gr in g["grads64"].items():
        assert float((sd[k].grad - gr.double()).norm()) / max(float(gr.double().norm()), floor) < 1e-4, k
    for k, v in g["buffers1"].items():
        if "num_batches" in k:
            assert int(nb[k]) == int(v), k
        else:
            assert rel(nb[k], v) < 1e-5, k
    sd_eval = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd0"].items()}
    sd_eval.update({k: v.double() if v.is_floating_point() else v for k, v in g["buffers1"].items()})
    oe, _ = O.unet_attention_forward(sd_eval, g["x"].double(), training=False)
    assert rel(oe, g["logits_eval"]) < 1e-4


def test_attention_module_matches_reference_interface():
    """UNet_attention container: same 210 state_dict keys and - under the same seed - bit-identical initial weights as the
    reference constructor (Model.py:299-345: gates keep torch's default init), with and without dropout."""
    import unet_torch_b200 as U

    g = torch.load(os.path.join(ROOT, "tests", "golden", "ref_attention.pt"), weights_only=False)["w4_c3_k2_dicebce"]
    ch, ncls, width, n, h, w, seed = g["cfg"]
    torch.manual_seed(seed)
    net = U.UNet_attention(ch, ncls, width)
    sd = net.state_dict()
    assert list(sd.keys()) == list(g["sd0"].keys()) and len(sd) == 210
    assert all(torch.equal(sd[k], g["sd0"][k]) for k in sd)
    import Model  # the root drop-in shim re-exports it (train.py:6)

    assert Model.UNet_attention is U.UNet_attention
    with pytest.raises(RuntimeError):
        net.attenion4(torch.zeros(1), torch.zeros(1))   # containers are not the product path


def test_attention_restatement_at_full_width_matches_reference_fp64():
    """The oracle's UNet_attention at the reference's default width (64), pinned to the unmodified reference's fp64 run
    (tests/golden/ref_attention_bf16_yardstick.pt, oracle/make_golden_attention_yardstick.py): same seed -> same weights
    (checksums stored with the golden) -> logits, loss, the gradients of every small parameter, eval logits."""
    import unet_torch_b200 as U

    g = torch.load(os.path.join(ROOT, "tests", "golden", "ref_attention_bf16_yardstick.pt"), weights_only=False)[
        "att_w64_c3_k2_dicebce_64"]
    ch, ncls, width, n, h, w, seed, loss_type = g["cfg"]
    torch.manual_seed(seed)
    sd0 = U.UNet_attention(ch, ncls, width).state_dict()
    for k, v in sd0.items():
        if v.is_floating_point():
            assert abs(float(v.double().sum()) - g["sd0_checksum"][k]) <= 1e-9 * max(1.0, abs(g["sd0_checksum"][k])), k
    sd = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else
              (v.double() if v.is_floating_point() else v)) for k, v in sd0.items()}
    out, nb = O.unet_attention_forward(sd, g["x"].double(), training=True)
    loss = O.calc_loss(out, g["y"].double(), loss_type, ncls)
    loss.backward()
    assert rel(out.detach(), g["logits64"]) < 1e-5          # the golden keeps the fp64 logits as fp32
    assert abs(float(loss) - g["loss64"]) < 1e-9 * max(1.0, abs(g["loss64"]))
    for k, gr in g["small_grads64"].items():
        assert float((sd[k].grad - gr.double()).norm()) / max(float(gr.double().norm()), g["grad_floor"]) < 1e-4, k
    for k, v in g["buffers1"].items():
        assert rel(nb[k], v) < 1e-5, k
    sd_eval = {k: (v.double() if v.is_floating_point() else v) for k, v in sd0.items()}
    sd_eval.update({k: v.double() for k, v in nb.items() if v.is_floating_point()})
    oe, _ = O.unet_attention_forward(sd_eval, g["x"].double(), training=False)
    assert rel(oe, g["logits_eval64"]) < 1e-5
