"""CPU: the host-side mirror of the reference interface (module tree / state_dict ABI / init RNG order / loss
dispatch) and the absence of any CPU fallback."""
import copy

import pytest
import torch


def checksum(v):
    f = v.double().flatten()
    return torch.tensor([f.sum(), f.abs().sum(), f[0], f[f.numel() // 2], f[-1]], dtype=torch.float64)


def test_state_dict_keys_shapes_and_init_match_reference(golden):
    import unet_torch_b200 as U

    for case, g in golden("ref_full_nets.pt").items():
        ch, ncls, width, n, h, w, seed = g["cfg"]
        torch.manual_seed(seed)
        net = U.UNet(ch, ncls, width)
        sd = net.state_dict()
        assert list(sd.keys()) == list(g["sd0_checksum"].keys()), case  # same keys, same order
        for k, v in sd.items():
            assert torch.allclose(checksum(v), g["sd0_checksum"][k], rtol=1e-12, atol=0), (case, k)
            assert v.dtype in (torch.float32, torch.int64)


def test_narrow_reference_checkpoint_loads(golden):
    import unet_torch_b200 as U

    g = golden("ref_small_nets.pt")["w4_c3_k5_dicebce"]
    net = U.UNet(3, 5, 4)
    missing = net.load_state_dict(g["sd0"], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    sd = copy.deepcopy(net.state_dict())  # Trainer.py:759 deep-copies the state_dict
    assert torch.equal(sd["outc.conv.weight"], g["sd0"]["outc.conv.weight"])


def test_constructor_contract():
    import unet_torch_b200 as U

    net = U.UNet(-2, 3, 64, True, False, 0.5)  # train.py:196-205 passes six positional arguments
    assert (net.n_channels, net.n_classes, net.initial_feature_map, net.usa_cuda, net.dropout, net.dropout_p) == (
        3, 3, 64, True, False, 0.5)
    assert U.UNet(-1, 2).n_channels == 1
    names = [n for n, _ in net.named_children()]
    assert names == ["inc", "down1", "down2", "down3", "down4", "up1", "up2", "up3", "up4", "outc"]
    d = U.UNet(3, 2, 64, True, True, 0.3)
    assert "down1.maxpool_conv.2.double_conv.0.weight" in d.state_dict()  # Dropout shifts the index (Model.py:34-39)


def test_no_cpu_fallback():
    import unet_torch_b200 as U

    net = U.UNet(3, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.randn(1, 3, 32, 32))
    with pytest.raises(RuntimeError, match="CUDA"):
        U.calc_loss(torch.randn(1, 2, 8, 8, requires_grad=True), torch.zeros(1, 8, 8), loss_type="dice_bce_mc")
    with pytest.raises(RuntimeError):
        net.inc(torch.randn(1, 3, 32, 32))  # blocks are parameter containers, not a torch fallback


def test_root_shims_mirror_reference_imports():
    import Model
    import loss
    import unet_torch_b200 as U

    assert Model.UNet is U.UNet
    loss.CLASS_NUMBER = 5  # train.py:163
    assert U.loss.CLASS_NUMBER == 5
    assert callable(loss.calc_loss) and loss.DiceLoss is U.DiceLoss
    assert Model.UNet_multitask is U.UNet_multitask and issubclass(Model.UNet_multitask, torch.nn.Module)
    assert Model.UNet_attention is U.UNet_attention and len(Model.UNet_attention(3, 2, 4).state_dict()) == 210
    assert isinstance(loss.MultitaskUncertaintyLoss(), torch.nn.Module) and callable(loss.MRAccuracy)  # Trainer.py:6
    with pytest.raises(NotImplementedError):
        loss.calc_loss(torch.zeros(1, 1, 4, 4), torch.zeros(1, 4, 4), loss_type="HausdorffDTLoss")


def test_multitask_module_mirrors_reference_layout():
    """UNet_multitask (Model.py:172-250): key names and order, parameter count, RNG consumption of the constructor."""
    import unet_torch_b200 as U

    torch.manual_seed(0)
    net = U.UNet_multitask(-2, 2, 8)
    keys = list(net.state_dict().keys())
    assert len(keys) == 176 and net.n_channels == 3
    assert keys[0] == "inc.double_conv.0.weight"
    order = [k.split(".")[0] for k in keys]
    first = {name: order.index(name) for name in ("down4", "up1_decod1", "outc_decod1", "up1_decod2", "outc_decod2")}
    assert first["down4"] < first["up1_decod1"] < first["outc_decod1"] < first["up1_decod2"] < first["outc_decod2"]
    assert net.up1_decod2.up.weight.shape == (128, 64, 2, 2) and net.outc_decod2.conv.weight.shape == (2, 8, 1, 1)
    # no Dropout layers are built whatever the flag says (Model.py:188-230 never pass it on)
    assert not any(isinstance(m, torch.nn.Dropout) for m in U.UNet_multitask(3, 2, 8, dropout=True).modules())
    # the two decoders draw different weights from the RNG stream
    assert not torch.equal(net.up1_decod1.up.weight, net.up1_decod2.up.weight)
    with pytest.raises(RuntimeError):
        net.inc(torch.zeros(1, 3, 16, 16))  # containers are not the product path


@pytest.mark.parametrize("cls_name,n_dec", [("UNet", 1), ("UNet_multitask", 2)])
def test_backward_order_covers_every_parameter_once(cls_name, n_dec):
    """The flat data-parallel gradient buffer is laid out in params_in_backward_order(): it must be a permutation of
    the module's parameters (both decoders of UNet_multitask included), heads first, encoder last."""
    import unet_torch_b200 as U

    net = getattr(U, cls_name)(3, 2)
    eng = net._get_engine()          # host-side bookkeeping only: no CUDA call until forward
    order = eng.params_in_backward_order()
    assert len(order) == len(list(net.parameters())) == len({id(p) for p in order})
    assert {id(p) for p in order} == {id(p) for p in net.parameters()}
    assert len(eng.decoders) == n_dec and len(eng.ups) == 4 * n_dec and len(eng.dec) == 4 * n_dec
    names = {id(p): n for n, p in net.named_parameters()}
    assert names[id(order[0])].startswith("outc") and names[id(order[-1])] == "inc.double_conv.0.weight"
    if n_dec == 2:  # the decoder that ran last in forward is differentiated first
        assert names[id(order[0])] == "outc_decod2.conv.weight"


def test_product_path_never_touches_the_oracle_or_a_cpu_fallback():
    """The oracle is test infrastructure: nothing under the package (or the root shims) may import or execute it, and
    importing the package must not pull it in as a side effect. bench.py may use it only in its CPU legs."""
    import ast
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = [os.path.join(root, "unet-torch_b200", f) for f in os.listdir(os.path.join(root, "unet-torch_b200")) if f.endswith(".py")]
    files += [os.path.join(root, f) for f in ("Model.py", "loss.py", "unet_torch_b200.py")]
    for path in files:
        tree = ast.parse(open(path).read())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            assert not any(n == "oracle" or n.startswith("oracle.") for n in names), f"{path} imports the oracle"
    code = "import sys; sys.path.insert(0, %r); import unet_torch_b200, Model, loss; print(any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules))" % root
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "False", (r.stdout, r.stderr[-500:])
    # bench.py: oracle use is confined to the CPU legs (cpu_baseline_leg / reference arm)
    bench = ast.parse(open(os.path.join(root, "bench.py")).read())
    for fn in [n for n in ast.walk(bench) if isinstance(n, ast.FunctionDef)]:
        uses = any(isinstance(n, (ast.Import, ast.ImportFrom)) and "oracle" in ast.dump(n) for n in ast.walk(fn))
        if uses:
            assert fn.name in ("cpu_baseline_leg", "reference_arm", "run_reference", "cpu_port_step") or "cpu" in fn.name or "reference" in fn.name, fn.name


def test_gate_weight_composition_algebra():
    """The rewrite the tensor-core engine applies to an attention gate (model.py `_GateOp`): ConvTranspose2d(C_q, C_q, 2, 2)
    followed by a 1x1 convolution (Model.py:287-288) equals ONE ConvTranspose2d with W'[c,h,i,j] = sum_d W_up[c,d,i,j] W_q[h,d],
    b' = b_q + W_q b_up, and the gradients of the four original tensors follow from (dW', db') by the formulas the engine's
    strided GEMMs evaluate. fp64 on the host against autograd through the reference's two-module form."""
    import torch
    import torch.nn.functional as F

    torch.manual_seed(0)
    cq, ch, n, h, w = 6, 3, 2, 4, 5
    q = torch.randn(n, cq, h, w, dtype=torch.float64)
    w_up = torch.randn(cq, cq, 2, 2, dtype=torch.float64, requires_grad=True)
    b_up = torch.randn(cq, dtype=torch.float64, requires_grad=True)
    w_q = torch.randn(ch, cq, 1, 1, dtype=torch.float64, requires_grad=True)
    b_q = torch.randn(ch, dtype=torch.float64, requires_grad=True)
    ref = F.conv2d(F.conv_transpose2d(q, w_up, b_up, stride=2), w_q, b_q)
    g = torch.randn_like(ref)
    (ref * g).sum().backward()
    wq2 = w_q.detach().view(ch, cq)
    wc = torch.einsum("cdij,hd->chij", w_up.detach(), wq2).requires_grad_(True)
    bc = (b_q.detach() + wq2 @ b_up.detach()).requires_grad_(True)
    out = F.conv_transpose2d(q, wc, bc, stride=2)
    assert torch.allclose(out, ref.detach(), rtol=1e-12, atol=1e-12)
    (out * g).sum().backward()
    assert torch.allclose(torch.einsum("chij,hd->cdij", wc.grad, wq2), w_up.grad, rtol=1e-12, atol=1e-12)
    # W_q enters W' AND b': the second path is the rank-one term db' (x) b_up (zero in expectation behind a train-mode BatchNorm,
    # not behind a frozen one)
    dwq = torch.einsum("chij,cdij->hd", wc.grad, w_up.detach()) + torch.outer(bc.grad, b_up.detach())
    assert torch.allclose(dwq, w_q.grad.view(ch, cq), rtol=1e-12, atol=1e-12)
    assert torch.allclose(wq2.t() @ bc.grad, b_up.grad, rtol=1e-12, atol=1e-12)
    assert torch.allclose(bc.grad, b_q.grad, rtol=1e-12, atol=1e-12)


def test_attention_engine_selection_and_parameter_coverage():
    """Which engine a UNet_attention gets (no CUDA needed to decide): the tensor-core engine at the reference's default width
    without dropout, the generic fp32 engine otherwise and in check mode; every parameter has a slot in the backward order
    (data-parallel flat gradient buffer); the gate holders see the reference's channel plan (Model.py:325-341)."""
    import torch

    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    x = torch.zeros(1, 3, 32, 32)
    net = U.UNet_attention(3, 2)
    eng = net._engine_for(x)
    assert isinstance(eng, UNetEngine) and len(eng.gates) == 4
    assert [(g.cq, g.cx, g.ch, g.chp) for g in eng.gates] == [(1024, 512, 256, 256), (512, 256, 128, 128), (256, 128, 64, 64),
                                                              (128, 64, 32, 64)]
    order = eng.params_in_backward_order()
    assert len(order) == len(set(order)) == len(list(net.parameters())) and set(order) == set(net.parameters())
    assert isinstance(net.set_check_mode(True)._engine_for(x), GenericEngine)
    for kw in (dict(initial_feature_map=128), dict(initial_feature_map=8), dict(dropout=True)):
        small = U.UNet_attention(3, 2, **{"initial_feature_map": 8, **kw}) if "dropout" in kw else U.UNet_attention(3, 2, **kw)
        assert isinstance(small._engine_for(x), GenericEngine), kw
    try:
        net._engine_for(torch.zeros(1, 3, 40, 40))
    except ValueError:
        pass
    else:
        raise AssertionError("UNet_attention must reject H, W not divisible by 16")
    # the plain UNet's engine has no gates; the two-decoder network can be captured as CUDA graphs now
    assert U.UNet(3, 2)._get_engine().gates is None
    assert U.UNet_multitask(3, 2).enable_cuda_graphs(True)._cuda_graphs is True


def test_profile_summaries_parse_the_committed_launch_lists():
    """scripts/launch_summary.py finds the step boundary (two launches of the fused first-layer kernel) in the committed ncu
    launch lists - the kernel names carry template arguments that have changed between rounds."""
    import os
    import subprocess
    import sys

    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name, launches in (("r2_launches.csv", 192), ("r2_attn_launches.csv", 298)):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "launch_summary.py"), os.path.join(ROOT, "profiles", name)],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr
        first = r.stdout.splitlines()[0]
        assert first.startswith("one step = launches") and f"{launches} launches" in first, first


def test_gate_checker_accepts_the_reference_and_flags_a_missing_term():
    """tests/gate_check.py (the one-operator-deep host check the GPU gate-replay test applies to the engine's trace) on records
    produced by an fp64 autograd run of the reference's gate: everything within 1e-9, in training and in frozen-BatchNorm mode;
    and it notices when dW_q lacks the rank-one term db' (x) b_up (only visible behind a frozen BatchNorm)."""
    import torch

    from gate_check import check_gate, gate_reference_run

    torch.manual_seed(0)
    cq, cx, ch, n, h, w = 6, 5, 4, 2, 6, 8
    r = lambda *s: torch.randn(*s, dtype=torch.float64)  # noqa: E731
    p = dict(W_up=r(cq, cq, 2, 2), b_up=r(cq), W_q=r(ch, cq, 1, 1), b_q=r(ch), W_x=r(ch, cx, 1, 1), b_x=r(ch), gq=r(ch).abs() + 0.5,
             bq=r(ch), gx=r(ch).abs() + 0.5, bx=r(ch), wpsi=r(ch), bpsi=r(1), gp=r(1).abs() + 0.5, bp=r(1))
    q, x, g = r(n, cq, h // 2, w // 2), r(n, cx, h, w), r(n, cx, h, w)
    stats = {"q": (r(ch), r(ch).abs() + 0.5), "x": (r(ch), r(ch).abs() + 0.5), "p": (r(1), r(1).abs() + 0.5)}
    for frozen in (False, True):
        rec = gate_reference_run(p, q, x, g, frozen=frozen, stats=stats)
        assert check_gate(rec, tol_map=1e-9, tol_sum=1e-9, tol_grad=1e-9) == [], frozen
    rec["grads"]["W_q"] = rec["grads"]["W_q"] - torch.outer(rec["grads"]["b_q"], p["b_up"]).view(ch, cq, 1, 1)
    assert [b[0] for b in check_gate(rec, tol_map=1e-9, tol_sum=1e-9, tol_grad=1e-9)] == ["dW_q"]


def test_conv_check_references_agree_with_torch():
    """tests/conv_check.py: the fp64 references of the exact convolution tests against F.conv2d / conv_transpose2d / autograd /
    torch.nn.grad.conv2d_weight on random fp64 data."""
    import torch.nn.functional as F

    import conv_check as C

    g = torch.Generator().manual_seed(3)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)  # noqa: E731
    x, w, dy = r(2, 5, 7, 6), r(4, 5, 3, 3), r(2, 4, 7, 6)
    xv = x.clone().requires_grad_(True)
    (F.conv2d(xv, w, padding=1) * dy).sum().backward()
    assert torch.allclose(C.conv3x3(x, w), F.conv2d(x, w, padding=1), rtol=1e-12, atol=1e-12)
    assert torch.allclose(C.conv3x3_dgrad(dy, w), xv.grad, rtol=1e-12, atol=1e-12)
    assert torch.allclose(C.conv3x3_wgrad(x, dy), torch.nn.grad.conv2d_weight(x, w.shape, dy, padding=1), rtol=1e-12, atol=1e-12)
    wt, b, du = r(5, 3, 2, 2), r(3), r(2, 3, 14, 12)
    xv = x.clone().requires_grad_(True)
    wv = wt.clone().requires_grad_(True)
    (F.conv_transpose2d(xv, wv, b, stride=2) * du).sum().backward()
    assert torch.allclose(C.convt2x2(x, wt, b), F.conv_transpose2d(x, wt, b, stride=2), rtol=1e-12, atol=1e-12)
    assert torch.allclose(C.convt2x2_dgrad(du, wt), xv.grad, rtol=1e-12, atol=1e-12)
    assert torch.allclose(C.convt2x2_wgrad(x, du), wv.grad, rtol=1e-12, atol=1e-12)
    w1, b1 = r(4, 5), r(4)
    assert torch.allclose(C.conv1x1(x, w1, b1), F.conv2d(x, w1[:, :, None, None], b1), rtol=1e-12, atol=1e-12)
    assert torch.allclose(C.conv1x1_wgrad(x, dy), torch.nn.grad.conv2d_weight(x, (4, 5, 1, 1), dy)[:, :, 0, 0], rtol=1e-12,
                          atol=1e-12)
    # eval BatchNorm + ReLU and the fused backward reduction, against autograd of the same module in fp64
    y, sc, sh, mean, rstd = r(2, 4, 7, 6), r(4), r(4), r(4), r(4).abs()
    assert torch.equal(C.bn_relu_eval(y, sc, sh), torch.relu(y * sc.view(1, -1, 1, 1) + sh.view(1, -1, 1, 1)))
    beta = r(4)
    bv = beta.clone().requires_grad_(True)
    gv = torch.ones(4, dtype=torch.float64, requires_grad=True)
    xhat = (y - mean.view(1, -1, 1, 1)) * rstd.view(1, -1, 1, 1)
    (torch.relu(gv.view(1, -1, 1, 1) * xhat + bv.view(1, -1, 1, 1)) * dy).sum().backward()
    s1, s2 = C.bn_backward_sums(dy, y, rstd, beta - mean * rstd, mean, rstd)
    assert torch.allclose(s1, bv.grad, rtol=1e-10, atol=1e-10) and torch.allclose(s2, gv.grad, rtol=1e-10, atol=1e-10)


def _emulate_fp32_conv(x, w, orders, gen):
    """An fp32 conv3x3 that accumulates its K = 9 * Cin products one at a time, in a shuffled order and split into K blocks whose
    fp32 partials are added at the end (like a split-K kernel), then rounds to bf16 nearest-even."""
    import torch.nn.functional as F

    import conv_check as C

    n, c, h, wd = x.shape
    cols = F.unfold(x.float(), 3, padding=1).view(n, c * 9, h * wd)              # [n, K, P]
    prods = cols[:, :, None, :] * w.float().view(w.shape[0], -1).t()[None, :, :, None]  # [n, K, Cout, P], exact
    outs = []
    for nsplit in orders:
        perm = torch.randperm(c * 9, generator=gen)
        parts = []
        for chunk in perm.chunk(nsplit):
            acc = torch.zeros(n, w.shape[0], h * wd)
            for k in chunk.tolist():
                acc = acc + prods[:, k]
            parts.append(acc)
        tot = parts[0]
        for p in parts[1:]:
            tot = tot + p
        outs.append(C.bf16_rne(tot.view(n, -1, h, wd)).double())
    return outs


@pytest.mark.parametrize("regime", ["sparse", "dense"])
def test_conv_check_exactness_holds_under_any_summation_order(regime):
    """The argument behind the exact GPU tests: under each regime's invariant, an fp32 accumulation in any order and any K split
    rounds to bf16_rne(exact fp64) bit for bit."""
    import conv_check as C

    g = torch.Generator().manual_seed(7 if regime == "sparse" else 8)
    x = C.operand((2, 64, 10, 12), regime, 9 * 64, g)
    w = C.operand((64, 64, 3, 3), regime, 9 * 64, g, sparse_input=False)
    y = C.conv3x3(x, w)
    C.check_regime(regime, y, C.conv3x3(x.abs(), w.abs()))
    for got in _emulate_fp32_conv(x, w, (1, 3, 8), g):
        C.assert_exact(C.nhwc(got), C.nhwc(C.bf16_rne(y)))


def test_conv_check_flags_the_defects_rel_l2_accepts():
    """Dense case N = 4, 160 x 160, 64 -> 64 (m = 12). A dropped tap on one edge pixel, one pixel written with its neighbour's
    values and round-toward-zero instead of nearest-even all pass the old `rel_l2 < 1e-2` comparison and all fail
    assert_exact; so do a statistics row left unwritten and an element written into the guard image."""
    import torch.nn.functional as F

    import conv_check as C

    g = torch.Generator().manual_seed(9)
    n, c, h, w = 4, 64, 160, 160
    assert C.dense_m(9 * c) == 12
    x = C.operand((n, c, h, w), C.DENSE, 9 * c, g)
    wt = C.operand((c, c, 3, 3), C.DENSE, 9 * c, g, sparse_input=False)
    y = C.conv3x3(x, wt)
    C.check_regime(C.DENSE, y, C.conv3x3(x.abs(), wt.abs()))
    want = C.nhwc(C.bf16_rne(y))
    C.assert_exact(want, want)
    # one tap (r = s = 0) missing on the bottom-right pixel of image 0, all channels
    dropped = y.clone()
    tap = (x[0, :, h - 2, w - 2][None, :] * wt[:, :, 0, 0]).sum(1)
    dropped[0, :, h - 1, w - 1] -= tap
    # pixel (5, 3) of image 1 holds pixel (5, 4)'s channels
    moved = C.bf16_rne(y)
    moved[1, :, 5, 3] = moved[1, :, 5, 4]
    defects = {"dropped tap": C.nhwc(C.bf16_rne(dropped)), "neighbour pixel": C.nhwc(moved), "round toward zero":
               C.nhwc(C.bf16_rz(y))}
    for what, got in defects.items():
        err = C.rel_l2(got, want)
        assert err < 1e-2, (what, err)                     # the old metric accepts it ...
        with pytest.raises(AssertionError, match="elements differ"):
            C.assert_exact(got, want, what)                # ... the exact comparison does not
    with pytest.raises(AssertionError, match=r"differ\n  \(n=0, h=159, w=159, c=\d+\).*image 0, 16x8 tile 199, 8x16 tile 199"):
        C.assert_exact(defects["dropped tap"], want)
    # statistics: one row left as its NaN sentinel
    rows = 7
    st = C.stats_buffer(rows, c, device="cpu")
    st.view(rows + 1, 2 * c)[:rows] = 1.0
    C.assert_stats_rows(st, rows, c)
    st.view(rows + 1, 2 * c)[3] = C.stats_buffer(0, c, device="cpu").view(1, 2 * c)
    with pytest.raises(AssertionError, match=r"rows \[3\]"):
        C.assert_stats_rows(st, rows, c)
    # output canvas: one element written into the guard image after the last one
    canvas, target = C.bf16_canvas(2, 3, 5, c, device="cpu")
    target.copy_(torch.zeros(2, 3, 5, c))
    C.assert_canvas_intact(canvas, 2, c)
    canvas[2, 1, 1, C.GUARD_C + 4] = 0.0
    with pytest.raises(AssertionError, match="1 elements outside the target"):
        C.assert_canvas_intact(canvas, 2, c)
    # and an input canvas carries NaN into a convolution that reads past its slice
    xcan, xs = C.input_canvas(torch.ones(1, 3, 5, 8), device="cpu")
    wide = C.nhwc(F.conv2d(C.nchw(xcan[:1, :, :, C.GUARD_C - 1:C.GUARD_C + 8].double()), torch.ones(1, 9, 3, 3, dtype=torch.float64),
                           padding=1))
    assert bool(torch.isnan(wide).all()) and torch.equal(xs.double(), torch.ones(1, 3, 5, 8, dtype=torch.float64))


def test_conv_check_recorder_reads_profiler_names():
    import conv_check as C

    assert C.kernel_name("void (anonymous namespace)::conv3_pair_kernel<256, 2, 6, 1>((anonymous namespace)::PairArgs)") == \
        "conv3_pair_kernel<256, 2, 6, 1>"
    assert C.kernel_name("void (anonymous namespace)::conv3_res_kernel<64, 1, 3, 2, 9, 0, 0, true>((anonymous namespace)::ResArgs)") \
        == "conv3_res_kernel<64, 1, 3, 2, 9, 0, 0, true>"
    assert C.kernel_name("(anonymous namespace)::wgrad_swap3_kernel((anonymous namespace)::WgradArgs)") == "wgrad_swap3_kernel"


def test_bench_dump_outputs_samples_each_array_by_its_own_size_within_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: an array longer than the per-array cap is cut to a fixed seeded sample that depends only on
    its own size (identical from run to run, and when other arrays come or go, so two builds compare element for
    element); shorter arrays are written whole; fp64 / integer data stay exact; a dump over the byte budget is refused."""
    import os

    import numpy as np

    import bench

    monkeypatch.setattr(bench, "DUMP_ELEMS", 5000)
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": torch.tensor(0.25), "output": torch.randn(4, 2, 64, 64, generator=g).bfloat16(),
              "grad.w": torch.randn(64, 32, 3, 3, generator=g), "state.b": torch.randn(7, generator=g).double(),
              "state.n": torch.tensor(12345678901, dtype=torch.int64)}
    dumps = []
    for run, names in (("a", list(arrays)), ("b", list(arrays)), ("c", ["grad.w"])):
        nbytes, sampled = bench.dump_outputs(str(tmp_path / run), {k: arrays[k] for k in names})
        files = sorted(os.listdir(tmp_path / run))
        assert files == sorted(k + ".npy" for k in names) and sorted(sampled) == [k for k in ("grad.w", "output") if k in names]
        assert sum(os.path.getsize(tmp_path / run / f) for f in files) <= nbytes <= bench.DUMP_BYTES
        dumps.append({k: np.load(tmp_path / run / (k + ".npy")) for k in names})
    a, b, c = dumps
    assert all(np.array_equal(a[k], b[k]) for k in arrays) and np.array_equal(a["grad.w"], c["grad.w"])
    assert a["output"].dtype == np.float32 and a["state.b"].dtype == np.float64 and int(a["state.n"]) == 12345678901
    assert np.array_equal(a["state.b"], arrays["state.b"].numpy()) and float(a["loss"]) == 0.25
    w = arrays["grad.w"].flatten().numpy()
    assert a["grad.w"].size == a["output"].size == 5000 and np.isin(a["grad.w"], w).all()
    monkeypatch.setattr(bench, "DUMP_BYTES", 30_000)
    with pytest.raises(RuntimeError, match="dump-outputs"):
        bench.dump_outputs(str(tmp_path / "d"), arrays)


def _f32_of_fraction(q):
    """Round an exact rational to fp32, nearest-even (subnormals included), as a Python float."""
    import math
    from fractions import Fraction

    if q == 0:
        return 0.0
    sign, q = (-1 if q < 0 else 1), abs(q)
    e = q.numerator.bit_length() - q.denominator.bit_length()
    while Fraction(2) ** e > q:
        e -= 1
    while Fraction(2) ** (e + 1) <= q:
        e += 1
    ulp = Fraction(2) ** (max(e, -126) - 23)
    m = q / ulp
    fl = math.floor(m)
    if m - fl > Fraction(1, 2) or (m - fl == Fraction(1, 2) and fl % 2 == 1):
        fl += 1
    return sign * float(fl * ulp)


def test_ew_check_fmaf_is_exact():
    """tests/ew_check.py: the fp64 emulation of fmaf equals exact rational arithmetic rounded once to fp32, on random fp32 x bf16
    and fp32 x fp32 operands and on the constructed fp32-midpoint cases, which must all take the double-rounding branch. There,
    rounding the fp64 sum to fp32 directly is wrong in one direction of the error term, and the forward's bf16 output tells
    the two results apart."""
    from fractions import Fraction

    import ew_check as E

    assert all(a * b == 2 ** 30 + rho and a < 2 ** 24 and b % 2 == 1 and b < 256 for a, b, rho in E.MIDPOINT_PRODUCTS)
    g = torch.Generator().manual_seed(11)
    n = 1500
    sc = (torch.randn(n, generator=g, dtype=torch.float64) * torch.exp2(torch.randint(-30, 30, (n,), generator=g))).float()
    y = (torch.randn(n, generator=g, dtype=torch.float64) * torch.exp2(torch.randint(-30, 30, (n,), generator=g))).bfloat16()
    sh = (torch.randn(n, generator=g, dtype=torch.float64) * torch.exp2(torch.randint(-30, 30, (n,), generator=g))).float()
    fb = torch.randn(n, generator=g).float()
    cases = [(sc, y.float()), (sc, fb)]
    mids = [E.midpoint_case(i, hb, j) for i in range(8) for hb in (0, 5, 63) for j in (-3, 0, 3)]
    msc, my, msh = (torch.tensor(v, dtype=torch.float32) for v in zip(*mids))
    assert torch.equal(my.bfloat16().float(), my)
    for a, b in cases + [(msc, my)]:
        c = sh[: a.numel()] if a.numel() == n else msh
        got, mid = E.fmaf(a, b, c)
        want = [_f32_of_fraction(Fraction(float(x)) * Fraction(float(z)) + Fraction(float(w))) for x, z, w in zip(a, b, c)]
        assert got.tolist() == want
    got, mid = E.fmaf(msc, my, msh)
    assert bool(mid.all()), "a constructed midpoint case missed the double-rounding branch"
    naive = (msc.double() * my.double() + msh.double()).float().double()
    rho = torch.tensor([E.MIDPOINT_PRODUCTS[i][2] for i in range(8) for _ in range(9)])
    assert bool((naive != got).all()), "rounding the fp64 sum to fp32 directly must get every constructed case wrong"
    assert bool((naive.float().bfloat16() != got.float().bfloat16()).all()), "the branch must be visible in bf16"


def test_ew_check_references_agree_with_autograd():
    """tests/ew_check.py: the backward formulas (dgamma, dbeta and the k1..k3 form of dy) equal autograd through BatchNorm with
    batch statistics + ReLU (+ MaxPool2d) in fp64; the pooling reference equals max_pool2d's indices; unpool equals autograd's
    gradient through the pool."""
    import torch.nn.functional as F

    import ew_check as E

    g = torch.Generator().manual_seed(12)
    n, c, h, w = 2, 5, 6, 8
    y = torch.randn(n, h, w, c, generator=g, dtype=torch.float64) * 2 + 0.5
    gamma, beta = torch.randn(c, generator=g, dtype=torch.float64), torch.randn(c, generator=g, dtype=torch.float64)
    g1 = torch.randn(n, h, w, c, generator=g, dtype=torch.float64)
    gp = torch.randn(n, h // 2, w // 2, c, generator=g, dtype=torch.float64)
    mean = y.mean((0, 1, 2))
    rstd = (y.var((0, 1, 2), unbiased=False) + 1e-5).rsqrt()
    yv, gv, bv = (t.clone().requires_grad_(True) for t in (y, gamma, beta))
    m_, r_ = yv.mean((0, 1, 2)), (yv.var((0, 1, 2), unbiased=False) + 1e-5).rsqrt()
    a = torch.relu((yv - m_) * r_ * gv + bv)
    pooled, flat = F.max_pool2d(a.permute(0, 3, 1, 2), 2, return_indices=True)
    ((a * g1).sum() + (pooled.permute(0, 2, 3, 1) * gp).sum()).backward()
    ad = a.detach()
    pv, idx = E.maxpool2x2(ad.float().to(torch.bfloat16))
    k = idx.permute(0, 3, 1, 2).long()
    hp, wp = torch.arange(h // 2).view(1, 1, -1, 1), torch.arange(w // 2).view(1, 1, 1, -1)
    assert torch.equal((2 * hp + k // 2) * w + (2 * wp + k % 2), flat)   # no ties in bf16 here: same windows
    da = torch.where(ad > 0, g1 + E.unpool(gp, idx, h, w), 0.0)
    sums = E.bwd_sums(da, y)
    dgamma, dbeta = E.param_grads(sums, mean, rstd)
    assert torch.allclose(dgamma, gv.grad, rtol=1e-10, atol=1e-10) and torch.allclose(dbeta, bv.grad, rtol=1e-10, atol=1e-10)
    dy, mag = E.dy_ref(da, y, gamma, mean, rstd, torch.stack([dbeta, dgamma]), n * h * w)
    assert torch.allclose(dy, yv.grad, rtol=1e-9, atol=1e-9) and bool((mag >= dy.abs() * (1 - 1e-12)).all())
    # grid formulas: config 2, level 0 (16 x 512 x 512 x 64): 443 pixels per backward thread, 1772 when pooled
    assert E.grid("bwd", E.work_items(16, 512, 512, 64, False)) == (296, 75776)
    assert E.terms_per_thread(16, 512, 512, 64, False) == 443 and E.terms_per_thread(16, 512, 512, 64, True) == 444
    assert E.grid("fwd", 7) == (1, 256) and E.grid("ew", 10 ** 9) == (1184, 303104)


def test_ew_check_flags_the_defects_rel_l2_accepts():
    """A one-ulp error in one activation, a swapped tie position, a sum that dropped its last item and one overwritten
    sentinel all pass the rel-L2 checks the BatchNorm+ReLU kernels used to have (4e-3 activations, 1e-2 dy, 2e-3 dgamma /
    dbeta) and all fail tests/ew_check.py's comparisons."""
    import conv_check as C
    import ew_check as E

    g = torch.Generator().manual_seed(13)
    n, h, w, c = 4, 32, 32, 64
    y = (torch.randn(n, h, w, c, generator=g) * 1.7 + 0.3).bfloat16()
    y[:, 0::2, 1::2] = y[:, 0::2, 0::2]                      # a tie in every window (positions 0 and 1)
    scale, shift = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.2
    a, pre, _ = E.bn_relu_fwd(y, scale, shift)
    # one ulp in one activation
    bad = a.clone()
    i = tuple((a > 0).nonzero()[100].tolist())
    bad.view(torch.int16)[i] += 1
    assert bad[i] != a[i] and C.rel_l2(bad, a) < 4e-3
    with pytest.raises(AssertionError, match="1 of"):
        E.assert_equal(bad, a, "activation")
    # a tie resolved to the later position
    pv, idx = E.maxpool2x2(a)
    tied = (a[:, 0::2, 0::2] == a[:, 0::2, 1::2]) & (idx == 0) & (a[:, 0::2, 0::2] > 0)
    i = tuple(tied.nonzero()[0].tolist())
    swapped = idx.clone()
    swapped[i] = 1
    with pytest.raises(AssertionError, match="1 of"):
        E.assert_equal(swapped, idx, "pool_idx")
    g1 = (torch.randn(n, h, w, c, generator=g) * 0.5 + 1).bfloat16()   # sums that do not cancel: the old relative check
    gp = (torch.randn(n, h // 2, w // 2, c, generator=g) * 0.5 + 1).bfloat16()  # is at its most sensitive
    gamma = torch.rand(c, generator=g) + 0.5
    mean, rstd = y.double().mean((0, 1, 2)).float(), (y.double().var((0, 1, 2)) + 1e-5).rsqrt().float()
    count = n * h * w
    da = E.bwd_da(y, g1, gp, idx, scale, shift)
    sums = E.bwd_sums(da, y)
    dgamma, dbeta = E.param_grads(sums, mean, rstd)
    want, mag = E.dy_ref(da, y, gamma, mean, rstd, torch.stack([dbeta, dgamma]), count)
    bound = E.dy_bound(want, mag, y, gamma, mean, rstd, count)
    assert E.assert_within(E.to_bf16(want), want, bound, "dy") <= 1.0
    da_s = E.bwd_da(y, g1, gp, swapped, scale, shift)
    got, _ = E.dy_ref(da_s, y, gamma, mean, rstd, torch.stack([dbeta, dgamma]), count)
    assert C.rel_l2(E.to_bf16(got), want) < 1e-2
    with pytest.raises(AssertionError, match="outside the bound"):
        E.assert_within(E.to_bf16(got), want, bound, "dy")
    # the last pixel dropped from the sums (all channels)
    k = E.terms_per_thread(n, h, w, c, True)
    bg, bb = E.sum_bounds(sums, mean, rstd, k)
    short = E.bwd_sums(da.reshape(-1, c)[:-1], y.reshape(-1, c)[:-1])
    sg, sb = E.param_grads(short, mean, rstd)
    assert C.rel_l2(sg, dgamma) < 2e-3 and C.rel_l2(sb, dbeta) < 2e-3
    for got_, want_, b_, what in ((sg, dgamma, bg, "dgamma"), (sb, dbeta, bb, "dbeta")):
        E.assert_within(want_.float(), want_, b_, what)
        with pytest.raises(AssertionError, match="outside the bound"):
            E.assert_within(got_.float(), want_, b_, what)
    # sentinels: one element past a contiguous output, one in the other half of a concat canvas, one position byte unwritten
    buf, view = E.guarded((2, 3, 4, 64), torch.bfloat16, device="cpu")
    view.zero_()
    E.assert_guard(buf, view.numel(), "pooled")
    buf[view.numel() + 5] = 0.0
    with pytest.raises(AssertionError, match="1 elements written past the end"):
        E.assert_guard(buf, view.numel(), "pooled")
    ibuf, iview = E.guarded((2, 3, 4, 64), torch.uint8, device="cpu")
    iview.fill_(3)
    E.assert_guard(ibuf, iview.numel(), "pool_idx")
    ibuf[17] = E.U8_SENTINEL
    with pytest.raises(AssertionError, match="1 elements left unwritten"):
        E.assert_guard(ibuf, iview.numel(), "pool_idx")
    cv, left = E.canvas2(1, 2, 2, 64, device="cpu")
    left.zero_()
    E.assert_right_half(cv, "a")
    cv[0, 1, 0, 64 + 9] = 1.0
    with pytest.raises(AssertionError, match="1 elements of the other half"):
        E.assert_right_half(cv, "a")
