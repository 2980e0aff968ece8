"""CPU: networks with up to 256 classes get the tensor-core engine, and the many-class entry points validate their arguments
(class count, channel count, null pointers) before anything is launched. No compute calls (no GPU here)."""
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    g.build()
    from unet_torch_b200 import _lib

    return _lib


@pytest.mark.parametrize("cls_name", ["UNet", "UNet_multitask", "UNet_attention"])
def test_engine_routing_by_class_count(cls_name):
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    x = torch.zeros(1, 3, 32, 32)
    for c in (9, 21, 256):
        net = getattr(U, cls_name)(3, c)
        assert isinstance(net._engine_for(x), UNetEngine), (cls_name, c)
    net = getattr(U, cls_name)(3, 257)
    if cls_name == "UNet_multitask":  # tensor-core engine only: outside it the network refuses
        with pytest.raises(ValueError, match="n_classes <= 256"):
            net._engine_for(x)
        return
    assert isinstance(net._engine_for(x), GenericEngine)
    with pytest.raises(ValueError, match="n_classes <= 256"):
        net._get_engine()
    assert isinstance(getattr(U, cls_name)(3, 21).set_check_mode(True)._engine_for(x), GenericEngine)


def test_head_family_is_chosen_by_class_count():
    from unet_torch_b200 import ops

    assert ops._head("b200unet_head_fprop", 8) == "b200unet_head_fprop"
    assert ops._head("b200unet_head_fprop", 9) == "b200unet_head_many_fprop"
    assert ops._head("b200unet_head_bwd_workspace_floats", 21) == "b200unet_head_many_bwd_workspace_floats"
    assert ops._head("b200unet_head_density", 256) == "b200unet_head_many_density"


def test_many_class_entry_points_validate_before_launching(lib):
    p = 16  # any non-null address: validation fails before it could be dereferenced
    for ncls in (0, 257):
        cases = [
            ("b200unet_head_many_fprop", (p, 64, p, p, p, 1, 8, 8, 64, ncls, None)),
            ("b200unet_head_many_bwd", (p, p, 64, p, p, 64, p, p, p, 1, 8, 8, 64, ncls, None)),
            ("b200unet_head_many_mask", (p, 64, p, p, p, 1, 8, 8, 64, ncls, None)),
            ("b200unet_head_many_density", (p, 64, p, p, p, p, 1, 8, 8, 64, ncls, 200.0, None)),
        ]
        for name, args in cases:
            with pytest.raises(RuntimeError, match="n_classes"):
                lib.call(name, *args)
        assert lib.query("b200unet_head_many_bwd_workspace_floats", 1, 8, 8, 64, ncls) == 0
        assert lib.query("b200unet_loss_sums_doubles_n", ncls) == (0 if ncls == 0 else 1286 + 1184 * 772 + 1184 * 12 * 264)
    with pytest.raises(RuntimeError, match="null pointer"):
        lib.call("b200unet_head_many_fprop", None, 64, p, p, p, 1, 8, 8, 64, 21, None)
    with pytest.raises(RuntimeError, match="null pointer"):
        lib.call("b200unet_head_many_bwd", p, p, 64, p, None, 64, p, p, p, 1, 8, 8, 64, 21, None)
    with pytest.raises(RuntimeError, match="null pointer"):
        lib.call("b200unet_head_many_mask", p, 64, p, p, None, 1, 8, 8, 64, 21, None)
    with pytest.raises(RuntimeError, match="null pointer"):
        lib.call("b200unet_head_many_density", p, 64, p, None, p, None, 1, 8, 8, 64, 21, 200.0, None)
    with pytest.raises(RuntimeError, match="Cin=96"):
        lib.call("b200unet_head_many_fprop", p, 96, p, p, p, 1, 8, 8, 96, 21, None)
    with pytest.raises(RuntimeError, match="empty input"):
        lib.call("b200unet_head_many_mask", p, 64, p, p, p, 0, 8, 8, 64, 21, None)
    # the loss and the argmax take any class count >= 1
    with pytest.raises(RuntimeError, match="n_classes=0"):
        lib.call("b200unet_loss_ce_dice_fwd", p, p, p, p, p, 1, 0, 64, 0, None)
    with pytest.raises(RuntimeError, match="n_classes=0"):
        lib.call("b200unet_softmax_argmax", p, p, 1, 0, 64, None)


def test_loss_and_head_workspace_sizes(lib):
    # up to 8 classes the loss keeps its fixed layout; past 8: [CE, I, Z, Y] and the backward's coefficients [cN, cD] (the
    # prefix the backward reads), then one fp64 row per forward block (148 x 8) and 8 warps' fp32 rows of 3 x (classes
    # padded to 8) per block
    assert lib.query("b200unet_loss_sums_doubles_n", 1) == lib.query("b200unet_loss_sums_doubles")
    assert lib.query("b200unet_loss_sums_doubles_n", 8) == lib.query("b200unet_loss_sums_doubles") == 25 * 16
    assert lib.query("b200unet_loss_sums_doubles_n", 9) == 46 + 1184 * 28 + 1184 * 12 * 16
    assert lib.query("b200unet_loss_sums_doubles_n", 21) == 106 + 1184 * 64 + 1184 * 12 * 24
    assert lib.query("b200unet_loss_sums_saved_doubles_n", 8) == 25 * 16
    assert lib.query("b200unet_loss_sums_saved_doubles_n", 21) == 1 + 5 * 21
    # head backward: per pixel slice x 8-class chunk one block; partials [slices][padded classes][Cin + 1]
    assert lib.query("b200unet_head_many_bwd_workspace_floats", 16, 512, 512, 64, 21) == 198 * 24 * 65
    assert lib.query("b200unet_head_many_bwd_workspace_floats", 1, 16, 16, 64, 256) == 1 * 256 * 65
    assert lib.query("b200unet_head_many_bwd_workspace_floats", 16, 512, 512, 128, 256) == 19 * 256 * 129


def test_c_abi_keeps_the_eight_class_head_contract(lib):
    """b200unet_head_fprop still rejects 9 classes: the many-class heads are a separate family."""
    with pytest.raises(RuntimeError, match="n_classes=9 must be in \\[1,8\\]"):
        lib.call("b200unet_head_fprop", None, 64, None, None, None, 1, 8, 8, 64, 9, None)
