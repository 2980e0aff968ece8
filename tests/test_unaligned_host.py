"""CPU: which engine runs an input whose H or W is not a multiple of 16, with and without `allow_unaligned_sizes()`, and the
argument checks of the floor-mode and pad-strip entry points (before anything is launched). No compute calls."""
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    g.build()
    from unet_torch_b200 import _lib

    return _lib


def _x(h, w):
    return torch.zeros(1, 3, h, w)


def test_routing_without_the_flag_is_unchanged():
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    net = U.UNet(3, 2)
    assert isinstance(net._engine_for(_x(32, 48)), UNetEngine)
    for h, w in ((17, 16), (97, 131), (30, 30), (40, 56)):
        assert isinstance(net._engine_for(_x(h, w)), GenericEngine)
        with pytest.raises(ValueError, match="multiples of 16"):
            U.UNet_multitask(3, 2)._engine_for(_x(h, w))
        with pytest.raises(ValueError, match="fused inference heads"):
            net.predict(_x(h, w))
    with pytest.raises(ValueError, match="multiple of 16"):
        U.predict_tiled(net.eval(), torch.zeros(100, 100, 3, dtype=torch.uint8).numpy(), 50)


@pytest.mark.parametrize("cls_name", ["UNet", "UNet_multitask"])
def test_routing_with_the_flag(cls_name):
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    cls = getattr(U, cls_name)
    net = cls(3, 2)
    assert net.allow_unaligned_sizes() is net
    for h, w in ((17, 16), (97, 131), (30, 30), (32, 48), (16, 16)):
        assert isinstance(net._engine_for(_x(h, w)), UNetEngine), (h, w)
    for h, w in ((15, 64), (64, 15), (8, 8)):
        with pytest.raises(ValueError, match=">= 16"):
            net._engine_for(_x(h, w))
    assert net.allow_unaligned_sizes(False) is net
    if cls_name == "UNet":
        assert isinstance(net._engine_for(_x(97, 131)), GenericEngine)
        # check mode and architectures outside the tensor-core envelope keep the generic engine
        assert isinstance(cls(3, 2).allow_unaligned_sizes().set_check_mode(True)._engine_for(_x(97, 131)), GenericEngine)
        assert isinstance(cls(3, 2, 32).allow_unaligned_sizes()._engine_for(_x(97, 131)), GenericEngine)
        assert isinstance(cls(3, 300).allow_unaligned_sizes()._engine_for(_x(97, 131)), GenericEngine)
    else:
        with pytest.raises(ValueError, match="multiples of 16"):
            net._engine_for(_x(97, 131))
        with pytest.raises(ValueError):
            cls(3, 2, 32).allow_unaligned_sizes()._engine_for(_x(97, 131))


def test_attention_keeps_rejecting_unaligned_sizes():
    import unet_torch_b200 as U

    net = U.UNet_attention(3, 2).allow_unaligned_sizes()
    for h, w in ((17, 16), (97, 131), (30, 30)):
        with pytest.raises(ValueError, match="divisible by 16"):
            net._engine_for(_x(h, w))


def test_floor_entry_points_validate_before_launch(lib):
    p = 16   # any non-null address: validation fails before it could be dereferenced
    launches = lib.query("b200unet_launch_count")

    def fwd(pooled, idx, h, w, c=64, y_cs=64, a_cs=128):
        lib.call("b200unet_bn_relu_fwd_floor", p, y_cs, p, p, p, a_cs, pooled, idx, 1, h, w, c, None)

    def reduce_rows(g1, g_pool, idx, h, w, c=64, y_cs=64, g1_cs=128):
        lib.call("b200unet_bn_relu_bwd_reduce_rows_floor", g1, g1_cs, g_pool, idx, p, y_cs, p, p, p, p, p, p, 1, h, w, c, None)

    def reduce(g1, g_pool, idx, h, w, c=64, y_cs=64, g1_cs=128):
        lib.call("b200unet_bn_relu_bwd_reduce_floor", g1, g1_cs, g_pool, idx, p, y_cs, p, p, p, p, p, p, 1, h, w, c, None)

    def apply(g1, g_pool, idx, h, w, c=64, y_cs=64, g1_cs=128):
        lib.call("b200unet_bn_relu_bwd_apply_floor", g1, g1_cs, g_pool, idx, p, y_cs, p, p, p, p, p, p, 8.0, None, p, y_cs, p, p,
                 1, h, w, c, None)

    with pytest.raises(RuntimeError, match="bn_relu_fwd_floor.*at least 2x2"):
        fwd(p, p, 1, 5)
    with pytest.raises(RuntimeError, match="bn_relu_fwd_floor.*at least 2x2"):
        fwd(p, None, 7, 1)
    with pytest.raises(RuntimeError, match="pool_idx without pooled"):
        fwd(None, p, 7, 5)
    with pytest.raises(RuntimeError, match="power of two"):
        fwd(p, p, 7, 5, c=96, y_cs=96, a_cs=192)
    with pytest.raises(RuntimeError, match="pitches"):
        fwd(p, p, 7, 5, y_cs=60)
    with pytest.raises(RuntimeError, match="pitches"):
        fwd(p, p, 7, 5, a_cs=32)
    with pytest.raises(RuntimeError, match="empty map"):
        fwd(None, None, 0, 5)
    for fn, name in ((reduce_rows, "bn_relu_bwd_reduce"), (reduce, "bn_relu_bwd_reduce"), (apply, "bn_relu_bwd_apply")):
        with pytest.raises(RuntimeError, match=rf"{name}_floor\(pool\): a pooled gradient needs pool_idx"):
            fn(p, p, None, 7, 5)
        with pytest.raises(RuntimeError, match=rf"{name}_floor\(pool\).*at least 2x2"):
            fn(p, p, p, 1, 5)
        with pytest.raises(RuntimeError, match=rf"{name}_floor\(pool\).*at least 2x2"):
            fn(None, p, p, 9, 1)
        with pytest.raises(RuntimeError, match="power of two"):
            fn(p, p, p, 7, 5, c=96, y_cs=96, g1_cs=192)
        with pytest.raises(RuntimeError, match="pitches"):
            fn(p, p, p, 7, 5, y_cs=32)
        with pytest.raises(RuntimeError, match="pitches"):
            fn(p, p, p, 7, 5, g1_cs=36)
        with pytest.raises(RuntimeError, match="no gradient source"):
            fn(None, None, None, 7, 5)
    with pytest.raises(RuntimeError, match="maxpool2x2_fwd: .*at least 2x2"):
        lib.call("b200unet_maxpool2x2_fwd_floor", p, 64, p, 64, p, 1, 1, 9, 64, None)
    with pytest.raises(RuntimeError, match="maxpool2x2_fwd: C=64 and the pitches"):
        lib.call("b200unet_maxpool2x2_fwd_floor", p, 64, p, 60, p, 1, 7, 9, 64, None)
    with pytest.raises(RuntimeError, match="null argument"):
        lib.call("b200unet_maxpool2x2_fwd_floor", p, 64, None, 64, None, 1, 7, 9, 64, None)
    assert lib.query("b200unet_launch_count") == launches


def test_the_even_only_entry_points_still_refuse_odd_maps(lib):
    p = 16
    launches = lib.query("b200unet_launch_count")
    with pytest.raises(RuntimeError, match=r"bn_relu_fwd\(pool\): H=7 W=4 must be even"):
        lib.call("b200unet_bn_relu_fwd", p, 64, p, p, p, 64, p, p, 1, 7, 4, 64, None)
    with pytest.raises(RuntimeError, match="must be even"):
        lib.call("b200unet_maxpool2x2_fwd", p, 64, p, 64, p, 1, 7, 4, 64, None)
    assert lib.query("b200unet_launch_count") == launches


def test_pad_strip_entry_points_validate_before_launch(lib):
    p = 16
    launches = lib.query("b200unet_launch_count")
    for name, extra in (("b200unet_pad_strip_zero", ()), ("b200unet_pad_strip_sub_colsum", (p,))):
        short = name[len("b200unet_"):]
        with pytest.raises(RuntimeError, match=f"{short}: null tensor"):
            lib.call(name, None, 64, 1, 7, 5, 64, *extra, None)
        with pytest.raises(RuntimeError, match=f"{short}: empty map"):
            lib.call(name, p, 64, 1, 0, 5, 64, *extra, None)
        with pytest.raises(RuntimeError, match=f"{short}: C=60 and the pixel pitch"):
            lib.call(name, p, 64, 1, 7, 5, 60, *extra, None)
        with pytest.raises(RuntimeError, match=f"{short}: C=64 and the pixel pitch 32"):
            lib.call(name, p, 32, 1, 7, 5, 64, *extra, None)
        with pytest.raises(RuntimeError, match=f"{short}: the slice must start on a 16-byte boundary"):
            lib.call(name, 8, 64, 1, 7, 5, 64, *extra, None)
    with pytest.raises(RuntimeError, match="pad_strip_sub_colsum: null out"):
        lib.call("b200unet_pad_strip_sub_colsum", p, 64, 1, 7, 5, 64, None, None)
    # even H and W: the strip is empty and nothing is launched (no device memory is touched either)
    lib.call("b200unet_pad_strip_zero", p, 64, 1, 8, 6, 64, None)
    lib.call("b200unet_pad_strip_sub_colsum", p, 64, 1, 8, 6, 64, p, None)
    assert lib.query("b200unet_launch_count") == launches


def test_backward_workspace_holds_the_pad_strip_rows(lib):
    """A floor-mode pooled reduce at an odd H or W runs two launches of up to 148 x 8 blocks each (the pooled windows, then
    the pad strip), each writing one row of 2C partial sums per block."""
    rows = 148 * 8
    for c in (64, 1024):
        assert lib.query("b200unet_bn_bwd_workspace_floats", 16, 512, 512, c) == rows * 2 * c
        for h, w in ((125, 125), (124, 125), (125, 124)):
            assert lib.query("b200unet_bn_bwd_workspace_floats", 16, h, w, c) == 2 * rows * 2 * c
