"""CPU: the dropout mask contract (DESIGN.md §4) as oracle/philox.py states it, the host-side threshold / scale, argument
validation of the dropout entry points, and which engine a dropout network gets. No compute calls (no GPU here)."""
import numpy as np
import pytest
import torch

from oracle import philox as PX


def test_philox_known_answers():
    """Random123's known-answer vectors for Philox4x32-10."""
    def run(ctr, key):
        return [int(v) for v in PX.philox4x32_10(ctr, key)]

    assert run([0, 0, 0, 0], [0, 0]) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    f = 0xFFFFFFFF
    assert run([f, f, f, f], [f, f]) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert run([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == [
        0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_mask_is_a_function_of_seed_site_and_element():
    """A channel slice of a site (also one starting at e % 4 != 0) sees exactly the site mask's channels; element e uses
    word e % 4 of the Philox call with counter (e / 4, site); site and seed (both key words) change the mask."""
    shape = (2, 3, 5, 26)
    full = PX.keep_mask(1234, 5, shape, 0.4)
    assert np.array_equal(PX.keep_mask(1234, 5, shape, 0.4, c_lo=6, nc=8), full[..., 6:14])
    assert np.array_equal(PX.keep_mask(1234, 5, shape, 0.4, c_lo=3, nc=16), full[..., 3:19])
    t, _ = PX.threshold_scale(0.4)
    for e in (0, 7, 26 * 7 + 5, 2 * 3 * 5 * 26 - 1):
        w = PX.philox4x32_10((e // 4, 0, 5, 0), (1234, 0))
        assert bool(full.reshape(-1)[e]) == bool(int(w[e % 4]) < t)
    assert not np.array_equal(PX.keep_mask(1234, 4, shape, 0.4), full)
    assert not np.array_equal(PX.keep_mask(1235, 5, shape, 0.4), full)
    assert not np.array_equal(PX.keep_mask(1234 + (1 << 32), 5, shape, 0.4), full)


@pytest.mark.parametrize("p", [0.0, 0.1, 0.3, 0.5, 0.999, 1.0])
def test_threshold_and_scale(p):
    from unet_torch_b200 import ops

    t, s = ops.dropout_threshold_scale(p)
    assert (t, s) == PX.threshold_scale(p)
    if p == 1.0:
        assert (t, s) == (0, 0.0)
    else:
        assert t == min(2 ** 32 - 1, int(np.floor((1 - p) * 2.0 ** 32)))
        assert s == float(np.float32(1 / (1 - p)))
    with pytest.raises(ValueError):
        ops.dropout_threshold_scale(1.5)


def test_keep_fraction_of_the_oracle():
    keep = PX.keep_mask(99, 3, (4, 16, 16, 96), 0.3)
    n = keep.size
    sigma = (0.3 * 0.7 / n) ** 0.5
    assert abs(keep.mean() - 0.7) < 5 * sigma


def test_dropout_entry_points_validate_before_launching():
    import __graft_entry__ as g

    g.build()
    from unet_torch_b200 import _lib

    assert _lib.query("b200unet_dropout_partial_rows", 16, 512, 512, 128) == 148 * 8
    assert _lib.query("b200unet_dropout_partial_rows", 1, 1, 3, 64) == 1          # 8 groups -> 32 pixels per block
    assert _lib.query("b200unet_dropout_partial_rows", 1, 1, 100, 64) == 4
    assert _lib.query("b200unet_dropout_partial_rows", 1, 1, 1, 12) == 0          # not a multiple of 8
    with pytest.raises(RuntimeError, match="multiples of 8"):
        _lib.call("b200unet_dropout_mul", 16, 64, 1, 1, 1, 64, 0, 12, 0, 16, 1 << 31, 2.0, None, 0, 0, None)
    with pytest.raises(RuntimeError, match="outside the site"):
        _lib.call("b200unet_dropout_mul", 16, 64, 1, 1, 1, 64, 8, 64, 0, 16, 1 << 31, 2.0, None, 0, 0, None)
    with pytest.raises(RuntimeError, match="null"):
        _lib.call("b200unet_dropout_mul", 16, 64, 1, 1, 1, 64, 0, 64, 0, None, 1 << 31, 2.0, None, 0, 0, None)
    with pytest.raises(RuntimeError, match="sum range"):
        _lib.call("b200unet_dropout_mul", 16, 64, 1, 1, 1, 64, 0, 64, 0, 16, 1 << 31, 2.0, 16, 32, 64, None)


def test_dropout_network_engine_selection():
    """UNet(dropout=True) runs on the tensor-core engine at widths 64 and 128 (one nn.Dropout holder per site); width 8,
    check mode and UNet_attention with dropout stay on the generic fp32 engine; UNet_multitask builds no dropout layer."""
    import unet_torch_b200 as U
    from unet_torch_b200.generic import GenericEngine
    from unet_torch_b200.model import UNetEngine

    x = torch.zeros(1, 3, 32, 32)
    for width in (64, 128):
        net = U.UNet(3, 2, width, dropout=True, dropout_p=0.3)
        eng = net._engine_for(x)
        assert isinstance(eng, UNetEngine), width
        want = [net.down1.maxpool_conv[1], net.down2.maxpool_conv[1], net.down3.maxpool_conv[1], net.down4.maxpool_conv[1],
                net.up1.dropout, net.up2.dropout, net.up3.dropout, net.up4.dropout]
        assert all(a is b for a, b in zip(eng.drop, want)) and len(eng.drop) == 8
        assert eng._drop_ps(True) == (0.3,) * 8 and eng._drop_ps(False) == (0.0,) * 8
        net.up2.dropout.p = 0.7   # read from each holder at every forward
        assert eng._drop_ps(True)[5] == 0.7
        assert isinstance(net.set_check_mode(True)._engine_for(x), GenericEngine)
    assert isinstance(U.UNet(3, 2, 8, dropout=True)._engine_for(x), GenericEngine)
    assert isinstance(U.UNet_attention(3, 2, dropout=True)._engine_for(x), GenericEngine)
    assert U.UNet(3, 2)._get_engine().drop == [None] * 8
    assert U.UNet_multitask(3, 2, dropout=True)._get_engine().drop == [None] * 8
