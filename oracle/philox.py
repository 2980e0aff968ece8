"""The dropout masks of the tensor-core engine (DESIGN.md §4) restated in numpy: the checker for csrc/dropout.cu.

For the element with NHWC linear index e = ((n*H + h)*W + w)*C + c of dropout site s (0..3 = down1..4 after the pooling,
4..7 = up1..4 after the concat, skip channels first):
    (r0, r1, r2, r3) = Philox4x32-10(counter = (lo32(e/4), hi32(e/4), s, 0), key = (lo32(seed), hi32(seed)))
    keep = r[e % 4] < T,   T = min(2^32 - 1, floor((1 - p) 2^32)),   kept elements are scaled by float32(1 / (1 - p)).
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(counter, key):
    """Random123's Philox4x32-10. counter: four uint32 values or arrays (broadcast together), key: two uint32 values.
    Returns the four output words as uint32 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) for c in counter))
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def threshold_scale(p):
    """(T, scale) for drop probability p, in double; p = 1 -> (0, 0.0)."""
    p = float(p)
    if p == 1.0:
        return 0, 0.0
    return min(2 ** 32 - 1, int(np.floor((1.0 - p) * 2.0 ** 32))), float(np.float32(1.0 / (1.0 - p)))


def keep_mask(seed, site, shape, p, c_lo=0, nc=None):
    """Boolean keep mask [N, H, W, nc] for channels [c_lo, c_lo + nc) of the site tensor of NHWC `shape` = (N, H, W, C)."""
    n, h, w, c = shape
    nc = c - c_lo if nc is None else nc
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    t, _ = threshold_scale(p)
    pix = np.arange(n * h * w, dtype=np.uint64)[:, None]
    e = pix * np.uint64(c) + np.uint64(c_lo) + np.arange(nc, dtype=np.uint64)[None, :]
    q = e >> np.uint64(2)
    words = philox4x32_10((q & _LO, q >> _32, site, 0), (seed & 0xFFFFFFFF, seed >> 32))
    r = np.choose((e & np.uint64(3)).astype(np.intp), words)
    return (r < np.uint32(t)).reshape(n, h, w, nc)


def site_shapes(n, h, w, width):
    """NHWC shape of each of the 8 site tensors: the pooled tensors of down1..4, then the concat tensors of up1..4."""
    out = [(n, h >> (s + 1), w >> (s + 1), width << s) for s in range(4)]
    out += [(n, h >> (7 - s), w >> (7 - s), 2 * (width << (7 - s))) for s in range(4, 8)]
    return out


def oracle_masks(seed, n, h, w, width, ps):
    """{"down1".."down4", "up1".."up4": NCHW float64 multipliers (keep * scale)} for unet_oracle.unet_forward(dropout_masks=),
    ps = drop probability per site (0 = ones)."""
    import torch

    names = [f"down{i}" for i in range(1, 5)] + [f"up{i}" for i in range(1, 5)]
    out = {}
    for s, (name, shape) in enumerate(zip(names, site_shapes(n, h, w, width))):
        if ps[s] > 0:
            _, scale = threshold_scale(ps[s])
            m = torch.from_numpy(keep_mask(seed, s, shape, ps[s])).double() * scale
        else:
            m = torch.ones(shape, dtype=torch.float64)
        out[name] = m.permute(0, 3, 1, 2).contiguous()
    return out
