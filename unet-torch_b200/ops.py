"""Tensor-level wrappers over the C ABI: each function takes torch CUDA tensors (device memory + stream plumbing
only) and launches the hand-written sm_100a kernels on the current stream. Activations are NHWC bf16 tensors of
shape [N, H, W, C]; a tensor may be a channel slice of a wider buffer (stride(2) = pixel pitch).
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

BF16 = torch.bfloat16


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _nhwc(t: torch.Tensor):
    """Validate an NHWC bf16 (possibly channel-sliced) tensor and return (ptr, pitch, N, H, W, C)."""
    if t.dtype != BF16 or t.dim() != 4 or not t.is_cuda:
        raise ValueError(f"expected a CUDA bf16 [N,H,W,C] tensor, got {t.dtype} {tuple(t.shape)} {t.device}")
    n, h, w, c = t.shape
    cs = t.stride(2)
    if t.stride(3) != 1 or t.stride(1) != w * cs or t.stride(0) != h * w * cs:
        raise ValueError(f"tensor is not NHWC with a uniform pixel pitch: shape {tuple(t.shape)} strides {t.stride()}")
    return t.data_ptr(), cs, n, h, w, c


def _f32(t: torch.Tensor):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
        raise ValueError(f"expected a contiguous CUDA fp32 tensor, got {t.dtype} {t.device} contiguous={t.is_contiguous()}")
    return t.data_ptr()


def _ptr(t):
    return None if t is None else t.data_ptr()


def tile_hw():
    return _lib.query("b200unet_tile_h"), _lib.query("b200unet_tile_w")


def num_pixel_tiles(n, h, w):
    th, tw = tile_hw()
    return n * ((h + th - 1) // th) * ((w + tw - 1) // tw)


def conv3x3_stat_rows(n, h, w, cin, cout):
    """Rows of the BatchNorm partial-statistics buffer conv3x3() fills for this shape."""
    return _lib.query("b200unet_conv3x3_stat_rows", n, h, w, cin, cout)


# --------------------------------------------------------------------------------------------- weights
def prep_conv3x3_weight(w: torch.Tensor, want_dgrad=True, out=(None, None)):
    """fp32 OIHW [K,C,3,3] -> (fprop operand [K,3,3,C] bf16, dgrad operand [C,3,3,K] bf16 with rotated taps).
    `out`: operand tensors of a previous call to refill in place."""
    k, c = w.shape[0], w.shape[1]
    wf, wd = out
    if wf is None or wf.device != w.device:
        wf = torch.empty((k, 3, 3, c), dtype=BF16, device=w.device)
        wd = torch.empty((c, 3, 3, k), dtype=BF16, device=w.device) if want_dgrad else None
    _lib.call("b200unet_prep_conv3x3_weight", _f32(w), wf.data_ptr(), _ptr(wd), k, c, _stream())
    return wf, wd


def prep_convt2x2_weight(w: torch.Tensor, out=(None, None)):
    """fp32 [Cin,Cup,2,2] -> (fprop operand [4*Cup, Cin] bf16, dgrad operand [Cin, 4*Cup] bf16)."""
    cin, cup = w.shape[0], w.shape[1]
    wf, wd = out
    if wf is None or wf.device != w.device:
        wf = torch.empty((4 * cup, cin), dtype=BF16, device=w.device)
        wd = torch.empty((cin, 4 * cup), dtype=BF16, device=w.device)
    _lib.call("b200unet_prep_convt2x2_weight", _f32(w), wf.data_ptr(), wd.data_ptr(), cin, cup, _stream())
    return wf, wd


# --------------------------------------------------------------------------------------------- tensor-core ops
def conv3x3(x: torch.Tensor, w_op: torch.Tensor, out: torch.Tensor, stats_partial: torch.Tensor | None = None):
    """out = conv3x3(x) with a prepared [Cout,3,3,Cin] bf16 operand (fprop or dgrad operand)."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w_op.shape) != (cout, 3, 3, cin) or w_op.dtype != BF16:
        raise ValueError(f"conv3x3: shape mismatch x{tuple(x.shape)} w{tuple(w_op.shape)} out{tuple(out.shape)}")
    if stats_partial is not None and stats_partial.numel() < conv3x3_stat_rows(n, h, w, cin, cout) * 2 * cout:
        raise ValueError("conv3x3: stats_partial too small")
    _lib.call("b200unet_conv3x3_igemm", xp, xcs, w_op.data_ptr(), op, ocs, _f32(stats_partial), n, h, w, cin, cout,
              _stream())
    return out


def conv3x3_dgrad_bnred(dy, w_dgrad, dx, bn_y, scale, shift, mean, rstd):
    """dx = conv3x3(dy, dgrad operand) with the first pass of the CONSUMER BatchNorm's backward fused into the epilogue
    (dx is the gradient at that BatchNorm+ReLU's output, bn_y its saved pre-BN tensor). Returns (partial, rows) for
    bn_relu_bwd(pre=...), or None when this shape has no fused form (the caller then runs the separate reduce pass)."""
    xp, xcs, n, h, w, cin = _nhwc(dy)
    op, ocs, n2, h2, w2, cout = _nhwc(dx)
    rows = _lib.query("b200unet_conv3x3_dgrad_bnred_rows", n, h, w, cin, cout)
    if rows <= 0 or mean is None or rstd is None:
        return None
    yp, ycs, n3, h3, w3, c3 = _nhwc(bn_y)
    if (n, h, w) != (n2, h2, w2) or (n3, h3, w3, c3) != (n, h, w, cout) or tuple(w_dgrad.shape) != (cout, 3, 3, cin):
        raise ValueError("conv3x3_dgrad_bnred: shape mismatch")
    partial = torch.empty(rows * 2 * cout, dtype=torch.float32, device=dy.device)
    _lib.call("b200unet_conv3x3_igemm_bnred", xp, xcs, w_dgrad.data_ptr(), op, ocs, yp, ycs, _f32(scale), _f32(shift), _f32(mean),
              _f32(rstd), partial.data_ptr(), n, h, w, cin, cout, _stream())
    return partial, rows


def conv3x3_bn_relu(x, w_op, scale, shift, out):
    """Eval mode: out = bf16(relu(scale * conv3x3(x) + shift)), BatchNorm (running statistics) and ReLU folded into the
    conv epilogue on the fp32 accumulators; `out` may be a channel slice of a concat buffer."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w_op.shape) != (cout, 3, 3, cin) or w_op.dtype != BF16:
        raise ValueError(f"conv3x3_bn_relu: shape mismatch x{tuple(x.shape)} w{tuple(w_op.shape)} out{tuple(out.shape)}")
    if scale.numel() != cout or shift.numel() != cout:
        raise ValueError("conv3x3_bn_relu: scale/shift must have Cout elements")
    _lib.call("b200unet_conv3x3_bn_relu_igemm", xp, xcs, w_op.data_ptr(), _f32(scale), _f32(shift), op, ocs, n, h, w, cin,
              cout, _stream())
    return out


def convt2x2(x, w_fprop, bias, out_canvas_slice, pad_top=0, pad_left=0):
    """ConvTranspose2d(k=2,s=2)+bias of x [N,H,W,Cin] written into out_canvas_slice [N,H2,W2,Cup] (a channel slice
    of the concat buffer) at offset (pad_top, pad_left)."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    op, ocs, n2, h2, w2, cup = _nhwc(out_canvas_slice)
    if tuple(w_fprop.shape) != (4 * cup, cin) or n != n2:
        raise ValueError("convt2x2: shape mismatch")
    _lib.call("b200unet_convt2x2_fprop", xp, xcs, w_fprop.data_ptr(), _f32(bias), op, ocs, n, h, w, cin, cup, h2, w2,
              pad_top, pad_left, _stream())


def convt2x2_dgrad(du_canvas_slice, w_dgrad, dx, pad_top=0, pad_left=0):
    up, ucs, n, h2, w2, cup = _nhwc(du_canvas_slice)
    xp, xcs, n2, h, w, cin = _nhwc(dx)
    if tuple(w_dgrad.shape) != (cin, 4 * cup) or n != n2:
        raise ValueError("convt2x2_dgrad: shape mismatch")
    _lib.call("b200unet_convt2x2_dgrad", up, ucs, w_dgrad.data_ptr(), xp, xcs, n, h, w, cin, cup, h2, w2, pad_top,
              pad_left, _stream())
    return dx


def _workspace(nfloats, device):
    return torch.empty((max(int(nfloats), 1),), dtype=torch.float32, device=device)


def conv3x3_wgrad(x, dy, dw_out: torch.Tensor):
    """dw_out (fp32 OIHW [Cout,Cin,3,3]) = weight gradient of conv3x3(x) given dy. Overwrites dw_out."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    yp, ycs, n2, h2, w2, cout = _nhwc(dy)
    if (n, h, w) != (n2, h2, w2) or tuple(dw_out.shape) != (cout, cin, 3, 3):
        raise ValueError("conv3x3_wgrad: shape mismatch")
    ws = _workspace(_lib.query("b200unet_conv3x3_wgrad_workspace_floats", n, h, w, cin, cout), x.device)
    _lib.call("b200unet_conv3x3_wgrad", xp, xcs, yp, ycs, ws.data_ptr(), _f32(dw_out), n, h, w, cin, cout, _stream())
    return dw_out


def convt2x2_wgrad(x, du_canvas_slice, dw_out, pad_top=0, pad_left=0):
    xp, xcs, n, h, w, cin = _nhwc(x)
    up, ucs, n2, h2, w2, cup = _nhwc(du_canvas_slice)
    if tuple(dw_out.shape) != (cin, cup, 2, 2) or n != n2:
        raise ValueError("convt2x2_wgrad: shape mismatch")
    ws = _workspace(_lib.query("b200unet_convt2x2_wgrad_workspace_floats", n, h, w, cin, cup), x.device)
    _lib.call("b200unet_convt2x2_wgrad", xp, xcs, up, ucs, ws.data_ptr(), _f32(dw_out), n, h, w, cin, cup, h2, w2,
              pad_top, pad_left, _stream())
    return dw_out


# --------------------------------------------------------------------------------------------- inc.conv1 (tensor cores)
def first_im2col(x_nchw: torch.Tensor, col: torch.Tensor):
    """fp32 NCHW network input -> 64-column bf16 im2col tensor [N,H,W,64] (column c*9+r*3+s, zero padded)."""
    if x_nchw.dtype != torch.float32 or not x_nchw.is_cuda or not x_nchw.is_contiguous() or x_nchw.dim() != 4:
        raise ValueError("first_im2col: expected a contiguous CUDA fp32 NCHW tensor")
    n, cin, h, w = x_nchw.shape
    cp, ccs, n2, h2, w2, c64 = _nhwc(col)
    if (n, h, w) != (n2, h2, w2) or c64 != 64:
        raise ValueError("first_im2col: shape mismatch")
    _lib.call("b200unet_first_im2col", x_nchw.data_ptr(), cp, ccs, n, h, w, cin, _stream())
    return col


def prep_first_weight(w: torch.Tensor, out=None):
    """fp32 OIHW [K,Cin,3,3] -> bf16 [K,64] operand matching first_im2col's columns."""
    k, cin = w.shape[0], w.shape[1]
    w1 = out if (out is not None and out.device == w.device) else torch.empty((k, 64), dtype=BF16, device=w.device)
    _lib.call("b200unet_prep_first_weight", _f32(w), w1.data_ptr(), k, cin, _stream())
    return w1


def conv3x3_first_tc(x_nchw: torch.Tensor, w1: torch.Tensor, out: torch.Tensor, stats_partial=None):
    """inc.conv1 fused: out = conv3x3(x) from the fp32 NCHW input with the im2col rows built in shared memory inside the
    tcgen05 kernel (no im2col tensor in HBM). w1 = prep_first_weight(w); statistics rows as conv1x1_c64()."""
    if x_nchw.dtype != torch.float32 or not x_nchw.is_cuda or not x_nchw.is_contiguous() or x_nchw.dim() != 4:
        raise ValueError("conv3x3_first_tc: expected a contiguous CUDA fp32 NCHW tensor")
    n, cin, h, w = x_nchw.shape
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w1.shape) != (cout, 64) or w1.dtype != BF16:
        raise ValueError("conv3x3_first_tc: shape mismatch")
    if stats_partial is not None and stats_partial.numel() < conv1x1_c64_stat_rows(n, h, w, cout) * 2 * cout:
        raise ValueError("conv3x3_first_tc: stats_partial too small")
    _lib.call("b200unet_conv3x3_first_igemm", x_nchw.data_ptr(), w1.data_ptr(), op, ocs, _f32(stats_partial), n, h, w, cin, cout,
              _stream())
    return out


def conv3x3_first_tc_bn_relu(x_nchw, w1, scale, shift, out):
    """Eval mode of conv3x3_first_tc: BatchNorm (running statistics) + ReLU folded into the epilogue."""
    n, cin, h, w = x_nchw.shape
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w1.shape) != (cout, 64) or w1.dtype != BF16 or x_nchw.dtype != torch.float32:
        raise ValueError("conv3x3_first_tc_bn_relu: shape mismatch")
    _lib.call("b200unet_conv3x3_first_bn_relu_igemm", x_nchw.contiguous().data_ptr(), w1.data_ptr(), _f32(scale), _f32(shift), op,
              ocs, n, h, w, cin, cout, _stream())
    return out


def conv3x3_first_tc_wgrad(x_nchw, dy, dw_out):
    """dw_out (fp32 OIHW [Cout,Cin,3,3]) = weight gradient of inc.conv1 from the fp32 NCHW input and dy (fused im2col)."""
    n, cin, h, w = x_nchw.shape
    yp, ycs, n2, h2, w2, cout = _nhwc(dy)
    if (n, h, w) != (n2, h2, w2) or tuple(dw_out.shape) != (cout, cin, 3, 3) or x_nchw.dtype != torch.float32:
        raise ValueError("conv3x3_first_tc_wgrad: shape mismatch")
    ws = _workspace(_lib.query("b200unet_conv3x3_first_tc_wgrad_workspace_floats", n, h, w, cout), dy.device)
    _lib.call("b200unet_conv3x3_first_tc_wgrad", x_nchw.data_ptr(), yp, ycs, ws.data_ptr(), _f32(dw_out), n, h, w, cin, cout,
              _stream())
    return dw_out


def conv1x1_c64_stat_rows(n, h, w, cout):
    return _lib.query("b200unet_conv1x1_c64_stat_rows", n, h, w, cout)


def conv1x1_c64(x, w1, out, stats_partial=None):
    """out[n,h,w,k] = sum_j x[n,h,w,j] w1[k,j] over a 64-channel input (+ BatchNorm partial statistics)."""
    xp, xcs, n, h, w, c = _nhwc(x)
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or c != 64 or tuple(w1.shape) != (cout, 64) or w1.dtype != BF16:
        raise ValueError("conv1x1_c64: shape mismatch")
    if stats_partial is not None and stats_partial.numel() < conv1x1_c64_stat_rows(n, h, w, cout) * 2 * cout:
        raise ValueError("conv1x1_c64: stats_partial too small")
    _lib.call("b200unet_conv1x1_c64_igemm", xp, xcs, w1.data_ptr(), op, ocs, _f32(stats_partial), n, h, w, cout, _stream())
    return out


def conv1x1_c64_bn_relu(x, w1, scale, shift, out):
    """Eval mode of conv1x1_c64: BatchNorm + ReLU folded into the epilogue."""
    xp, xcs, n, h, w, c = _nhwc(x)
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or c != 64 or tuple(w1.shape) != (cout, 64) or w1.dtype != BF16:
        raise ValueError("conv1x1_c64_bn_relu: shape mismatch")
    if scale.numel() != cout or shift.numel() != cout:
        raise ValueError("conv1x1_c64_bn_relu: scale/shift must have Cout elements")
    _lib.call("b200unet_conv1x1_c64_bn_relu_igemm", xp, xcs, w1.data_ptr(), _f32(scale), _f32(shift), op, ocs, n, h, w, cout,
              _stream())
    return out


def conv1x1_c64_wgrad(col, dy, dw_out):
    """dw_out (fp32 OIHW [Cout,Cin,3,3]) = weight gradient of inc.conv1 from its im2col'ed input and dy."""
    cp, ccs, n, h, w, c = _nhwc(col)
    yp, ycs, n2, h2, w2, cout = _nhwc(dy)
    if (n, h, w) != (n2, h2, w2) or c != 64 or dw_out.shape[0] != cout or dw_out[0].numel() > 64:
        raise ValueError("conv1x1_c64_wgrad: shape mismatch")
    ws = _workspace(_lib.query("b200unet_conv1x1_c64_wgrad_workspace_floats", n, h, w, cout), dy.device)
    _lib.call("b200unet_conv1x1_c64_wgrad", cp, ccs, yp, ycs, ws.data_ptr(), _f32(dw_out), n, h, w, dw_out[0].numel(),
              cout, _stream())
    return dw_out


# --------------------------------------------------------------------------------------------- first layer / head
def conv3x3_first(x_nchw: torch.Tensor, w_oihw: torch.Tensor, out, stats_partial=None):
    n, cin, h, w = x_nchw.shape
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w_oihw.shape) != (cout, cin, 3, 3):
        raise ValueError("conv3x3_first: shape mismatch")
    if stats_partial is not None and stats_partial.numel() < first_conv_stat_rows(n, h, w) * 2 * cout:
        raise ValueError("conv3x3_first: stats_partial too small")
    _lib.call("b200unet_conv3x3_first_fprop", _f32(x_nchw), _f32(w_oihw), op, ocs, _f32(stats_partial), n, h, w, cin,
              cout, _stream())
    return out


def first_conv_stat_rows(n, h, w):
    return (n * h * w + 127) // 128


def conv3x3_first_wgrad(x_nchw, dy, dw_out):
    n, cin, h, w = x_nchw.shape
    yp, ycs, n2, h2, w2, cout = _nhwc(dy)
    ws = _workspace(_lib.query("b200unet_conv3x3_first_wgrad_workspace_floats", n, h, w, cin, cout), dy.device)
    _lib.call("b200unet_conv3x3_first_wgrad", _f32(x_nchw), yp, ycs, ws.data_ptr(), _f32(dw_out), n, h, w, cin, cout,
              _stream())
    return dw_out


# The OutConv kernels compiled per class count cover up to HEAD_FIXED_CLASSES classes; the head_many family takes
# 1..HEAD_MAX_CLASSES (uint8 class masks) with the class count at run time.
HEAD_FIXED_CLASSES, HEAD_MAX_CLASSES = 8, 256


def _head(name, ncls):
    return name.replace("head_", "head_many_", 1) if ncls > HEAD_FIXED_CLASSES else name


def head_fprop(a, w, bias, logits_nchw):
    ap, acs, n, h, wd, cin = _nhwc(a)
    ncls = w.shape[0]
    _lib.call(_head("b200unet_head_fprop", ncls), ap, acs, _f32(w.view(ncls, cin)), _f32(bias), _f32(logits_nchw), n, h,
              wd, cin, ncls, _stream())
    return logits_nchw


def head_bwd(dz_nchw, a, w, da, dw, db):
    ap, acs, n, h, wd, cin = _nhwc(a)
    dp, dcs, *_ = _nhwc(da)
    ncls = w.shape[0]
    ws = _workspace(_lib.query(_head("b200unet_head_bwd_workspace_floats", ncls), n, h, wd, cin, ncls), a.device)
    _lib.call(_head("b200unet_head_bwd", ncls), _f32(dz_nchw), ap, acs, _f32(w.view(ncls, cin)), dp, dcs, ws.data_ptr(),
              _f32(dw), _f32(db), n, h, wd, cin, ncls, _stream())


# --------------------------------------------------------------------------------------------- BN / ReLU / pool
def bn_reduce_partials(stats_partial, rows, c, sums_f64):
    _lib.call("b200unet_bn_reduce_partials", _f32(stats_partial), rows, c, sums_f64.data_ptr(), _stream())


def bn_finalize(sums_f64, count, gamma, beta, eps, momentum, running_mean, running_var, mean, rstd, scale, shift):
    c = gamma.numel()
    _lib.call("b200unet_bn_finalize", sums_f64.data_ptr(), float(count), _f32(gamma), _f32(beta), eps, momentum,
              _ptr(running_mean), _ptr(running_var), _f32(mean), _f32(rstd), _f32(scale), _f32(shift), c, _stream())


def bn_reduce_finalize(stats_partial, rows, count, gamma, beta, eps, momentum, running_mean, running_var, num_batches_tracked,
                       mean, rstd, scale, shift):
    """bn_reduce_partials + bn_finalize + `num_batches_tracked += 1` in one launch (single-GPU forward)."""
    _lib.call("b200unet_bn_reduce_finalize", _f32(stats_partial), rows, gamma.numel(), float(count), _f32(gamma), _f32(beta),
              eps, momentum, _ptr(running_mean), _ptr(running_var), _ptr(num_batches_tracked), _f32(mean), _f32(rstd),
              _f32(scale), _f32(shift), _stream())


FOLD_ROWS_ABOVE, FOLD_ROWS_TO = 4096, 296


def fold_rows(stats_partial, rows, ncols):
    """Statistics rows [rows][ncols] -> ([FOLD_ROWS_TO][ncols], FOLD_ROWS_TO) when there are more than FOLD_ROWS_ABOVE of them
    (one per pixel tile from the attention gates' GEMM epilogues), else unchanged."""
    if stats_partial is None or rows <= FOLD_ROWS_ABOVE:
        return stats_partial, rows
    out = torch.empty(FOLD_ROWS_TO * ncols, dtype=torch.float32, device=stats_partial.device)
    _lib.call("b200unet_fold_rows", _f32(stats_partial), rows, ncols, out.data_ptr(), FOLD_ROWS_TO, _stream())
    return out, FOLD_ROWS_TO


def bn_eval_affine(gamma, beta, running_mean, running_var, eps, scale, shift):
    _lib.call("b200unet_bn_eval_affine", _f32(gamma), _f32(beta), _f32(running_mean), _f32(running_var), eps,
              _f32(scale), _f32(shift), gamma.numel(), _stream())


def bn_eval_stats(running_mean, running_var, eps, mean, rstd):
    """mean = running_mean, rstd = rsqrt(running_var + eps): what the backward kernels need after an eval-mode forward."""
    _lib.call("b200unet_bn_eval_stats", _f32(running_mean), _f32(running_var), eps, _f32(mean), _f32(rstd), mean.numel(),
              _stream())


def bn_relu_fwd(y, scale, shift, a, pooled=None, pool_idx=None):
    yp, ycs, n, h, w, c = _nhwc(y)
    ap, acs, *_ = _nhwc(a)
    _lib.call("b200unet_bn_relu_fwd", yp, ycs, _f32(scale), _f32(shift), ap, acs, _ptr(pooled), _ptr(pool_idx), n, h, w,
              c, _stream())


def bn_relu_bwd(g1, g_pool, pool_idx, y, gamma, scale, shift, mean, rstd, dy, dgamma, dbeta, count=None,
                allreduce=None, frozen=False, pre=None):
    """Backward of BN->ReLU(->skip+pool). g1: gradient w.r.t. the activation (may be a channel slice, or None);
    g_pool/pool_idx: gradient through the 2x2 max pool (or None). Writes dy (may alias y), dgamma, dbeta.
    allreduce: optional DataParallelContext (SyncBN): the sums are exchanged between the two passes - one fused NVLink kernel
    on the unreduced block partials when available, otherwise reduce_partials + all_reduce_sum.
    pre: (partial, rows) already produced by the epilogue of the kernel that computed g1 (conv3x3_dgrad_bnred): the reduce
    pass over g1 and y is skipped.
    frozen: the forward normalised with RUNNING statistics (module.eval() under autograd): mean/rstd are the running ones,
    statistics do not depend on y, so dy = gamma * rstd * da (the batch-statistics correction terms vanish: the apply pass
    gets an all-zero sums vector) while dgamma / dbeta keep the reduced sums."""
    if mean is None or rstd is None:
        raise RuntimeError("bn_relu_bwd: this forward did not save BatchNorm statistics (mean/rstd)")
    yp, ycs, n, h, w, c = _nhwc(y)
    g1p, g1cs = (None, 0)
    if g1 is not None:
        g1p, g1cs, *_ = _nhwc(g1)
    dp, dcs, *_ = _nhwc(dy)
    ws = _workspace(_lib.query("b200unet_bn_bwd_workspace_floats", n, h, w, c), y.device)
    sums = torch.empty((2 * c,), dtype=torch.float64, device=y.device)
    sums_local = None
    if count is None:
        count = n * h * w
    use_rows = allreduce is not None and not frozen and allreduce.supports_rows(c)
    if pre is not None or use_rows:
        if pre is not None:
            if g_pool is not None:
                raise ValueError("bn_relu_bwd: a fused reduction cannot include a pooled gradient")
            ws, nrows = pre
        else:
            rows = ctypes.c_int(0)
            _lib.call("b200unet_bn_relu_bwd_reduce_rows", g1p, g1cs, _ptr(g_pool), _ptr(pool_idx), yp, ycs, _f32(scale),
                      _f32(shift), _f32(mean), _f32(rstd), ws.data_ptr(), ctypes.byref(rows), n, h, w, c, _stream())
            nrows = rows.value
        if use_rows:
            sums_local = torch.empty_like(sums)
            allreduce.rows_allreduce(ws, nrows, c, sums_local, sums)
        else:
            bn_reduce_partials(ws, nrows, c, sums)
            if frozen:
                sums_local = sums
                sums = torch.zeros_like(sums)
            elif allreduce is not None:
                sums_local = sums.clone()
                allreduce.all_reduce_sum(sums)
    else:
        _lib.call("b200unet_bn_relu_bwd_reduce", g1p, g1cs, _ptr(g_pool), _ptr(pool_idx), yp, ycs, _f32(scale), _f32(shift),
                  _f32(mean), _f32(rstd), ws.data_ptr(), sums.data_ptr(), n, h, w, c, _stream())
        if frozen:
            sums_local = sums
            sums = torch.zeros_like(sums)
        elif allreduce is not None:
            sums_local = sums.clone()
            allreduce.all_reduce_sum(sums)
    _lib.call("b200unet_bn_relu_bwd_apply", g1p, g1cs, _ptr(g_pool), _ptr(pool_idx), yp, ycs, _f32(gamma), _f32(scale),
              _f32(shift), _f32(mean), _f32(rstd), sums.data_ptr(), float(count), _ptr(sums_local), dp, dcs,
              _f32(dgamma), _f32(dbeta), n, h, w, c, _stream())


def partial_colsum(stats_partial, rows, row_pitch, col_lo, n, out):
    """out[c] = sum over the statistics rows of column col_lo + c (see conv3x3(stats_partial=...))."""
    _lib.call("b200unet_partial_colsum", _f32(stats_partial), rows, row_pitch, col_lo, n, _f32(out), _stream())
    return out


def maxpool2x2(a, pooled, pool_idx=None):
    """pooled = MaxPool2d(2)(a) over NHWC bf16 (a may be a channel slice); optional 1-byte window positions."""
    ap, acs, n, h, w, c = _nhwc(a)
    pp, pcs, n2, h2, w2, c2 = _nhwc(pooled)
    if (n2, h2, w2, c2) != (n, h // 2, w // 2, c):
        raise ValueError(f"maxpool2x2: shapes {tuple(a.shape)} -> {tuple(pooled.shape)}")
    _lib.call("b200unet_maxpool2x2_fwd", ap, acs, pp, pcs, _ptr(pool_idx), n, h, w, c, _stream())
    return pooled


def nhwc_copy(src, dst):
    """dst[..., :] = src over NHWC bf16 channel slices (skip half of a second decoder's concat buffer)."""
    sp, scs, n, h, w, c = _nhwc(src)
    dp, dcs, n2, h2, w2, c2 = _nhwc(dst)
    if (n, h, w, c) != (n2, h2, w2, c2):
        raise ValueError(f"nhwc_copy: shapes differ {tuple(src.shape)} vs {tuple(dst.shape)}")
    _lib.call("b200unet_nhwc_copy", sp, scs, dp, dcs, n * h * w, c, _stream())
    return dst


def nhwc_add(a, b, out=None):
    """out = a + b over NHWC bf16 channel slices (out defaults to a: in-place accumulation)."""
    out = a if out is None else out
    ap, acs, n, h, w, c = _nhwc(a)
    bp, bcs, *sb = _nhwc(b)
    op, ocs, *so = _nhwc(out)
    if sb != [n, h, w, c] or so != [n, h, w, c]:
        raise ValueError(f"nhwc_add: shapes differ {tuple(a.shape)} {tuple(b.shape)} {tuple(out.shape)}")
    _lib.call("b200unet_nhwc_add", ap, acs, bp, bcs, op, ocs, n * h * w, c, _stream())
    return out


def dropout_threshold_scale(p):
    """(threshold, scale) of the dropout mask for drop probability p, in double as DESIGN.md §4 fixes them: an element is kept
    when its 32-bit Philox word is below threshold = min(2^32 - 1, floor((1 - p) 2^32)); kept elements are multiplied by
    float(1 / (1 - p)). p = 1 keeps nothing and scales by 0 (no inf * 0)."""
    p = float(p)
    if not 0.0 <= p <= 1.0:
        raise ValueError(f"dropout probability has to be between 0 and 1, but got {p}")
    if p == 1.0:
        return 0, 0.0
    return min(2 ** 32 - 1, int((1.0 - p) * 2.0 ** 32)), float(torch.tensor(1.0 / (1.0 - p), dtype=torch.float32))


def dropout_mul(x, site, seed, p, c_site=None, c_lo=0, sums=None):
    """nn.Dropout(p) in place on x (NHWC bf16, possibly a channel slice), mask of `site` (0..3 = down1..4, 4..7 = up1..4)
    drawn from the int64 device tensor `seed`. x holds channels [c_lo, c_lo + C) of a site tensor with c_site channels
    (default: x is the whole site tensor). sums = (lo, out): out[c] = sum over pixels of the dropped x[..., lo + c], for the
    channels lo.. of x (fp32 [C - lo], fixed-order reduction)."""
    xp, xcs, n, h, w, c = _nhwc(x)
    if seed.dtype != torch.int64 or not seed.is_cuda or seed.numel() != 1:
        raise ValueError("dropout_mul: seed must be one int64 on the device")
    threshold, scale = dropout_threshold_scale(p)
    part, lo, cnt, rows = None, 0, 0, 0
    if sums is not None:
        lo, out = sums
        cnt = c - lo
        rows = _lib.query("b200unet_dropout_partial_rows", n, h, w, c)
        part = torch.empty(rows * cnt, dtype=torch.float32, device=x.device)
    _lib.call("b200unet_dropout_mul", xp, xcs, n, h, w, c if c_site is None else c_site, c_lo, c, site, seed.data_ptr(),
              threshold, scale, _ptr(part), lo, cnt, _stream())
    if sums is not None:
        partial_colsum(part, rows, cnt, 0, cnt, out)
    return x


def channel_sum(x, out):
    xp, xcs, n, h, w, c = _nhwc(x)
    ws = _workspace(_lib.query("b200unet_channel_sum_workspace_floats", c), x.device)
    _lib.call("b200unet_channel_sum", xp, xcs, ws.data_ptr(), _f32(out), n * h * w, c, _stream())
    return out


# --------------------------------------------------------------------------------------------- attention gates
def convt2x2_stats(x, w_fprop, bias, out, stats_partial, stat_channels):
    """convt2x2() into a plain [N,2H,2W,Cup] tensor, also filling the BatchNorm partial-statistics rows of the first
    stat_channels channels of its output ([convt2x2_stat_rows][2][stat_channels] fp32)."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    op, ocs, n2, h2, w2, cup = _nhwc(out)
    if tuple(w_fprop.shape) != (4 * cup, cin) or (n2, h2, w2) != (n, 2 * h, 2 * w):
        raise ValueError("convt2x2_stats: shape mismatch")
    _lib.call("b200unet_convt2x2_fprop_stats", xp, xcs, w_fprop.data_ptr(), _f32(bias), op, ocs, _f32(stats_partial), stat_channels,
              n, h, w, cin, cup, h2, w2, 0, 0, _stream())
    return out


def convt2x2_stat_rows(n, h, w):
    return _lib.query("b200unet_convt2x2_stat_rows", n, h, w)


def conv1x1_stat_rows(n, h, w):
    return _lib.query("b200unet_conv1x1_stat_rows", n, h, w)


def conv1x1(x, w_op, bias, out, stats_partial=None, stat_channels=None):
    """out = 1x1 convolution of x with a bf16 [Cout, Cin] operand (+ fp32 bias [Cout] or None); optional BatchNorm
    partial-statistics rows [conv1x1_stat_rows][2][stat_channels] (default Cout). With the transposed operand it is the
    backward-data."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    op, ocs, n2, h2, w2, cout = _nhwc(out)
    if (n, h, w) != (n2, h2, w2) or tuple(w_op.shape) != (cout, cin) or w_op.dtype != BF16 or not w_op.is_contiguous():
        raise ValueError(f"conv1x1: shape mismatch x{tuple(x.shape)} w{tuple(w_op.shape)} out{tuple(out.shape)}")
    _lib.call("b200unet_conv1x1_fprop", xp, xcs, w_op.data_ptr(), _f32(bias), op, ocs, _f32(stats_partial),
              cout if stat_channels is None else stat_channels, n, h, w, cin, cout, _stream())
    return out


def conv1x1_wgrad(x, dy, dw_out):
    """dw_out fp32 [Cout_real, Cin(,1,1)] = sum over pixels of dy[.., k] * x[.., c]; dy may carry zero-padded channels beyond
    Cout_real."""
    xp, xcs, n, h, w, cin = _nhwc(x)
    yp, ycs, n2, h2, w2, cout = _nhwc(dy)
    creal = dw_out.shape[0]
    if (n, h, w) != (n2, h2, w2) or dw_out.numel() != creal * cin or creal > cout:
        raise ValueError("conv1x1_wgrad: shape mismatch")
    ws = _workspace(_lib.query("b200unet_conv1x1_wgrad_workspace_floats", n, h, w, cin, cout), x.device)
    _lib.call("b200unet_conv1x1_wgrad", xp, xcs, yp, ycs, ws.data_ptr(), _f32(dw_out), n, h, w, cin, cout, creal, _stream())
    return dw_out


def sgemm_strided(a, b, c, m, n, k, a_strides, b_strides, c_strides, bias_m=None, batch=1, batch_strides=(0, 0, 0),
                  accumulate=False, offsets=(0, 0, 0)):
    """c[z][i][j] (+)= sum_l a[z][i][l] * b[z][l][j] (+ bias_m[i]) over fp32 tensors addressed by ELEMENT strides
    (a_strides = (row, k), b_strides = (k, col), c_strides = (row, col)); offsets are element offsets into a, b, c."""
    for t in (a, b, c):
        if t.dtype != torch.float32 or not t.is_cuda:
            raise ValueError("sgemm_strided: fp32 CUDA tensors expected")
    _lib.call("b200unet_sgemm_strided", a.data_ptr() + 4 * offsets[0], b.data_ptr() + 4 * offsets[1], c.data_ptr() + 4 * offsets[2],
              _ptr(bias_m), m, n, k, a_strides[0], a_strides[1], b_strides[0], b_strides[1], c_strides[0], c_strides[1], batch,
              batch_strides[0], batch_strides[1], batch_strides[2], 1 if accumulate else 0, _stream())
    return c


def sum_batches(part, out):
    """out = part.sum(0) for a contiguous fp32 [batches, ...] tensor (fixed summation order)."""
    _lib.call("b200unet_sum_batches", _f32(part), _f32(out), out.numel(), part.shape[0], _stream())
    return out


def gate_stat_rows(pixels, c):
    return _lib.query("b200unet_gate_stat_rows", pixels, c)


def gate_psi_fwd(q1, x1, scale_q, shift_q, scale_x, shift_x, w_psi, b_psi, s, stats_partial=None):
    """s[n,h,w] = b_psi + sum_c w_psi[c] * relu(scale_q*q1 + shift_q + scale_x*x1 + shift_x)[c] over the C real channels of
    the two pre-BatchNorm maps (channel slices of possibly wider tensors)."""
    qp, qcs, n, h, w, c = _nhwc(q1)
    xp, xcs, *sx = _nhwc(x1)
    if sx != [n, h, w, c] or s.numel() != n * h * w:
        raise ValueError("gate_psi_fwd: shape mismatch")
    _lib.call("b200unet_gate_psi_fwd", qp, qcs, xp, xcs, _f32(scale_q), _f32(shift_q), _f32(scale_x), _f32(shift_x), _f32(w_psi),
              _f32(b_psi), _f32(s), _f32(stats_partial), n * h * w, c, _stream())
    return s


def gate_apply_fwd(x, s, scale_p, shift_p, out):
    xp, xcs, n, h, w, c = _nhwc(x)
    op, ocs, *so = _nhwc(out)
    if so != [n, h, w, c] or s.numel() != n * h * w:
        raise ValueError("gate_apply_fwd: shape mismatch")
    _lib.call("b200unet_gate_apply_fwd", xp, xcs, _f32(s), _f32(scale_p), _f32(shift_p), op, ocs, n * h * w, c, _stream())
    return out


def gate_apply_bwd(g, x, s, scale_p, shift_p, mean_p, rstd_p, dx, dz, sums2):
    """dz, sums2 (and dx = g * A unless dx is None: the engine adds that term with gate_dx afterwards)."""
    gp, gcs, n, h, w, c = _nhwc(g)
    xp, xcs, *sx = _nhwc(x)
    dp, dcs, sd = None, 0, [n, h, w, c]
    if dx is not None:
        dp, dcs, *sd = _nhwc(dx)
    if sx != [n, h, w, c] or sd != [n, h, w, c] or s.numel() != n * h * w or dz.numel() != n * h * w:
        raise ValueError("gate_apply_bwd: shape mismatch")
    ws = _workspace(_lib.query("b200unet_gate_workspace_floats", 32), g.device)
    _lib.call("b200unet_gate_apply_bwd", gp, gcs, xp, xcs, _f32(s), _f32(scale_p), _f32(shift_p), _f32(mean_p), _f32(rstd_p), dp, dcs,
              _f32(dz), ws.data_ptr(), sums2.data_ptr(), n * h * w, c, _stream())


def gate_dx(g, s, scale_p, shift_p, dx):
    """dx <- g * sigmoid(scale_p * s + shift_p) + dx, in place."""
    gp, gcs, n, h, w, c = _nhwc(g)
    dp, dcs, *sd = _nhwc(dx)
    if sd != [n, h, w, c] or s.numel() != n * h * w:
        raise ValueError("gate_dx: shape mismatch")
    _lib.call("b200unet_gate_dx", gp, gcs, _f32(s), _f32(scale_p), _f32(shift_p), dp, dcs, n * h * w, c, _stream())
    return dx


def gate_bwd_reduce(q1, x1, aff_q, aff_x, w_psi, s, dz, gamma_p, mean_p, rstd_p, sums2, count, ds, sums):
    """aff_q / aff_x = (scale, shift, mean, rstd) of the two BatchNorms. Fills ds and sums (fp64 [4C + 8])."""
    qp, qcs, n, h, w, c = _nhwc(q1)
    xp, xcs, *_ = _nhwc(x1)
    ws = _workspace(_lib.query("b200unet_gate_workspace_floats", c), q1.device)
    _lib.call("b200unet_gate_bwd_reduce", qp, qcs, xp, xcs, _f32(aff_q[0]), _f32(aff_q[1]), _f32(aff_x[0]), _f32(aff_x[1]),
              _f32(aff_q[2]), _f32(aff_q[3]), _f32(aff_x[2]), _f32(aff_x[3]), _f32(w_psi), _f32(s), _f32(dz), _f32(gamma_p),
              _f32(mean_p), _f32(rstd_p), sums2.data_ptr(), float(count), _f32(ds), ws.data_ptr(), sums.data_ptr(), n * h * w, c,
              _stream())


def gate_bwd_apply(q1, x1, aff_q, aff_x, gamma_q, gamma_x, w_psi, ds, sums, sums_local, sums2_local, count, grads, dbias):
    """Overwrites q1 / x1 with the gradients at the two pre-BatchNorm maps. grads = (dgamma_q, dbeta_q, dgamma_x, dbeta_x,
    dw_psi, db_psi, dgamma_p, dbeta_p) fp32 outputs; dbias fp32 [2C] = channel sums of the two stored gradients."""
    qp, qcs, n, h, w, c = _nhwc(q1)
    xp, xcs, *_ = _nhwc(x1)
    ws = _workspace(_lib.query("b200unet_gate_workspace_floats", c), q1.device)
    _lib.call("b200unet_gate_bwd_apply", qp, qcs, xp, xcs, _f32(aff_q[0]), _f32(aff_q[1]), _f32(aff_x[0]), _f32(aff_x[1]),
              _f32(gamma_q), _f32(aff_q[2]), _f32(aff_q[3]), _f32(gamma_x), _f32(aff_x[2]), _f32(aff_x[3]), _f32(w_psi), _f32(ds),
              sums.data_ptr(), _ptr(sums_local), sums2_local.data_ptr(), float(count), *[g.data_ptr() for g in grads],
              ws.data_ptr(), _f32(dbias), n * h * w, c, _stream())


# --------------------------------------------------------------------------------------------- losses / inference
def loss_ce_dice_fwd(logits, target, mode):
    n, ncls, h, w = logits.shape
    sums = torch.empty((_lib.query("b200unet_loss_sums_doubles_n", ncls),), dtype=torch.float64, device=logits.device)
    out = torch.empty((3,), dtype=torch.float32, device=logits.device)
    err = torch.empty((1,), dtype=torch.int32, device=logits.device)
    _lib.call("b200unet_loss_ce_dice_fwd", _f32(logits), _f32(target), sums.data_ptr(), out.data_ptr(), err.data_ptr(),
              n, ncls, h * w, mode, _stream())
    keep = _lib.query("b200unet_loss_sums_saved_doubles_n", ncls)
    if keep < sums.numel():  # past 8 classes the rest is forward-only scratch: do not keep it alive until the backward
        sums = sums[:keep].clone()
    return out, sums, err


def loss_ce_dice_bwd(logits, target, sums, grad_out, mode):
    n, ncls, h, w = logits.shape
    dz = torch.empty_like(logits)
    _lib.call("b200unet_loss_ce_dice_bwd", _f32(logits), _f32(target), sums.data_ptr(), _f32(grad_out), dz.data_ptr(),
              n, ncls, h * w, mode, _stream())
    return dz


def mse_fwd(pred, target, relu_input=False):
    s = torch.empty((1,), dtype=torch.float64, device=pred.device)
    out = torch.empty((1,), dtype=torch.float32, device=pred.device)
    _lib.call("b200unet_mse_fwd", _f32(pred), _f32(target), s.data_ptr(), out.data_ptr(), pred.numel(),
              int(relu_input), _stream())
    return out


def mse_bwd(pred, target, grad_out, relu_input=False):
    d = torch.empty_like(pred)
    _lib.call("b200unet_mse_bwd", _f32(pred), _f32(target), _f32(grad_out), d.data_ptr(), pred.numel(),
              int(relu_input), _stream())
    return d


def softmax_argmax(logits):
    n, ncls, h, w = logits.shape
    mask = torch.empty((n, h, w), dtype=torch.int64, device=logits.device)
    _lib.call("b200unet_softmax_argmax", _f32(logits), mask.data_ptr(), n, ncls, h * w, _stream())
    return mask


# --------------------------------------------------------------------------------------------- edges of the path
def znorm_to_chw(img_u8: torch.Tensor, reverse_channels: bool = True) -> torch.Tensor:
    """uint8 [N,H,W,C] (or [H,W,C] / [H,W]) -> z-normalised fp32 [N,C,H,W] (DataLoader.py:661-671)."""
    if img_u8.dtype != torch.uint8 or not img_u8.is_cuda:
        raise TypeError("znorm_to_chw expects a CUDA uint8 tensor (no CPU fallback)")
    if img_u8.dim() == 2:
        img_u8 = img_u8[None, :, :, None]
    elif img_u8.dim() == 3:
        img_u8 = img_u8[None]
    img_u8 = img_u8.contiguous()
    n, h, w, c = img_u8.shape
    out = torch.empty((n, c, h, w), dtype=torch.float32, device=img_u8.device)
    ws = torch.empty(_lib.query("b200unet_znorm_workspace_bytes", n, c), dtype=torch.uint8, device=img_u8.device)
    _lib.call("b200unet_znorm_to_chw", img_u8.data_ptr(), ws.data_ptr(), _f32(out), n, h, w, c,
              int(bool(reverse_channels) and c > 1), _stream())
    return out


def head_mask(a, w, bias):
    """OutConv + softmax + argmax + uint8 in one pass (test_mc3serousv5.py:879-887); a: NHWC bf16."""
    ap, acs, n, h, wd, cin = _nhwc(a)
    ncls = w.shape[0]
    mask = torch.empty((n, h, wd), dtype=torch.uint8, device=a.device)
    _lib.call(_head("b200unet_head_mask", ncls), ap, acs, _f32(w.view(ncls, cin)), _f32(bias), mask.data_ptr(), n, h, wd,
              cin, ncls, _stream())
    return mask


def head_sigmoid_mask(a, w, bias, threshold=0.5):
    """OutConv channel 0 + sigmoid + `>= threshold` -> {0,1} uint8 [N,H,W] (test.py:393-399); a: NHWC bf16."""
    ap, acs, n, h, wd, cin = _nhwc(a)
    if w.shape[0] > HEAD_FIXED_CLASSES:  # only channel 0 is thresholded: its row and bias make a 1-class head
        w, bias = w[:1], bias[:1]
    ncls = w.shape[0]
    mask = torch.empty((n, h, wd), dtype=torch.uint8, device=a.device)
    _lib.call("b200unet_head_sigmoid_mask", ap, acs, _f32(w.view(ncls, cin)), _f32(bias), mask.data_ptr(), n, h, wd, cin,
              ncls, float(threshold), _stream())
    return mask


def head_density(a, w, bias, divisor=200.0, with_counts=True):
    """OutConv + F.relu + /divisor -> fp32 NCHW maps (+ fp64 [N,ncls] sums) (test_mc3serousv5.py:961-974)."""
    ap, acs, n, h, wd, cin = _nhwc(a)
    ncls = w.shape[0]
    out = torch.empty((n, ncls, h, wd), dtype=torch.float32, device=a.device)
    counts = torch.empty((n, ncls), dtype=torch.float64, device=a.device) if with_counts else None
    _lib.call(_head("b200unet_head_density", ncls), ap, acs, _f32(w.view(ncls, cin)), _f32(bias), _f32(out),
              counts.data_ptr() if counts is not None else None, n, h, wd, cin, ncls, float(divisor), _stream())
    return out, counts
