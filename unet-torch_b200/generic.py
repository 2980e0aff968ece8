"""Generic fp32 engine of the B200 UNet: the same network (reference Model.py:95-153) executed by the plain CUDA-core
kernels of csrc/generic_f32.cu on NCHW fp32 tensors.

Two uses:
  * CHECK MODE (`net.set_check_mode(True)` or B200UNET_CHECK_FP32=1): the reference's own precision, so logits and
    loss agree with the reference to ~1e-6 (north_star asks 1e-4) - separates "is the algorithm right" from bf16 noise.
  * the documented slow-but-correct route for inputs the tensor-core engine does not take: H or W not divisible by
    16 (floor-mode pooling + the F.pad branch, Model.py:69-73), `initial_feature_map` not a multiple of 64, and the
    dropout variants (Model.py:34-39, 81-82). Still CUDA, still this library's kernels: there is no PyTorch fallback.
Dropout masks are drawn with torch's generator (`F.dropout` on a ones tensor of the reference's shape, in the
reference's order), applied and back-propagated by the library's kernel.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import _lib, ops
from .dist import DataParallelContext


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _v(t: torch.Tensor):
    """(pointer, batch stride) of an NCHW fp32 view whose (C,H,W) block is dense."""
    if t.dtype != torch.float32 or not t.is_cuda or t.dim() != 4:
        raise ValueError(f"expected a CUDA fp32 NCHW tensor, got {t.dtype} {tuple(t.shape)}")
    n, c, h, w = t.shape
    if t.stride(3) != 1 or t.stride(2) != w or t.stride(1) != h * w:
        raise ValueError(f"NCHW view is not channel-dense: shape {tuple(t.shape)} strides {t.stride()}")
    return t.data_ptr(), t.stride(0)


def _dc(mod):
    return mod.double_conv


class GenericEngine:
    def __init__(self, net):
        self.net = net
        downs = [net.down1, net.down2, net.down3, net.down4]
        ups = [net.up1, net.up2, net.up3, net.up4]
        enc_dc = [_dc(net.inc)] + [_dc(d.maxpool_conv[-1]) for d in downs]
        self.enc = [((s[0], s[1]), (s[3], s[4])) for s in enc_dc]
        self.ups = [u.up for u in ups]
        self.dec = [((_dc(u.conv)[0], _dc(u.conv)[1]), (_dc(u.conv)[3], _dc(u.conv)[4])) for u in ups]
        self.head = net.outc.conv
        # UNet_attention (Model.py:299-375): one Attention_block per Up, gating the skip connection (None for UNet)
        gates = getattr(net, "_attention_gates", None)
        self.gates = gates() if gates is not None else None

    def params_in_backward_order(self):
        out = [self.head.weight, self.head.bias]
        for j in (3, 2, 1, 0):
            (c1, b1), (c2, b2) = self.dec[j]
            out += [b2.weight, b2.bias, c2.weight, b1.weight, b1.bias, c1.weight, self.ups[j].bias, self.ups[j].weight]
            if self.gates is not None:
                a = self.gates[j]
                out += [a.psi[1].weight, a.psi[1].bias, a.psi[0].weight, a.psi[0].bias,
                        a.W_q[1].weight, a.W_q[1].bias, a.W_q[0].weight, a.W_q[0].bias, a.up.bias, a.up.weight,
                        a.W_x[1].weight, a.W_x[1].bias, a.W_x[0].weight, a.W_x[0].bias]
        for l in (4, 3, 2, 1, 0):
            (c1, b1), (c2, b2) = self.enc[l]
            out += [b2.weight, b2.bias, c2.weight, b1.weight, b1.bias, c1.weight]
        return out

    def graphed_step(self, x, training, save):
        return None

    def refresh_operands(self):
        pass

    # ------------------------------------------------------------------ pieces
    def _conv_bn_relu(self, conv, bn, inp, a_out, training, dp, save=False):
        n, cin, h, w = inp.shape
        k = conv.weight.shape[0]
        dev = inp.device
        y = torch.empty((n, k, h, w), dtype=torch.float32, device=dev)
        ip, ins = _v(inp)
        _lib.call("b200unet_gen_conv3x3", ip, ins, conv.weight.data_ptr(), y.data_ptr(), y.stride(0), n, cin, k, h, w, 0,
                  _stream())
        scale, shift, mean, rstd, count, _ = self._bn_affine(bn, y, training, dp, save)
        ap, ans = _v(a_out)
        _lib.call("b200unet_gen_bn_relu_fwd", y.data_ptr(), y.stride(0), scale.data_ptr(), shift.data_ptr(), ap, ans, n, k,
                  h * w, _stream())
        return (inp, y, scale, shift, mean, rstd, count, not training)

    def _bn_affine(self, bn, y, training, dp, save):
        """BatchNorm2d statistics -> (scale, shift, mean, rstd, count, frozen); updates the running buffers in training."""
        n, k, h, w = y.shape
        dev = y.device
        scale = torch.empty(k, dtype=torch.float32, device=dev)
        shift = torch.empty(k, dtype=torch.float32, device=dev)
        mean = rstd = None
        count = n * h * w
        if not training:
            if bn.running_mean is None:
                raise RuntimeError("eval-mode BatchNorm2d without running statistics (track_running_stats=False) is not supported")
            ops.bn_eval_affine(bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, scale, shift)
            if save:
                mean = torch.empty(k, dtype=torch.float32, device=dev)
                rstd = torch.empty(k, dtype=torch.float32, device=dev)
                ops.bn_eval_stats(bn.running_mean, bn.running_var, bn.eps, mean, rstd)
        else:
            sums = torch.empty(2 * k, dtype=torch.float64, device=dev)
            _lib.call("b200unet_gen_channel_stats", y.data_ptr(), y.stride(0), sums.data_ptr(), n, k, h * w, _stream())
            if dp is not None and dp.sync_bn:
                dp.all_reduce_sum(sums)
                count = count * dp.world_size
            mean = torch.empty(k, dtype=torch.float32, device=dev)
            rstd = torch.empty(k, dtype=torch.float32, device=dev)
            mom, rm, rv, nbt = ops.bn_train_buffers(bn)
            ops.bn_finalize(sums, count, bn.weight, bn.bias, bn.eps, mom, rm, rv, mean, rstd, scale, shift)
            if nbt is not None:
                bn.num_batches_tracked += 1
            ops.bn_cumulative_update(bn, rm, rv)
        return scale, shift, mean, rstd, count, not training

    def _conv1x1_bn(self, seq, inp, act, training, dp, save):
        """nn.Sequential(Conv2d 1x1 + bias, BatchNorm2d[, Sigmoid]) of an Attention_block (Model.py:260-281).
        Returns (output, record for backward)."""
        conv, bn = seq[0], seq[1]
        n, cin, h, w = inp.shape
        j = conv.weight.shape[0]
        y = torch.empty((n, j, h, w), dtype=torch.float32, device=inp.device)
        ip, ins = _v(inp)
        _lib.call("b200unet_gen_conv1x1_fwd", ip, ins, conv.weight.data_ptr(), conv.bias.data_ptr(), y.data_ptr(), n, cin, j,
                  h * w, _stream())
        scale, shift, mean, rstd, count, frozen = self._bn_affine(bn, y, training, dp, save)
        out = torch.empty_like(y)
        _lib.call("b200unet_gen_bn_act_fwd", y.data_ptr(), y.stride(0), scale.data_ptr(), shift.data_ptr(), out.data_ptr(),
                  out.stride(0), n, j, h * w, act, _stream())
        return out, (inp, y, scale, shift, mean, rstd, count, frozen)

    def _gate_fwd(self, att, q, x, out, training, dp, save):
        """Attention_block.forward(q, x) (Model.py:286-296): out = x * sigmoid(BN(psi(relu(BN(W_q(up(q))) + BN(W_x(x))))))."""
        n, cq, hq, wq = q.shape
        _, cx, h, w = x.shape
        if (2 * hq, 2 * wq) != (h, w):
            raise ValueError(f"UNet_attention needs H and W divisible by 16: the gate adds a {2 * hq}x{2 * wq} map to a {h}x{w} one "
                             "(the reference fails the same way)")
        qu = torch.empty((n, cq, h, w), dtype=torch.float32, device=q.device)
        qp, qns = _v(q)
        _lib.call("b200unet_gen_convt2x2_fprop", qp, qns, att.up.weight.data_ptr(), att.up.bias.data_ptr(), qu.data_ptr(),
                  qu.stride(0), n, cq, cq, hq, wq, h, w, 0, 0, _stream())
        q1, rq = self._conv1x1_bn(att.W_q, qu, 0, training, dp, save)
        x1, rx = self._conv1x1_bn(att.W_x, x, 0, training, dp, save)
        e = torch.empty_like(q1)
        _lib.call("b200unet_gen_add_relu", q1.data_ptr(), x1.data_ptr(), e.data_ptr(), e.numel(), _stream())
        a, rp = self._conv1x1_bn(att.psi, e, 2, training, dp, save)
        xp, xns = _v(x)
        op, ons = _v(out)
        _lib.call("b200unet_gen_gate_fwd", xp, xns, a.data_ptr(), op, ons, n, cx, h * w, _stream())
        return (q, x, rq, rx, e, rp, a) if save else None

    def _conv1x1_bn_bwd(self, ctx, seq, rec, g, need_dx=True):
        """Backward of _conv1x1_bn for the identity activation: g = gradient w.r.t. the BatchNorm output."""
        conv, bn = seq[0], seq[1]
        inp, y, scale, shift, mean, rstd, count, frozen = rec
        dy = self._bn_bwd(ctx, bn, (y, scale, shift, mean, rstd, count, frozen), g, relu=False)
        n, cin, h, w = inp.shape
        j = conv.weight.shape[0]
        dx = torch.empty((n, cin, h, w), dtype=torch.float32, device=ctx.dev)
        dw, db = ctx.gbuf(conv.weight), ctx.gbuf(conv.bias)
        ip, ins = _v(inp)
        _lib.call("b200unet_gen_conv1x1_bwd", dy.data_ptr(), ip, ins, conv.weight.data_ptr(), dx.data_ptr(), dx.stride(0),
                  dw.data_ptr(), db.data_ptr(), n, cin, j, h * w, _stream())
        ctx.grads[conv.weight], ctx.grads[conv.bias] = dw, db
        ctx.done(bn.weight, bn.bias, conv.weight, conv.bias)
        return dx

    def _gate_bwd(self, ctx, att, rec, dout):
        """Backward of _gate_fwd: returns (gradient w.r.t. x, gradient w.r.t. q)."""
        q, x, rq, rx, e, rp, a = rec
        n, cx, h, w = x.shape
        cq, hq, wq = q.shape[1], q.shape[2], q.shape[3]
        dx = torch.empty((n, cx, h, w), dtype=torch.float32, device=ctx.dev)
        dpre = torch.empty((n, 1, h, w), dtype=torch.float32, device=ctx.dev)   # gradient at the sigmoid's input
        dp_, dns = _v(dout)
        xp, xns = _v(x)
        _lib.call("b200unet_gen_gate_bwd", dp_, dns, xp, xns, a.data_ptr(), dx.data_ptr(), dx.stride(0), dpre.data_ptr(), n, cx,
                  h * w, _stream())
        de = self._conv1x1_bn_bwd(ctx, att.psi, rp, dpre)
        dsum = torch.empty_like(e)                                              # dQ1 = dX1 = dE * [E > 0]
        _lib.call("b200unet_gen_relu_bwd", de.data_ptr(), e.data_ptr(), dsum.data_ptr(), e.numel(), _stream())
        # _bn_bwd overwrites y with dy but reads g first element-wise per position; W_q and W_x share dsum read-only
        dqu = self._conv1x1_bn_bwd(ctx, att.W_q, rq, dsum)
        dq = self._convt_bwd(ctx, att.up, q, dqu, (n, cq, cq, hq, wq, h, w), (0, 0))
        dx_gate = self._conv1x1_bn_bwd(ctx, att.W_x, rx, dsum)
        _lib.call("b200unet_gen_add_inplace", dx.data_ptr(), dx.stride(0), dx_gate.data_ptr(), dx_gate.stride(0), n, cx * h * w,
                  _stream())
        return dx, dq

    def _dropout(self, t, training):
        """nn.Dropout on `t` (an NCHW view), mask drawn like the reference does; returns the mask or None."""
        net = self.net
        if not (net.dropout and training and net.dropout_p > 0):
            return None
        mask = F.dropout(torch.ones(t.shape, dtype=torch.float32, device=t.device), net.dropout_p, True)
        tp, tns = _v(t)
        _lib.call("b200unet_gen_mul", tp, tns, mask.data_ptr(), t.shape[0], t.shape[1] * t.shape[2] * t.shape[3], _stream())
        return mask

    # ------------------------------------------------------------------ forward
    def forward(self, x, training, save):
        net = self.net
        if x.dim() != 4 or x.shape[1] != net.n_channels:
            raise ValueError(f"UNet expects [B,{net.n_channels},H,W] input, got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("the B200 UNet runs on CUDA (sm_100a) only; there is no CPU fallback")
        x = x.contiguous().float()
        n, _, h, w = x.shape
        if h < 16 or w < 16:
            raise ValueError(f"input {h}x{w} is too small for four 2x2 poolings")
        dev = x.device
        dp = DataParallelContext.current() if training else None
        f = net.initial_feature_map
        ch = [f << l for l in range(5)]
        hs, wsz = [h], [w]
        for _ in range(4):
            hs.append(hs[-1] // 2)
            wsz.append(wsz[-1] // 2)
        cat = []
        for l in range(4):
            padded = (2 * hs[l + 1] != hs[l]) or (2 * wsz[l + 1] != wsz[l])
            mk = torch.zeros if padded else torch.empty
            cat.append(mk((n, 2 * ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev))
        enc_rec, dec_rec = [], []
        inp = x
        for l in range(5):
            (c1, b1), (c2, b2) = self.enc[l]
            a1 = torch.empty((n, ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev)
            r1 = self._conv_bn_relu(c1, b1, inp, a1, training, dp, save)
            if l < 4:
                # UNet: the skip is written straight into the concat buffer; UNet_attention: the gate writes x * A there
                a2 = (cat[l][:, : ch[l]] if self.gates is None
                      else torch.empty((n, ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev))
                r2 = self._conv_bn_relu(c2, b2, a1, a2, training, dp, save)
                pooled = torch.empty((n, ch[l], hs[l + 1], wsz[l + 1]), dtype=torch.float32, device=dev)
                idx = torch.empty((n, ch[l], hs[l + 1], wsz[l + 1]), dtype=torch.uint8, device=dev) if save else None
                ap, ans = _v(a2)
                _lib.call("b200unet_gen_maxpool2x2", ap, ans, pooled.data_ptr(), None if idx is None else idx.data_ptr(), n,
                          ch[l], hs[l], wsz[l], _stream())
                pmask = self._dropout(pooled, training)  # Down: MaxPool2d -> Dropout -> DoubleConv (Model.py:34-39)
                enc_rec.append((r1, r2, a2, idx, pmask))
                inp = pooled
            else:
                a2 = torch.empty((n, ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev)
                r2 = self._conv_bn_relu(c2, b2, a1, a2, training, dp, save)
                enc_rec.append((r1, r2, a2, None, None))
        d_in = enc_rec[4][2]
        for j in range(4):
            l = 3 - j
            up = self.ups[j]
            pt, pl = (hs[l] - 2 * hs[l + 1]) // 2, (wsz[l] - 2 * wsz[l + 1]) // 2  # F.pad (Model.py:69-73)
            grec = None
            if self.gates is not None:  # x_attention = attention(q=x, x=skip) feeds Up as the skip (Model.py:354-364)
                grec = self._gate_fwd(self.gates[j], d_in, enc_rec[l][2], cat[l][:, : ch[l]], training, dp, save)
            dpp, dns = _v(d_in)
            op, ons = _v(cat[l][:, ch[l]:])
            _lib.call("b200unet_gen_convt2x2_fprop", dpp, dns, up.weight.data_ptr(), up.bias.data_ptr(), op, ons, n,
                      ch[l + 1], ch[l], hs[l + 1], wsz[l + 1], hs[l], wsz[l], pt, pl, _stream())
            cmask = self._dropout(cat[l], training)  # Up: cat -> Dropout -> DoubleConv (Model.py:79-83)
            (c1, b1), (c2, b2) = self.dec[j]
            a1 = torch.empty((n, ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev)
            r1 = self._conv_bn_relu(c1, b1, cat[l], a1, training, dp, save)
            a2 = torch.empty((n, ch[l], hs[l], wsz[l]), dtype=torch.float32, device=dev)
            r2 = self._conv_bn_relu(c2, b2, a1, a2, training, dp, save)
            dec_rec.append((d_in, r1, r2, a2, cmask, (pt, pl), grec))
            d_in = a2
        logits = torch.empty((n, net.n_classes, h, w), dtype=torch.float32, device=dev)
        hp_, hns = _v(d_in)
        _lib.call("b200unet_gen_conv1x1_fwd", hp_, hns, self.head.weight.data_ptr(), self.head.bias.data_ptr(),
                  logits.data_ptr(), n, ch[0], net.n_classes, h * w, _stream())
        saved = None
        if save:
            saved = dict(enc=enc_rec, dec=dec_rec, head_in=d_in, shapes=(n, ch, hs, wsz), dp=dp)
        return logits, saved

    # ------------------------------------------------------------------ backward
    class _Ctx:
        """Gradient buffers of one backward pass (plain tensors, or views of the data-parallel flat buffer)."""

        def __init__(self, eng, dp, dev):
            self.dp, self.dev, self.grads = dp, dev, {}
            self.flat = dp.make_flat_grads(eng.params_in_backward_order()) if dp is not None else None

        def gbuf(self, p):
            if self.flat is not None:
                return self.flat.view_for(p)
            return torch.empty_like(p, memory_format=torch.contiguous_format)

        def done(self, *ps):
            if self.flat is not None:
                self.flat.mark_ready(ps)

        def finish(self):
            if self.flat is not None:
                self.flat.finish()
            return self.grads

    def _bn_bwd(self, ctx, bn, rec_bn, g, relu=True):
        """Backward of BatchNorm2d (+ReLU when relu) given g = gradient w.r.t. its output; overwrites y with dy and returns it.
        rec_bn = (y, scale, shift, mean, rstd, count, frozen)."""
        y, scale, shift, mean, rstd, count, frozen = rec_bn
        if mean is None:
            raise RuntimeError("backward of a forward that ran without autograd (no BatchNorm statistics saved)")
        nn_, k, hh, ww = y.shape
        dp = ctx.dp
        gp, gns = _v(g)
        sums = torch.empty(2 * k, dtype=torch.float64, device=ctx.dev)
        _lib.call("b200unet_gen_bn_bwd_reduce", gp, gns, y.data_ptr(), y.stride(0), scale.data_ptr(), shift.data_ptr(),
                  mean.data_ptr(), rstd.data_ptr(), sums.data_ptr(), nn_, k, hh * ww, int(relu), _stream())
        sums_local = None
        if frozen:  # running-statistics BatchNorm: dy = gamma * rstd * da, dgamma / dbeta from the local sums
            sums_local, sums = sums, torch.zeros_like(sums)
        elif dp is not None and dp.sync_bn:
            sums_local = sums.clone()
            dp.all_reduce_sum(sums)
        dgamma, dbeta = ctx.gbuf(bn.weight), ctx.gbuf(bn.bias)
        _lib.call("b200unet_gen_bn_bwd_apply", gp, gns, y.data_ptr(), y.stride(0), bn.weight.data_ptr(), scale.data_ptr(),
                  shift.data_ptr(), mean.data_ptr(), rstd.data_ptr(), sums.data_ptr(), float(count),
                  None if sums_local is None else sums_local.data_ptr(), y.data_ptr(), y.stride(0), dgamma.data_ptr(),
                  dbeta.data_ptr(), nn_, k, hh * ww, int(relu), _stream())
        ctx.grads[bn.weight], ctx.grads[bn.bias] = dgamma, dbeta
        return y  # dy, in place

    def _bn_conv_bwd(self, ctx, conv, bn, rec, g, need_dx):
        inp, y, scale, shift, mean, rstd, count, frozen = rec
        dy = self._bn_bwd(ctx, bn, (y, scale, shift, mean, rstd, count, frozen), g, relu=True)
        nn_, k, hh, ww = y.shape
        dw = ctx.gbuf(conv.weight)
        ip, ins = _v(inp)
        cin = inp.shape[1]
        _lib.call("b200unet_gen_conv3x3_wgrad", ip, ins, dy.data_ptr(), dy.stride(0), dw.data_ptr(), nn_, cin, k, hh, ww,
                  _stream())
        ctx.grads[conv.weight] = dw
        ctx.done(bn.weight, bn.bias, conv.weight)
        if not need_dx:
            return None
        dx = torch.empty((nn_, cin, hh, ww), dtype=torch.float32, device=ctx.dev)
        _lib.call("b200unet_gen_conv3x3", dy.data_ptr(), dy.stride(0), conv.weight.data_ptr(), dx.data_ptr(),
                  dx.stride(0), nn_, k, cin, hh, ww, 1, _stream())
        return dx

    @staticmethod
    def _mul_mask(t, mask):
        if mask is not None:
            tp, tns = _v(t)
            _lib.call("b200unet_gen_mul", tp, tns, mask.data_ptr(), t.shape[0], t.shape[1] * t.shape[2] * t.shape[3], _stream())

    def _head_bwd(self, ctx, head, head_in, dlogits, n, c0, hw):
        g = torch.empty((n, c0) + tuple(head_in.shape[2:]), dtype=torch.float32, device=ctx.dev)
        dwh, dbh = ctx.gbuf(head.weight), ctx.gbuf(head.bias)
        hp_, hns = _v(head_in)
        _lib.call("b200unet_gen_conv1x1_bwd", dlogits.data_ptr(), hp_, hns, head.weight.data_ptr(), g.data_ptr(), g.stride(0),
                  dwh.data_ptr(), dbh.data_ptr(), n, c0, head.weight.shape[0], hw, _stream())
        ctx.grads[head.weight], ctx.grads[head.bias] = dwh, dbh
        ctx.done(head.weight, head.bias)
        return g

    def _convt_bwd(self, ctx, up, d_in, du, shapes, pad, need_dx=True):
        """ConvTranspose2d(k2,s2) backward: weight / bias gradients and (optionally) the input gradient."""
        n, cin, cup, h, w, h2, w2 = shapes
        pt, pl = pad
        db, dwu = ctx.gbuf(up.bias), ctx.gbuf(up.weight)
        dip, dins = _v(d_in)
        up_, uns = _v(du)
        _lib.call("b200unet_gen_convt2x2_wgrad", dip, dins, up_, uns, dwu.data_ptr(), db.data_ptr(), n, cin, cup, h, w, h2, w2,
                  pt, pl, _stream())
        ctx.grads[up.bias], ctx.grads[up.weight] = db, dwu
        ctx.done(up.bias, up.weight)
        if not need_dx:
            return None
        g = torch.empty((n, cin, h, w), dtype=torch.float32, device=ctx.dev)
        _lib.call("b200unet_gen_convt2x2_dgrad", up_, uns, up.weight.data_ptr(), g.data_ptr(), g.stride(0), n, cin, cup, h, w,
                  h2, w2, pt, pl, _stream())
        return g

    def _encoder_bwd(self, ctx, saved, g, skip_grads):
        n, ch, hs, wsz = saved["shapes"]
        g_pool = None
        for l in (4, 3, 2, 1, 0):
            r1, r2, _, idx, pmask = saved["enc"][l]
            (c1, b1), (c2, b2) = self.enc[l]
            if l == 4:
                g1 = self._bn_conv_bwd(ctx, c2, b2, r2, g, True)
            else:
                gs = skip_grads[l]
                self._mul_mask(g_pool, pmask)
                sp, sns = _v(gs)
                _lib.call("b200unet_gen_unpool_add", g_pool.data_ptr(), idx.data_ptr(), sp, sns, n, ch[l], hs[l], wsz[l],
                          _stream())
                g1 = self._bn_conv_bwd(ctx, c2, b2, r2, gs, True)
            g_pool = self._bn_conv_bwd(ctx, c1, b1, r1, g1, need_dx=(l > 0))

    def backward(self, saved, dlogits):
        n, ch, hs, wsz = saved["shapes"]
        ctx = self._Ctx(self, saved["dp"], dlogits.device)
        dlogits = dlogits.contiguous().float()
        g = self._head_bwd(ctx, self.head, saved["head_in"], dlogits, n, ch[0], hs[0] * wsz[0])
        skip_grads = [None] * 4
        for j in (3, 2, 1, 0):
            l = 3 - j
            d_in, r1, r2, _, cmask, (pt, pl), grec = saved["dec"][j]
            (c1, b1), (c2, b2) = self.dec[j]
            g = self._bn_conv_bwd(ctx, c2, b2, r2, g, True)
            dcat = self._bn_conv_bwd(ctx, c1, b1, r1, g, True)
            self._mul_mask(dcat, cmask)
            skip_grads[l] = dcat[:, : ch[l]]
            g = self._convt_bwd(ctx, self.ups[j], d_in, dcat[:, ch[l]:],
                                (n, ch[l + 1], ch[l], hs[l + 1], wsz[l + 1], hs[l], wsz[l]), (pt, pl))
            if grec is not None:  # the gate consumed both the skip and the decoder input q
                skip_grads[l], dq = self._gate_bwd(ctx, self.gates[j], grec, dcat[:, : ch[l]])
                _lib.call("b200unet_gen_add_inplace", g.data_ptr(), g.stride(0), dq.data_ptr(), dq.stride(0), n,
                          ch[l + 1] * hs[l + 1] * wsz[l + 1], _stream())
        self._encoder_bwd(ctx, saved, g, skip_grads)
        return ctx.finish()
