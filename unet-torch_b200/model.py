"""Drop-in `UNet` for the reference's Model.py:95-169, executed by hand-written sm_100a kernels.

The module tree (inc / down1-4 / up1-4 / outc and their children) only HOLDS parameters and buffers so that the
118 state_dict keys, their shapes/dtypes (fp32) and the constructor's RNG consumption match the reference
(Model.py:7-92, 96-140, 167-169). `UNet.forward` never calls those children: the whole encoder-decoder runs as ONE
torch.autograd.Function whose forward/backward are chains of C-ABI launches on NHWC bf16 buffers
(see include/b200unet.h). There is no PyTorch/cuDNN fallback for this model.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from . import ops
from .dist import DataParallelContext

BF16 = torch.bfloat16


def _device_guard(x):
    """Kernels launch on the current device's stream: make the tensor's device current (CPU tensors are rejected later)."""
    import contextlib

    return torch.cuda.device(x.device) if x.is_cuda else contextlib.nullcontext()


# ------------------------------------------------------------------------------------------------ containers
def _double_conv(cin, cout):
    # keys: double_conv.{0,1,3,4}.*  (Model.py:14-23)
    return nn.Sequential(
        nn.Conv2d(cin, cout, kernel_size=3, padding=1, bias=False),
        nn.BatchNorm2d(cout),
        nn.ReLU(inplace=True),
        nn.Conv2d(cout, cout, kernel_size=3, padding=1, bias=False),
        nn.BatchNorm2d(cout),
        nn.ReLU(inplace=True),
    )


class _Holder(nn.Module):
    """Parameter container: its forward is never the product path."""

    def forward(self, *a, **k):  # pragma: no cover - guard
        raise RuntimeError(
            f"{type(self).__name__} is a parameter container of the B200 UNet; call UNet.forward(x) "
            "(sub-blocks are executed by fused sm_100a kernels, not module by module)"
        )


class DoubleConv(_Holder):
    def __init__(self, in_channels, out_channels, mid_channels=None):
        super().__init__()
        if mid_channels not in (None, out_channels):
            raise ValueError("mid_channels != out_channels is not used by UNet and not supported")
        self.double_conv = _double_conv(in_channels, out_channels)


class Down(_Holder):
    def __init__(self, in_channels, out_channels, dropout=False, dropout_p=0.5):
        super().__init__()
        mods = [nn.MaxPool2d(2)]
        if dropout:
            mods.append(nn.Dropout(p=dropout_p))  # shifts DoubleConv to index 2, as in Model.py:34-39
        mods.append(DoubleConv(in_channels, out_channels))
        self.maxpool_conv = nn.Sequential(*mods)


class Up(_Holder):
    def __init__(self, in_channels, out_channels, dropout_flag=False, dropout_p=0.5):
        super().__init__()
        self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
        self.conv = DoubleConv(in_channels, out_channels)
        self.dropout_flag = dropout_flag
        if dropout_flag:
            self.dropout = nn.Dropout(p=dropout_p)


class OutConv(_Holder):
    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=1)


# ------------------------------------------------------------------------------------------------ engine
class _ConvBN:
    """One conv3x3 + BatchNorm2d pair: fp32 master parameters and cached bf16 GEMM operands."""

    def __init__(self, conv: nn.Conv2d, bn: nn.BatchNorm2d, first: bool):
        self.conv, self.bn, self.first = conv, bn, first
        self._ver = None
        self.wf = self.wd = None

    def operands(self):
        w = self.conv.weight
        key = (w._version, w.data_ptr())
        if key != self._ver:
            with torch.no_grad():
                # the operand tensors are re-filled IN PLACE once they exist (captured CUDA graphs hold their addresses)
                if self.first:  # inc.conv1 runs as a 1x1 GEMM over the im2col'ed input: [Cout, 64] operand, no dgrad
                    self.wf, self.wd = ops.prep_first_weight(w.detach(), self.wf), None
                else:
                    self.wf, self.wd = ops.prep_conv3x3_weight(w.detach(), out=(self.wf, self.wd))
            self._ver = key
        return self.wf, self.wd


class _UpOp:
    def __init__(self, up: nn.ConvTranspose2d):
        self.up = up
        self._ver = None
        self.wf = self.wd = None

    def operands(self):
        w = self.up.weight
        key = (w._version, w.data_ptr())
        if key != self._ver:
            with torch.no_grad():
                self.wf, self.wd = ops.prep_convt2x2_weight(w.detach(), out=(self.wf, self.wd))
            self._ver = key
        return self.wf, self.wd


class _BNRef:
    """A BatchNorm2d that does not follow a conv3x3 (the gates' three): what UNetEngine._bn_affine needs of a _ConvBN."""

    def __init__(self, bn: nn.BatchNorm2d):
        self.bn = bn


class _GateOp:
    """One Attention_block (Model.py:257-296) on the tensor-core engine. `up` (ConvTranspose2d C_q -> C_q) is only consumed by
    W_q (1x1, C_q -> C_h), so the two are ONE ConvTranspose2d C_q -> C_h with the composed weight
        W'[c,h,i,j] = sum_d W_up[c,d,i,j] W_q[h,d],   b'[h] = b_q[h] + sum_d W_q[h,d] b_up[d]
    (the C_q-channel upsampled map - 1 GB at level 0 of config 2 - never exists; 3x fewer GEMM FLOPs). The composition and
    its backward (dW_up = dW' W_q, dW_q = sum dW'^T W_up + db' (x) b_up, db_up = W_q^T db', db_q = db') are fp32 GEMMs on
    the weights (tests/test_host_logic.py::test_gate_weight_composition_algebra). Channel counts are padded to a multiple of 64 for the GEMMs (level 0 of a
    width-64 network has C_h = 32): zero weight rows, so the padded channels of the two maps are exact zeros."""

    def __init__(self, att):
        self.att = att
        self.cq = att.up.weight.shape[0]
        self.ch, self.cx = att.W_x[0].weight.shape[0], att.W_x[0].weight.shape[1]
        self.chp = (self.ch + 63) // 64 * 64
        self.bn_q, self.bn_x, self.bn_p = _BNRef(att.W_q[1]), _BNRef(att.W_x[1]), _BNRef(att.psi[1])
        self._ver = None
        self.wc = self.bc = self.wcf = self.wcd = self.wxf = self.wxd = self.bx = None

    def params(self):
        a = self.att
        return [a.up.weight, a.up.bias, a.W_q[0].weight, a.W_q[0].bias, a.W_x[0].weight, a.W_x[0].bias]

    def operands(self):
        """(composed convT fprop operand, its dgrad operand, composed bias, W_x operand, its transpose, W_x bias)."""
        ps = self.params()
        key = tuple((p._version, p.data_ptr()) for p in ps)
        if key != self._ver:
            w_up, b_up, w_q, b_q, w_x, b_x = [p.detach() for p in ps]
            cq, ch, chp, cx = self.cq, self.ch, self.chp, self.cx
            dev = w_up.device
            with torch.no_grad():
                if self.wc is None or self.wc.device != dev:  # allocated once: captured CUDA graphs hold the addresses
                    self.wc = torch.zeros((cq, chp, 2, 2), dtype=torch.float32, device=dev)
                    self.bc = torch.zeros((chp,), dtype=torch.float32, device=dev)
                    self.bx = torch.zeros((chp,), dtype=torch.float32, device=dev)
                    self.wxf = torch.zeros((chp, cx), dtype=BF16, device=dev)
                    self.wxd = torch.zeros((cx, chp), dtype=BF16, device=dev)
                    self.wcf = self.wcd = None
                # per (i,j): W'[:, :, ij] = W_up[:, :, ij] @ W_q^T
                ops.sgemm_strided(w_up, w_q, self.wc, cq, ch, cq, (4 * cq, 4), (1, cq), (4 * chp, 4), batch=4,
                                  batch_strides=(1, 0, 1))
                ops.sgemm_strided(w_q, b_up, self.bc, ch, 1, cq, (cq, 1), (1, 1), (1, 1), bias_m=b_q)
                self.wcf, self.wcd = ops.prep_convt2x2_weight(self.wc, out=(self.wcf, self.wcd))
                w2 = w_x.view(ch, cx)
                self.wxf[:ch].copy_(w2)
                self.wxd[:, :ch].copy_(w2.t())
                self.bx[:ch].copy_(b_x)
            self._ver = key
        return self.wcf, self.wcd, self.bc, self.wxf, self.wxd, self.bx


class _Saved:
    # drop: (int64 device seed or None, drop probability per dropout site) of this forward; backward regenerates the masks
    __slots__ = ("x", "enc", "dec", "head_in", "shapes", "dp", "drop")


def _dc(mod) -> nn.Sequential:
    return mod.double_conv


class UNetEngine:
    """Executes the forward and backward of the whole network as chains of C-ABI launches."""

    def __init__(self, net: "UNet"):
        self.net = net
        inc, downs, decoders = net._topology()
        enc_dc = [_dc(inc)] + [_dc(d.maxpool_conv[-1]) for d in downs]
        self.enc = [(_ConvBN(s[0], s[1], first=(i == 0)), _ConvBN(s[3], s[4], first=False)) for i, s in enumerate(enc_dc)]
        # one entry per decoder (UNet: one; UNet_multitask: two over the same encoder): (ups, dec, head) where
        # decoder index j = 0..3 <-> up1..up4, operating at level 3-j
        self.decoders = []
        for ups, outc in decoders:
            self.decoders.append((
                [_UpOp(u.up) for u in ups],
                [(_ConvBN(_dc(u.conv)[0], _dc(u.conv)[1], False), _ConvBN(_dc(u.conv)[3], _dc(u.conv)[4], False)) for u in ups],
                outc.conv))
        # flat views over all decoders (operand refresh, FusedSGD)
        self.ups = [u for d in self.decoders for u in d[0]]
        self.dec = [c for d in self.decoders for c in d[1]]
        self.head = self.decoders[0][2]
        # UNet_attention: one gate per decoder block (j = 0..3 <-> attenion4..attenion1), else None
        gates = net._attention_gates() if hasattr(net, "_attention_gates") else None
        self.gates = [_GateOp(a) for a in gates] if gates else None
        # the nn.Dropout holder of each dropout site (0..3 = down1..4 after the pooling, 4..7 = up1..4 after the concat), or
        # None; their `p` is read at every forward, as the reference's modules do
        self.drop = ([next((m for m in d.maxpool_conv if isinstance(m, nn.Dropout)), None) for d in downs]
                     + [u.dropout if getattr(u, "dropout_flag", False) else None for u in decoders[0][0]])
        self._graphs = {}     # (shape, device, training, save) -> _GraphedStep
        self._seen = set()    # keys that already ran once eagerly (kernel attributes configured, allocator warm)
        # B200UNET_WGRAD_STREAM=1: weight-gradient kernels on a second stream (nothing downstream in backward depends on
        # them), overlapping the bandwidth-bound BN/ReLU backward of the next layer. Measured neutral on B200 (687-691
        # img/s either way: the step runs at the 1000 W power cap, so co-scheduling does not add throughput) -> off.
        # eval forward without saving for backward: BN + ReLU are folded into the conv epilogues (the four pooled layers
        # are followed by a plain max-pool pass); B200UNET_FOLD_EVAL_BN=0 keeps the separate BN-apply pass
        self.fold_eval_bn = os.environ.get("B200UNET_FOLD_EVAL_BN", "1") not in ("", "0")
        # inc.conv1 with the im2col rows built in shared memory (no 537 MB im2col tensor); B200UNET_FIRST_FUSED=0 = round-1 path
        self.first_fused = os.environ.get("B200UNET_FIRST_FUSED", "1") not in ("", "0")
        # ... but under data parallel it pays: the weight-gradient kernels fill the bubbles in which the main stream waits for
        # the slowest rank inside a SyncBN exchange (8 x B200: 5364 -> 5431 img/s, +1.3 %). Unset = on under data parallel only.
        env = os.environ.get("B200UNET_WGRAD_STREAM", "")
        self.wgrad_overlap = None if env == "" else env != "0"
        self._wgrad_stream = None
        # Test hook (tests/test_gpu_replay.py): set to a list and every operator of forward / backward appends a record of
        # the tensors it read and wrote (tensors that are later overwritten in place are cloned), so the dataflow can be
        # replayed operator by operator on the host. None = off (no cost).
        self.trace = None

    def _tr(self, kind, **kw):
        if self.trace is not None:
            self.trace.append((kind, kw))

    def _drop_ps(self, training):
        """Drop probability of each of the 8 dropout sites for this forward (0.0 = the site does nothing)."""
        return tuple(float(m.p) if (training and m is not None) else 0.0 for m in self.drop)

    def _dropout(self, t, site, seed, p, sums=None, backward=False):
        before = t.clone() if self.trace is not None else None
        ops.dropout_mul(t, site, seed, p, sums=sums)
        if before is not None:
            self._tr("dropout", site=site, p=p, seed=seed, before=before, after=t.clone(), backward=backward)

    def graphed_step(self, x, training, save):
        """The captured step for this input, or None when the call must run eagerly: graphs disabled, data parallel
        over a backend whose collectives cannot be captured, or first call for this shape (eager warm-up: kernel
        attributes, allocator, NCCL communicators)."""
        net = self.net
        if not net._cuda_graphs or not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
            return None
        dp = DataParallelContext.current() if training else None
        if dp is not None and not dp.graph_capturable:
            return None
        if torch.cuda.is_current_stream_capturing():
            return None
        # the drop probabilities are launch arguments of the captured graph (and decide which passes it holds)
        key = (tuple(x.shape), x.device.index, bool(training), bool(save), dp is not None, self._drop_ps(training))
        st = self._graphs.get(key)
        if st is None:
            if key not in self._seen:
                self._seen.add(key)
                return None
            st = self._graphs[key] = _GraphedStep(self, x, training, save)
        return st

    def refresh_operands(self):
        """Re-derive the bf16 GEMM operands of every parameter whose version changed (no-op otherwise)."""
        for c1, c2 in self.enc + self.dec:
            c1.operands()
            c2.operands()
        for u in self.ups:
            u.operands()
        for g in self.gates or ():
            g.operands()

    # parameters in the order their gradients are produced by backward (used for DP bucketing)
    def params_in_backward_order(self):
        out = []
        for ups, dec, head in reversed(self.decoders):
            out += [head.weight, head.bias]
            for j in (3, 2, 1, 0):
                c1, c2 = dec[j]
                out += [c2.bn.weight, c2.bn.bias, c2.conv.weight, c1.bn.weight, c1.bn.bias, c1.conv.weight,
                        ups[j].up.bias, ups[j].up.weight]
                if self.gates is not None:
                    a = self.gates[j].att
                    out += [a.psi[1].weight, a.psi[1].bias, a.psi[0].weight, a.psi[0].bias, a.W_q[1].weight, a.W_q[1].bias,
                            a.W_x[1].weight, a.W_x[1].bias, a.W_x[0].weight, a.W_x[0].bias, a.W_q[0].weight, a.W_q[0].bias,
                            a.up.weight, a.up.bias]
        for l in (4, 3, 2, 1, 0):
            c1, c2 = self.enc[l]
            out += [c2.bn.weight, c2.bn.bias, c2.conv.weight, c1.bn.weight, c1.bn.bias, c1.conv.weight]
        return out

    # ------------------------------------------------------------------ BN helpers
    def _bn_affine(self, cb: _ConvBN, stats_partial, rows, count, training, dp, need_stats=False):
        bn = cb.bn
        c = bn.num_features
        dev = bn.weight.device
        scale = torch.empty(c, dtype=torch.float32, device=dev)
        shift = torch.empty(c, dtype=torch.float32, device=dev)
        if not training:
            if bn.running_mean is None:
                raise RuntimeError("eval-mode BatchNorm2d without running statistics (track_running_stats=False) is not supported")
            ops.bn_eval_affine(bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, scale, shift)
            mean = rstd = None
            if need_stats:  # eval forward under autograd (frozen-BN fine-tuning, saliency): backward needs mean / rstd
                mean = torch.empty(c, dtype=torch.float32, device=dev)
                rstd = torch.empty(c, dtype=torch.float32, device=dev)
                ops.bn_eval_stats(bn.running_mean, bn.running_var, bn.eps, mean, rstd)
            return scale, shift, mean, rstd, count
        mean = torch.empty(c, dtype=torch.float32, device=dev)
        rstd = torch.empty(c, dtype=torch.float32, device=dev)
        stats_partial, rows = ops.fold_rows(stats_partial, rows, 2 * c)
        mom = bn.momentum if bn.momentum is not None else 0.1
        track = bn.track_running_stats and bn.running_mean is not None
        if dp is None or not dp.sync_bn:  # single GPU: partial rows -> statistics -> affine -> running buffers, one launch
            ops.bn_reduce_finalize(stats_partial, rows, count, bn.weight, bn.bias, bn.eps, mom,
                                   bn.running_mean if track else None, bn.running_var if track else None,
                                   bn.num_batches_tracked if track else None, mean, rstd, scale, shift)
            return scale, shift, mean, rstd, count
        if dp.supports_rows(c):  # SyncBN over NVLink: rows -> exchange -> finalise in one multi-block kernel
            count = count * dp.world_size
            dp.bn_rows_sync_finalize(stats_partial, rows, count, bn, bn.eps, mom, track, mean, rstd, scale, shift)
            return scale, shift, mean, rstd, count
        sums = torch.empty(2 * c, dtype=torch.float64, device=dev)
        ops.bn_reduce_partials(stats_partial, rows, c, sums)
        if dp is not None and dp.sync_bn:
            count = count * dp.world_size
            if dp.has_nvl and 2 * c <= dp.nvl_max_doubles:  # one kernel: NVLink one-shot all-reduce of [sum, sum^2] + finalisation
                dp.bn_sync_finalize(sums, count, bn, bn.eps, mom, track, mean, rstd, scale, shift)
                if track:
                    bn.num_batches_tracked += 1
                return scale, shift, mean, rstd, count
            dp.all_reduce_sum(sums)
        ops.bn_finalize(sums, count, bn.weight, bn.bias, bn.eps, mom, bn.running_mean if track else None,
                        bn.running_var if track else None, mean, rstd, scale, shift)
        if track:
            bn.num_batches_tracked += 1
        return scale, shift, mean, rstd, count

    # ------------------------------------------------------------------ attention gates
    def _gate_forward(self, gate: _GateOp, q, xs, out, training, dp, save):
        """Attention_block.forward(q, x) (Model.py:286-296): out = xs * sigmoid(BN(psi(relu(BN(W_q(up(q))) + BN(W_x(xs)))))).
        q: [n, h/2, w/2, C_q], xs: [n, h, w, C_x], out: the skip half of the concat buffer."""
        n, h, w, cx = xs.shape
        dev = xs.device
        ch, chp = gate.ch, gate.chp
        wcf, _, bc, wxf, _, bx = gate.operands()
        q1 = torch.empty((n, h, w, chp), dtype=BF16, device=dev)   # W_q(up(q)) before its BatchNorm
        x1 = torch.empty((n, h, w, chp), dtype=BF16, device=dev)   # W_x(xs) before its BatchNorm
        rows_q, rows_x = ops.convt2x2_stat_rows(n, h // 2, w // 2), ops.conv1x1_stat_rows(n, h, w)
        st_q = st_x = None
        if training:
            st_q = torch.empty(rows_q * 2 * ch, dtype=torch.float32, device=dev)
            st_x = torch.empty(rows_x * 2 * ch, dtype=torch.float32, device=dev)
            ops.convt2x2_stats(q, wcf, bc, q1, st_q, ch)
        else:
            ops.convt2x2(q, wcf, bc, q1)
        ops.conv1x1(xs, wxf, bx, x1, st_x, ch)
        count = n * h * w
        aq = self._bn_affine(gate.bn_q, st_q, rows_q, count, training, dp, need_stats=save)
        ax = self._bn_affine(gate.bn_x, st_x, rows_x, count, training, dp, need_stats=save)
        psi = gate.att.psi[0]
        w_psi, b_psi = psi.weight.detach().view(-1), psi.bias.detach()
        s = torch.empty((n, h, w), dtype=torch.float32, device=dev)
        rows_p = ops.gate_stat_rows(count, ch)
        st_p = torch.empty(rows_p * 2, dtype=torch.float32, device=dev) if training else None
        q1v, x1v = q1[..., :ch], x1[..., :ch]
        ops.gate_psi_fwd(q1v, x1v, aq[0], aq[1], ax[0], ax[1], w_psi, b_psi, s, st_p)
        ap = self._bn_affine(gate.bn_p, st_p, rows_p, count, training, dp, need_stats=save)
        ops.gate_apply_fwd(xs, s, ap[0], ap[1], out)
        if self.trace is not None:
            self._tr("gate", gate=gate, q=q, x=xs, q1=q1v.clone(), x1=x1v.clone(), s=s, aq=aq, ax=ax, ap=ap, out=out,
                     training=training)
        if not save:
            return None
        return (q1, x1, s, aq, ax, ap, xs, not training)

    def _gate_backward(self, gate: _GateOp, grec, g, q, gbuf, done, grads, sync, on_wgrad_stream, keep_alive):
        """Backward of _gate_forward. g: gradient w.r.t. the gated skip (a slice of dcat). Returns (gradient w.r.t. xs,
        gradient w.r.t. q). The two maps q1 / x1 are overwritten with their gradients."""
        q1, x1, s, aq, ax, ap, xs, frozen = grec
        att = gate.att
        n, h, w, cx = xs.shape
        dev = xs.device
        ch, chp, cq = gate.ch, gate.chp, gate.cq
        _, wcd, _, _, wxd, _ = gate.operands()
        q1v, x1v = q1[..., :ch], x1[..., :ch]
        scale_p, shift_p, mean_p, rstd_p, count = ap
        psi, bn_p, bn_q, bn_x = att.psi[0], att.psi[1], att.W_q[1], att.W_x[1]
        w_psi = psi.weight.detach().view(-1)
        # ---- the product x * A and the sigmoid (the g * A term of the skip gradient joins the W_x backward-data below)
        dz = torch.empty((n, h, w), dtype=torch.float32, device=dev)
        sums2 = torch.empty(2, dtype=torch.float64, device=dev)
        ops.gate_apply_bwd(g, xs, s, scale_p, shift_p, mean_p, rstd_p, None, dz, sums2)
        sums2_local = sums2
        if frozen:
            sums2 = torch.zeros_like(sums2)       # running statistics: no batch-statistics correction terms
        elif sync is not None:
            sums2_local = sums2.clone()
            sync.all_reduce_sum(sums2)
        # ---- BatchNorm2d(1) + psi + ReLU + the two BatchNorms
        ds = torch.empty((n, h, w), dtype=torch.float32, device=dev)
        sums = torch.empty(4 * ch + 8, dtype=torch.float64, device=dev)
        ops.gate_bwd_reduce(q1v, x1v, aq[:4], ax[:4], w_psi, s, dz, bn_p.weight.detach(), mean_p, rstd_p, sums2, count, ds, sums)
        sums_local = None
        if frozen:
            sums_local, sums = sums, torch.zeros_like(sums)
        elif sync is not None:
            sums_local = sums.clone()
            sync.all_reduce_sum(sums)
        names = (bn_q.weight, bn_q.bias, bn_x.weight, bn_x.bias, psi.weight, psi.bias, bn_p.weight, bn_p.bias)
        outs = [gbuf(p) for p in names]
        dbias = torch.empty(2 * ch, dtype=torch.float32, device=dev)
        ops.gate_bwd_apply(q1v, x1v, aq[:4], ax[:4], bn_q.weight.detach(), bn_x.weight.detach(), w_psi, ds, sums, sums_local,
                           sums2_local, aq[4], outs, dbias)
        for p, o in zip(names, outs):
            grads[p] = o
        done(*names)
        dq1, dx1 = q1, x1   # gradients at the two pre-BatchNorm maps (padded channels are still exact zeros)
        # ---- W_x: backward-data into the skip gradient, weight and bias gradients
        dxs = torch.empty((n, h, w, cx), dtype=BF16, device=dev)
        ops.conv1x1(dx1, wxd, None, dxs)
        ops.gate_dx(g, s, scale_p, shift_p, dxs)   # + g * A in the same pass
        wx, bxp = att.W_x[0].weight, att.W_x[0].bias
        dwx, dbx = gbuf(wx), gbuf(bxp)
        on_wgrad_stream(lambda: ops.conv1x1_wgrad(xs, dx1, dwx))
        dbx.copy_(dbias[ch:])
        grads[wx], grads[bxp] = dwx, dbx
        done(wx, bxp)
        # ---- the composed ConvTranspose2d: backward-data into q's gradient, then the weight gradient split into up / W_q
        dq = torch.empty((n, h // 2, w // 2, cq), dtype=BF16, device=dev)
        ops.convt2x2_dgrad(dq1, wcd, dq)
        w_up, b_up, w_q, b_q = att.up.weight, att.up.bias, att.W_q[0].weight, att.W_q[0].bias
        dwup, dbup, dwq, dbq = gbuf(w_up), gbuf(b_up), gbuf(w_q), gbuf(b_q)

        def weight_side():
            dwc = torch.empty((cq, chp, 2, 2), dtype=torch.float32, device=dev)
            ops.convt2x2_wgrad(q, dq1, dwc)
            # dW_up[c,d,ij] = sum_h dW'[c,h,ij] W_q[h,d];  dW_q[h,d] = sum_{c,ij} dW'[c,h,ij] W_up[c,d,ij] + db'[h] b_up[d]
            ops.sgemm_strided(dwc, w_q.detach(), dwup, cq, cq, ch, (4 * chp, 4), (cq, 1), (4 * cq, 4), batch=4,
                              batch_strides=(1, 0, 1))
            part = torch.empty((4, ch, cq), dtype=torch.float32, device=dev)  # one partial product per (i,j), in parallel
            ops.sgemm_strided(dwc, w_up.detach(), part, ch, cq, cq, (4, 4 * chp), (4 * cq, 4), (cq, 1), batch=4,
                              batch_strides=(1, 1, ch * cq))
            ops.sum_batches(part, dwq)
            # ... + db' (x) b_up: W_q also enters the composed bias b' = b_q + W_q b_up
            ops.sgemm_strided(dbias, b_up.detach(), dwq, ch, cq, 1, (1, 1), (1, 1), (cq, 1), accumulate=True)

        # (the closure only touches tensors that live until backward returns - q, the saved maps, parameters, gradient buffers,
        # dbias through keep_alive - and what it allocates itself: the side stream is invisible to the caching allocator)
        keep_alive.append(dbias)
        on_wgrad_stream(weight_side)
        # b' = b_q + W_q b_up:  db_q = db',  db_up[d] = sum_h W_q[h,d] db'[h]
        ops.sgemm_strided(w_q.detach(), dbias, dbup, cq, 1, ch, (1, cq), (1, 1), (1, 1))
        dbq.copy_(dbias[:ch])
        grads[w_up], grads[b_up], grads[w_q], grads[b_q] = dwup, dbup, dwq, dbq
        done(w_up, b_up, w_q, b_q)
        if self.trace is not None:
            self._tr("gate_bwd", gate=gate, g=g, dxs=dxs, dq=dq, dq1=dq1[..., :ch], dx1=dx1[..., :ch], ds=ds, dz=dz,
                     grads={p: grads[p] for p in (*names, wx, bxp, w_up, b_up, w_q, b_q)})
        return dxs, dq

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor, training: bool, save: bool, head: str = "logits", head_arg: float = 0.0):
        """head: "logits" (Model.py:152, fp32 NCHW), or one of the fused inference epilogues "mask" (uint8 class mask,
        test_mc3serousv5.py:879-887) / "sigmoid" (channel 0 thresholded at `head_arg`, test.py:393-399) / "density"
        ((relu(z) / head_arg, per-map sums), test_mc3serousv5.py:961-974)."""
        net = self.net
        if x.dim() != 4 or x.shape[1] != net.n_channels:
            raise ValueError(f"UNet expects [B,{net.n_channels},H,W] input, got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("the B200 UNet runs on CUDA (sm_100a) only; there is no CPU fallback")
        n, _, h, w = x.shape
        if h % 16 or w % 16:
            raise ValueError(f"tensor-core engine: H and W must be multiples of 16 (got {h}x{w}); the generic engine "
                             "takes other sizes")
        x = x.contiguous().float()
        dev = x.device
        dp = DataParallelContext.current() if training else None
        f = net.initial_feature_map
        ch = [f * (1 << l) for l in range(5)]
        hs = [h >> l for l in range(5)]
        wsz = [w >> l for l in range(5)]
        # concat buffers of decoder levels 0..3: [skip | upsampled]
        cat = [torch.empty((n, hs[l], wsz[l], 2 * ch[l]), dtype=BF16, device=dev) for l in range(4)]
        saved = _Saved() if save else None
        enc_rec, dec_rec = [], []
        # dropout: one seed per training forward, drawn on the device from torch's CUDA generator (a captured graph draws a
        # new one at every replay); the masks are functions of (seed, site, element) and are regenerated in backward
        drop_ps = self._drop_ps(training)
        seed = torch.empty(1, dtype=torch.int64, device=dev).random_() if any(p > 0 for p in drop_ps) else None

        def conv_bn_relu(cb: _ConvBN, inp, c_out, hh, ww, a_out, pooled=None, pool_idx=None):
            if not training and not save and self.fold_eval_bn:
                # inference: BatchNorm (running statistics) + ReLU folded into the conv epilogue; y never reaches HBM
                scale, shift, _, _, _ = self._bn_affine(cb, None, 0, n * hh * ww, False, None)
                if cb.first and self.first_fused:
                    ops.conv3x3_first_tc_bn_relu(inp, cb.operands()[0], scale, shift, a_out)
                elif cb.first:
                    col = torch.empty((n, hh, ww, 64), dtype=BF16, device=dev)
                    ops.first_im2col(inp, col)
                    ops.conv1x1_c64_bn_relu(col, cb.operands()[0], scale, shift, a_out)
                else:
                    ops.conv3x3_bn_relu(inp, cb.operands()[0], scale, shift, a_out)
                if pooled is not None:
                    ops.maxpool2x2(a_out, pooled)
                return None
            y = torch.empty((n, hh, ww, c_out), dtype=BF16, device=dev)
            stats = None
            if cb.first:
                rows = ops.conv1x1_c64_stat_rows(n, hh, ww, c_out)
                if training:
                    stats = torch.empty(rows * 2 * c_out, dtype=torch.float32, device=dev)
                w1, _ = cb.operands()
                if self.first_fused:  # im2col rows built in shared memory; the fp32 input itself is saved for the wgrad
                    ops.conv3x3_first_tc(inp, w1, y, stats)
                else:
                    col = torch.empty((n, hh, ww, 64), dtype=BF16, device=dev)
                    ops.first_im2col(inp, col)
                    inp = col  # saved for the weight gradient
                    ops.conv1x1_c64(col, w1, y, stats)
            else:
                rows = ops.conv3x3_stat_rows(n, hh, ww, inp.shape[3], c_out)
                if training:
                    stats = torch.empty(rows * 2 * c_out, dtype=torch.float32, device=dev)
                wf, _ = cb.operands()
                ops.conv3x3(inp, wf, y, stats)
            scale, shift, mean, rstd, count = self._bn_affine(cb, stats, rows, n * hh * ww, training, dp, need_stats=save)
            ops.bn_relu_fwd(y, scale, shift, a_out, pooled, pool_idx)
            if self.trace is not None:
                self._tr("conv_bn_relu", cb=cb, x=(x if cb.first else inp), y=y.clone(), scale=scale, shift=shift, mean=mean,
                         rstd=rstd, count=count, a=a_out, pooled=pooled, pool_idx=pool_idx, training=training)
            return (inp, y, scale, shift, mean, rstd, count, not training)

        # ---- encoder
        inp = x
        for l in range(5):
            c1, c2 = self.enc[l]
            a1 = torch.empty((n, hs[l], wsz[l], ch[l]), dtype=BF16, device=dev)
            r1 = conv_bn_relu(c1, inp, ch[l], hs[l], wsz[l], a1)
            if l < 4:
                # the skip activation goes straight into the concat buffer - unless an attention gate sits in between
                a2 = cat[l][..., : ch[l]] if self.gates is None else torch.empty((n, hs[l], wsz[l], ch[l]), dtype=BF16, device=dev)
                pooled = torch.empty((n, hs[l + 1], wsz[l + 1], ch[l]), dtype=BF16, device=dev)
                idx = torch.empty((n, hs[l + 1], wsz[l + 1], ch[l]), dtype=torch.uint8, device=dev) if save else None
                r2 = conv_bn_relu(c2, a1, ch[l], hs[l], wsz[l], a2, pooled, idx)
                if drop_ps[l] > 0:  # Down: MaxPool2d -> Dropout (the pool indices are those of the undropped maxima)
                    self._dropout(pooled, l, seed, drop_ps[l])
                inp = pooled
            else:
                a2 = torch.empty((n, hs[l], wsz[l], ch[l]), dtype=BF16, device=dev)
                idx = None
                r2 = conv_bn_relu(c2, a1, ch[l], hs[l], wsz[l], a2)
            enc_rec.append((r1, r2, a2, idx))
        # ---- decoder(s)
        outs, heads_in = [], []
        for k, (ups, dec, head_conv) in enumerate(self.decoders):
            if k == 0:
                catk = cat
            else:  # a further decoder over the same encoder: its own concat buffers, skip halves copied in
                catk = [torch.empty_like(c) for c in cat]
                for l in range(4):
                    ops.nhwc_copy(cat[l][..., : ch[l]], catk[l][..., : ch[l]])
            d_in = enc_rec[4][2]
            rec = []
            for j in range(4):
                l = 3 - j
                upo = ups[j]
                grec = None
                if self.gates is not None:  # x_l_attention = attenion_l(q = d_in, x = skip) -> skip half of the concat buffer
                    grec = self._gate_forward(self.gates[j], d_in, enc_rec[l][2], catk[l][..., : ch[l]], training, dp, save)
                wf, _ = upo.operands()
                ops.convt2x2(d_in, wf, upo.up.bias.detach(), catk[l][..., ch[l]:])
                self._tr("convt", up=upo, x=d_in, out=catk[l][..., ch[l]:], cat=catk[l], skip=enc_rec[l][2])
                if drop_ps[4 + j] > 0:  # Up: cat -> Dropout over both halves; nothing reads the skip half after this
                    self._dropout(catk[l], 4 + j, seed, drop_ps[4 + j])
                c1, c2 = dec[j]
                a1 = torch.empty((n, hs[l], wsz[l], ch[l]), dtype=BF16, device=dev)
                r1 = conv_bn_relu(c1, catk[l], ch[l], hs[l], wsz[l], a1)
                a2 = torch.empty((n, hs[l], wsz[l], ch[l]), dtype=BF16, device=dev)
                r2 = conv_bn_relu(c2, a1, ch[l], hs[l], wsz[l], a2)
                rec.append((d_in, r1, r2, a2, grec))
                d_in = a2
            dec_rec.append(rec)
            heads_in.append(d_in)
            # ---- head
            hw_, hb_ = head_conv.weight.detach(), head_conv.bias.detach()
            if head == "mask":
                outs.append(ops.head_mask(d_in, hw_, hb_))
            elif head == "sigmoid":
                outs.append(ops.head_sigmoid_mask(d_in, hw_, hb_, head_arg))
            elif head == "density":
                outs.append(ops.head_density(d_in, hw_, hb_, head_arg))
            else:
                logits = torch.empty((n, hw_.shape[0], h, w), dtype=torch.float32, device=dev)
                outs.append(ops.head_fprop(d_in, hw_, hb_, logits))
                self._tr("head", conv=head_conv, x=d_in, logits=logits)
        out = outs[0] if len(outs) == 1 else tuple(outs)
        if save and head == "logits":
            saved.x, saved.enc, saved.dec, saved.head_in = x, enc_rec, dec_rec, heads_in
            saved.shapes = (n, ch, hs, wsz)
            saved.dp = dp
            saved.drop = (seed, drop_ps)
        return out, saved

    # ------------------------------------------------------------------ backward
    def backward(self, saved: _Saved, dlogits):
        """dlogits: one tensor, or one per decoder (None = that output did not take part in the loss)."""
        n, ch, hs, wsz = saved.shapes
        dlogits_all = list(dlogits) if isinstance(dlogits, (tuple, list)) else [dlogits]
        ref = next(d for d in dlogits_all if d is not None)
        dev = ref.device
        dlogits_all = [(torch.zeros((n, dc[2].weight.shape[0], hs[0], wsz[0]), dtype=torch.float32, device=dev)
                        if d is None else d.contiguous().float()) for d, dc in zip(dlogits_all, self.decoders)]
        dp = saved.dp
        seed, drop_ps = saved.drop
        grads = {}
        flat = dp.make_flat_grads(self.params_in_backward_order()) if dp is not None else None

        def gbuf(p):
            if flat is not None:
                return flat.view_for(p)
            return torch.empty_like(p, memory_format=torch.contiguous_format)

        def done(*ps):
            if flat is not None:
                flat.mark_ready(ps)

        sync = dp if (dp is not None and dp.sync_bn) else None  # SyncBN: ops.bn_relu_bwd exchanges the sums through it
        side = None
        if self.wgrad_overlap if self.wgrad_overlap is not None else dp is not None:
            if self._wgrad_stream is None:
                self._wgrad_stream = torch.cuda.Stream(device=dev)
            side = self._wgrad_stream
            side.wait_stream(torch.cuda.current_stream())  # fork (also puts the stream into an ongoing graph capture)
            if dp is not None:
                dp.extra_wait_streams = [side]

        def on_wgrad_stream(launch):
            """Run `launch()` (weight-gradient kernels reading tensors that stay alive until backward returns) on the
            side stream, ordered after everything enqueued so far."""
            if side is None:
                return launch()
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(side):
                side.wait_event(ev)
                launch()

        def bn_conv_bwd(cb: _ConvBN, rec, g1, g_pool, pool_idx, hh, ww, need_dx, dx_colsum=None, pre=None, fuse_next=None):
            """Backward of one conv+BN+ReLU. pre: (partial, rows) if the kernel that produced g1 already reduced this
            layer's BatchNorm sums; fuse_next: the record of the layer in FRONT (whose output is this conv's input): its
            BatchNorm reduction is fused into this layer's backward-data launch when a fused form exists. Returns dx, or
            (dx, pre_for_next) when fuse_next is given."""
            inp, y, scale, shift, mean, rstd, count, frozen = rec
            bn = cb.bn
            dgamma, dbeta = gbuf(bn.weight), gbuf(bn.bias)
            ops.bn_relu_bwd(g1, g_pool, pool_idx, y, bn.weight.detach(), scale, shift, mean, rstd, y, dgamma, dbeta,
                            count=count, allreduce=None if frozen else sync, frozen=frozen, pre=pre)
            dy = y  # dy overwrote y in place
            rec_t = dict(cb=cb, g1=g1, g_pool=g_pool, pool_idx=pool_idx, dy=dy, dgamma=dgamma, dbeta=dbeta, inp=inp) \
                if self.trace is not None else None
            dw = gbuf(cb.conv.weight)
            if cb.first and inp.dtype == torch.float32:
                on_wgrad_stream(lambda: ops.conv3x3_first_tc_wgrad(inp, dy, dw))
            elif cb.first:
                on_wgrad_stream(lambda: ops.conv1x1_c64_wgrad(inp, dy, dw))
            else:
                on_wgrad_stream(lambda: ops.conv3x3_wgrad(inp, dy, dw))
            grads[bn.weight], grads[bn.bias], grads[cb.conv.weight] = dgamma, dbeta, dw
            done(bn.weight, bn.bias, cb.conv.weight)
            if rec_t is not None:
                rec_t["dw"] = dw
                self.trace.append(("conv_bn_relu_bwd", rec_t))
            if not need_dx:
                return None
            _, wd = cb.operands()
            cdx = wd.shape[0]
            dx = torch.empty((n, hh, ww, cdx), dtype=BF16, device=dev)
            if fuse_next is not None:
                _, y_n, scale_n, shift_n, mean_n, rstd_n, _, _ = fuse_next
                pre_n = ops.conv3x3_dgrad_bnred(dy, wd, dx, y_n, scale_n, shift_n, mean_n, rstd_n)
                if pre_n is None:
                    ops.conv3x3(dy, wd, dx)
                if rec_t is not None:
                    rec_t["dx"] = dx.clone() if len(self.decoders) > 1 else dx
                return dx, pre_n
            if dx_colsum is None:
                ops.conv3x3(dy, wd, dx)
            else:
                # per-channel pixel sums of dx[..., lo:] from the conv epilogue's statistics rows (convT bias gradient)
                lo, out = dx_colsum
                rows = ops.conv3x3_stat_rows(n, hh, ww, dy.shape[3], cdx)
                part = torch.empty(rows * 2 * cdx, dtype=torch.float32, device=dev)
                ops.conv3x3(dy, wd, dx, part)
                ops.partial_colsum(part, rows, 2 * cdx, lo, cdx - lo, out)
            if rec_t is not None:  # two decoders accumulate the skip gradients in place later on: keep this operator's own output
                rec_t["dx"] = dx.clone() if len(self.decoders) > 1 else dx
            return dx

        # ---- decoder(s): head, then up4 -> up1; the skip and bottleneck gradients of several decoders are summed
        skip_grads = [None] * 4
        keep_alive = []   # tensors read on the weight-gradient stream that nothing else references until backward returns
        g5 = None
        for k in reversed(range(len(self.decoders))):
            ups, dec, head_conv = self.decoders[k]
            dz = dlogits_all[k]
            hw_, hb_ = head_conv.weight, head_conv.bias
            g = torch.empty((n, hs[0], wsz[0], ch[0]), dtype=BF16, device=dev)
            dwh, dbh = gbuf(hw_), gbuf(hb_)
            ops.head_bwd(dz, saved.head_in[k], hw_.detach(), g, dwh, dbh)
            self._tr("head_bwd", conv=head_conv, dz=dz, x=saved.head_in[k], g=g, dw=dwh, db=dbh)
            grads[hw_], grads[hb_] = dwh, dbh
            done(hw_, hb_)
            for j in (3, 2, 1, 0):
                l = 3 - j
                d_in, r1, r2, _, grec = saved.dec[k][j]
                c1, c2 = dec[j]
                g, pre = bn_conv_bwd(c2, r2, g, None, None, hs[l], wsz[l], True, fuse_next=r1)
                upo = ups[j]
                db, dwu = gbuf(upo.up.bias), gbuf(upo.up.weight)
                p_up = drop_ps[4 + j]
                dcat = bn_conv_bwd(c1, r1, g, None, None, hs[l], wsz[l], True, dx_colsum=None if p_up > 0 else (ch[l], db),
                                   pre=pre)
                if p_up > 0:  # the concat's mask on both halves; the bias gradient sums the masked upsampled half
                    self._dropout(dcat, 4 + j, seed, p_up, sums=(ch[l], db), backward=True)
                dq_gate = None
                # the side stream reads dcat's upsampled half (ConvTranspose2d weight gradient below). A plain single-decoder
                # network keeps the storage referenced through skip_grads; behind a gate, or for a second decoder, nothing else
                # would - and the caching allocator does not see the side stream
                keep_alive.append(dcat)
                if grec is not None:  # through the attention gate: gradient w.r.t. the skip activation and w.r.t. q = d_in
                    skip_grads[l], dq_gate = self._gate_backward(self.gates[j], grec, dcat[..., : ch[l]], d_in, gbuf, done, grads,
                                                                 sync, on_wgrad_stream, keep_alive)
                elif skip_grads[l] is None:
                    skip_grads[l] = dcat[..., : ch[l]]
                else:
                    ops.nhwc_add(skip_grads[l], dcat[..., : ch[l]])
                du = dcat[..., ch[l]:]
                on_wgrad_stream(lambda d_in=d_in, du=du, dwu=dwu: ops.convt2x2_wgrad(d_in, du, dwu))
                grads[upo.up.bias], grads[upo.up.weight] = db, dwu
                done(upo.up.bias, upo.up.weight)
                _, wd = upo.operands()
                g = torch.empty((n, hs[l + 1], wsz[l + 1], ch[l + 1]), dtype=BF16, device=dev)
                ops.convt2x2_dgrad(du, wd, g)
                if dq_gate is not None:
                    ops.nhwc_add(g, dq_gate)
                if self.trace is not None:
                    multi = len(self.decoders) > 1
                    self._tr("convt_bwd", up=upo, x=d_in, dcat=dcat, du=du.clone() if multi else du, dw=dwu, db=db,
                             dx=g.clone() if multi else g)
            g5 = g if g5 is None else ops.nhwc_add(g5, g)
        g = g5
        # ---- encoder, level 4 -> 0
        g_pool = None
        for l in (4, 3, 2, 1, 0):
            r1, r2, _, idx = saved.enc[l]
            c1, c2 = self.enc[l]
            if l == 4:
                g1, pre = bn_conv_bwd(c2, r2, g, None, None, hs[l], wsz[l], True, fuse_next=r1)
            else:
                g1, pre = bn_conv_bwd(c2, r2, skip_grads[l], g_pool, idx, hs[l], wsz[l], True, fuse_next=r1)
            g_pool = bn_conv_bwd(c1, r1, g1, None, None, hs[l], wsz[l], need_dx=(l > 0), pre=pre)
            if l > 0 and drop_ps[l - 1] > 0:  # gradient w.r.t. the pooled tensor of level l - 1, through its mask
                self._dropout(g_pool, l - 1, seed, drop_ps[l - 1], backward=True)
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)  # join
        if flat is not None:
            flat.finish()
        return grads


class _GraphedStep:
    """Forward (and backward) of one (input shape, mode) captured as CUDA graphs that share a private memory pool.

    The ~270 launches of a step are mostly short; replaying them as a graph removes the host launch path and the
    inter-kernel gaps. Everything a graph touches is static: the input is copied into `x`, activations / saved
    tensors / gradients live in the pool, the bf16 weight operands are refreshed in place OUTSIDE the graph
    (UNetEngine.refresh_operands) before each replay. One forward may be in flight per shape: a second forward
    overwrites the saved activations of the first, so its backward is refused."""

    def __init__(self, engine: "UNetEngine", x: torch.Tensor, training: bool, save: bool):
        self.engine, self.training, self.save = engine, training, save
        self.x = torch.empty_like(x)
        self.pool = torch.cuda.graph_pool_handle()
        # data parallel: the NCCL watchdog thread queries CUDA events while this thread captures, which the default
        # "global" capture mode would reject
        dp = DataParallelContext.current() if training else None
        self.capture_mode = "thread_local" if dp is not None else "global"
        if dp is not None:
            dp._graph_owners.add(engine)  # DataParallelContext.disable() drops these graphs before NCCL teardown
        self.fwd = self.bwd = None
        self.logits = self.saved = self.dlogits = self.grads = None
        self.epoch = 0
        self.bwd_done_epoch = 0

    def forward(self, x):
        self.engine.refresh_operands()
        self.x.copy_(x)
        if self.fwd is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self.pool, capture_error_mode=self.capture_mode):
                self.logits, self.saved = self.engine.forward(self.x, self.training, self.save)
            self.fwd = g
        self.fwd.replay()
        self.epoch += 1
        # the caller may keep its logits across the next replay (one tensor, or one per decoder)
        return tuple(l.clone() for l in self.logits) if isinstance(self.logits, tuple) else self.logits.clone()

    def backward(self, epoch, dlogits):
        if epoch != self.epoch:
            raise RuntimeError("CUDA-graph mode keeps ONE set of saved activations per input shape: backward of an "
                               "older forward was requested after a newer forward ran (disable graphs with "
                               "net.enable_cuda_graphs(False) for this pattern)")
        if self.bwd_done_epoch == epoch:
            raise RuntimeError("UNet backward called twice: activations are consumed in place")
        multi = isinstance(self.logits, tuple)
        if self.dlogits is None:
            self.dlogits = tuple(torch.empty_like(l) for l in self.logits) if multi else torch.empty_like(self.logits)
        if multi:
            for dst, src in zip(self.dlogits, dlogits):
                dst.zero_() if src is None else dst.copy_(src)
        else:
            self.dlogits.copy_(dlogits)
        if self.bwd is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self.pool, capture_error_mode=self.capture_mode):
                self.grads = self.engine.backward(self.saved, self.dlogits)
            self.bwd = g
        self.bwd.replay()
        self.bwd_done_epoch = epoch
        # the static gradient tensors stay referenced here, so autograd copies them into .grad instead of adopting them
        return self.grads


class _UNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, x, *params):
        training = engine.net.training
        ctx.device = x.device
        with _device_guard(x):  # launches go to the current device's stream: make the input's device current
            step = engine.graphed_step(x, training, save=True)
            if step is not None:
                logits = step.forward(x)
                ctx.step, ctx.epoch, ctx.saved = step, step.epoch, None
            else:
                logits, saved = engine.forward(x, training=training, save=True)
                ctx.step, ctx.saved = None, saved
        ctx.engine, ctx.params = engine, params
        return logits  # one tensor, or one per decoder

    @staticmethod
    def backward(ctx, *dlogits):
        with torch.cuda.device(ctx.device):  # a CPU input was rejected in forward
            if ctx.step is not None:
                grads = ctx.step.backward(ctx.epoch, dlogits if len(dlogits) > 1 else dlogits[0].contiguous().float())
                if ctx.engine.net._share_grads:
                    # hand the graph's static gradient tensors to .grad directly: autograd would copy every one of them
                    # (they stay referenced by the graph, so it cannot adopt them) - 124 MB of device copies per step
                    for p in ctx.params:
                        g = grads.get(p)
                        if g is None or not p.requires_grad:
                            continue
                        if p.grad is None:
                            p.grad = g
                        elif p.grad.data_ptr() != g.data_ptr():
                            p.grad.add_(g)   # a gradient from elsewhere is already there: accumulate like autograd
                    return (None, None) + tuple(None for _ in ctx.params)
                return (None, None) + tuple(grads.get(p) for p in ctx.params)
            if ctx.saved is None:
                raise RuntimeError("UNet backward called twice: activations are consumed in place")
            grads = ctx.engine.backward(ctx.saved, dlogits if len(dlogits) > 1 else dlogits[0])
            ctx.saved = None
            return (None, None) + tuple(grads.get(p) for p in ctx.params)


# ------------------------------------------------------------------------------------------------ public module
class UNet(nn.Module):
    """Same constructor and forward(x) as the reference (Model.py:96, :142)."""

    def __init__(self, n_channels, n_classes, initial_feature_map=64, usa_cuda=True, dropout=False, dropout_p=0.5):
        super().__init__()
        self.usa_cuda = usa_cuda
        self.n_channels = {-2: 3, -1: 1}.get(n_channels, n_channels)  # Model.py:99-104
        self.n_classes = n_classes
        self.initial_feature_map = initial_feature_map
        self.dropout = dropout
        self.dropout_p = dropout_p
        f = initial_feature_map
        # creation + init order fixes the RNG stream (Model.py:107-140): build a block, then re-init its Conv2d's
        blocks = [("inc", lambda: DoubleConv(self.n_channels, f))]
        for i in range(4):
            blocks.append((f"down{i + 1}", lambda i=i: Down(f << i, f << (i + 1), dropout, dropout_p)))
        for i in range(4):
            blocks.append((f"up{i + 1}", lambda i=i: Up(f << (4 - i), f << (3 - i), dropout, dropout_p)))
        blocks.append(("outc", lambda: OutConv(f, n_classes)))
        for name, make in blocks:
            mod = make()
            setattr(self, name, mod)
            mod.apply(self.weights_init)
        self._engine = None
        self._generic = None
        self._check_fp32 = os.environ.get("B200UNET_CHECK_FP32", "0") not in ("", "0")
        self._cuda_graphs = os.environ.get("B200UNET_CUDA_GRAPHS", "0") not in ("", "0")
        self._share_grads = False

    def _topology(self):
        """(inc, [down1..4], [([up1..4], outc)]) - what the engines execute."""
        return self.inc, [self.down1, self.down2, self.down3, self.down4], [
            ([self.up1, self.up2, self.up3, self.up4], self.outc)]

    def enable_cuda_graphs(self, flag: bool = True, share_grads: bool = False):
        """Replay forward/backward as captured CUDA graphs (per input shape; first call of a shape runs eagerly).
        Off by default: outputs are copies of static buffers and one forward per shape may be in flight.
        share_grads=True additionally makes `p.grad` the graph's own static gradient tensors instead of copies of them
        (saves 124 MB of device copies per step): they are valid until the next backward of the same input shape, so clear
        them with `zero_grad(set_to_none=True)` (torch's default) every step and do not accumulate gradients over several
        backward calls in this mode."""
        self._cuda_graphs = bool(flag)
        self._share_grads = bool(flag) and bool(share_grads)
        if self._engine is not None:
            self._engine._graphs.clear()
        return self

    def weights_init(self, m):
        if isinstance(m, nn.Conv2d):  # Model.py:167-169: ConvTranspose2d keeps torch's default init
            nn.init.kaiming_normal_(m.weight)

    def refresh_operands(self, force: bool = True):
        """Re-derive the bf16 GEMM operands from the fp32 parameters. Done automatically when a parameter's autograd version
        changes (optimizer steps, load_state_dict, in-place ops); writes that bypass the version counter - `p.data.copy_()`,
        `dist.broadcast(p.data)` after the first forward - need this call (force=True re-derives all of them)."""
        if self._engine is not None:
            if force:
                for c1, c2 in self._engine.enc + self._engine.dec:
                    c1._ver = c2._ver = None
                for u in self._engine.ups:
                    u._ver = None
            self._engine.refresh_operands()
        return self

    def set_check_mode(self, flag: bool = True):
        """fp32 check mode: run every operator with the generic fp32 CUDA-core kernels (reference precision)."""
        self._check_fp32 = bool(flag)
        return self

    def _fast_supported(self) -> bool:
        """Can the tensor-core engine run this architecture at all (input size is checked per call)?"""
        # widths: the BN / head kernels take power-of-two channel counts in [64, 2048] -> base width 64 or 128
        return self.initial_feature_map in (64, 128) and self.n_channels <= 7 and 1 <= self.n_classes <= ops.HEAD_MAX_CLASSES

    def _get_engine(self) -> UNetEngine:
        """The tensor-core engine; raises if the architecture is outside its envelope."""
        if self._engine is None:
            if not self._fast_supported():
                raise ValueError("tensor-core engine needs initial_feature_map in (64, 128), n_channels <= 7 and "
                                 "n_classes <= 256 (UNet_attention: width 64 and dropout=False); other variants run on the "
                                 "generic fp32 engine")
            object.__setattr__(self, "_engine", UNetEngine(self))
        return self._engine

    def _engine_for(self, x):
        """Tensor-core engine when the architecture and this input fit it, otherwise (or in check mode) the generic
        fp32 engine. Both are CUDA kernels of this library; there is no PyTorch / CPU fallback."""
        fast = (not self._check_fp32 and self._fast_supported() and x.dim() == 4 and x.shape[2] % 16 == 0
                and x.shape[3] % 16 == 0)
        if fast:
            return self._get_engine()
        if self._generic is None:
            from .generic import GenericEngine

            object.__setattr__(self, "_generic", GenericEngine(self))
        return self._generic

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        object.__setattr__(self, "_engine", None)  # parameters may have been re-created (.to / .half / ...)
        object.__setattr__(self, "_generic", None)
        return out

    def forward(self, x):
        eng = self._engine_for(x)
        params = eng.params_in_backward_order()
        if x.is_cuda and params[0].device != x.device:
            raise RuntimeError(f"UNet parameters live on {params[0].device} but the input is on {x.device}")
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return _UNetFn.apply(eng, x, *params)
        with _device_guard(x):
            step = eng.graphed_step(x, self.training, save=False)
            if step is not None:
                return step.forward(x)
            logits, _ = eng.forward(x, training=self.training, save=False)
        return logits

    # ---- fused inference epilogues (SURVEY.md 8f rank 4): the logits never reach HBM
    def _fused_head(self, x, head, head_arg=0.0):
        eng = self._engine_for(x)
        if not isinstance(eng, UNetEngine):
            raise ValueError("fused inference heads run on the tensor-core engine (H, W multiples of 16, default widths); "
                             "use predict_mask(net(x)) for other variants")
        with torch.no_grad(), _device_guard(x):
            out, _ = eng.forward(x, training=self.training, save=False, head=head, head_arg=head_arg)
        return out

    def predict(self, x):
        """np.uint8(argmax(softmax(self(x), 1), 1)) of test_mc3serousv5.py:879-887 as one fused epilogue -> uint8 [B,H,W]."""
        return self._fused_head(x, "mask")

    def predict_binary(self, x, threshold=0.5):
        """(torch.sigmoid(self(x))[:, 0] >= threshold) of test.py:393-399 as one fused epilogue -> {0,1} uint8 [B,H,W]."""
        return self._fused_head(x, "sigmoid", threshold)

    def predict_density(self, x, divisor=200.0):
        """(F.relu(self(x)) / divisor, per-map sums) of test_mc3serousv5.py:961-974 -> (fp32 [B,C,H,W], fp64 [B,C])."""
        return self._fused_head(x, "density", divisor)

    def use_checkpointing(self):
        raise NotImplementedError("activation checkpointing is not needed: bf16 activations fit in HBM3e")


class UNet_multitask(UNet):
    """Same constructor, state_dict keys (inc, down1-4, up{1-4}_decod{1,2}, outc_decod{1,2}), RNG consumption and
    forward(x) -> (logits_decod1, logits_decod2) as the reference's two-decoder network (Model.py:172-250): one encoder
    pass, two decoder passes over it with the same kernels; backward sums the two decoders' skip / bottleneck gradients.
    As in the reference, `dropout` is stored but no Dropout layer is built (Model.py:188-230 pass no dropout flag)."""

    def __init__(self, n_channels, n_classes, initial_feature_map=64, usa_cuda=True, dropout=False, dropout_p=0.5):
        nn.Module.__init__(self)
        self.usa_cuda = usa_cuda
        self.n_channels = {-2: 3, -1: 1}.get(n_channels, n_channels)  # Model.py:176-181
        self.n_classes = n_classes
        self.initial_feature_map = initial_feature_map
        self.dropout = dropout
        self.dropout_p = dropout_p
        f = initial_feature_map
        blocks = [("inc", lambda: DoubleConv(self.n_channels, f))]
        for i in range(4):
            blocks.append((f"down{i + 1}", lambda i=i: Down(f << i, f << (i + 1))))
        for d in (1, 2):
            for i in range(4):
                blocks.append((f"up{i + 1}_decod{d}", lambda i=i: Up(f << (4 - i), f << (3 - i))))
            blocks.append((f"outc_decod{d}", lambda: OutConv(f, n_classes)))
        for name, make in blocks:
            mod = make()
            setattr(self, name, mod)
            mod.apply(self.weights_init)
        self._engine = None
        self._generic = None
        self._check_fp32 = False
        self._cuda_graphs = False
        self._share_grads = False

    def _topology(self):
        return self.inc, [self.down1, self.down2, self.down3, self.down4], [
            ([getattr(self, f"up{i}_decod{d}") for i in (1, 2, 3, 4)], getattr(self, f"outc_decod{d}")) for d in (1, 2)]

    def _fast_supported(self) -> bool:
        return self.initial_feature_map in (64, 128) and self.n_channels <= 7 and 1 <= self.n_classes <= ops.HEAD_MAX_CLASSES

    def _engine_for(self, x):
        if x.dim() != 4 or x.shape[2] % 16 or x.shape[3] % 16 or not self._fast_supported():
            raise ValueError("UNet_multitask runs on the tensor-core engine only: H and W multiples of 16, "
                             "initial_feature_map in (64, 128), n_channels <= 7, n_classes <= 256")
        return self._get_engine()

    def set_check_mode(self, flag: bool = True):
        raise NotImplementedError("the fp32 check engine covers UNet and UNet_attention")

    def _fused_head(self, x, head, head_arg=0.0):
        raise NotImplementedError("fused inference heads cover UNet / UNet_attention; apply predict_mask / F.relu to the two outputs")


class Attention_block(_Holder):
    """Parameter container of the reference's attention gate (Model.py:257-296): W_q / W_x = 1x1 conv + bias + BatchNorm,
    up = ConvTranspose2d(C_q, C_q, 2, 2), psi = 1x1 conv to one channel + BatchNorm + Sigmoid. Same construction order (RNG
    consumption) and state_dict keys as the reference; executed by the engine (generic.py `_gate_fwd` / `_gate_bwd`)."""

    def __init__(self, C_q, C_x, C_hidden):
        super().__init__()
        self.W_q = nn.Sequential(nn.Conv2d(C_q, C_hidden, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(C_hidden))
        self.up = nn.ConvTranspose2d(C_q, C_q, kernel_size=2, stride=2)
        self.W_x = nn.Sequential(nn.Conv2d(C_x, C_hidden, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(C_hidden))
        self.psi = nn.Sequential(nn.Conv2d(C_hidden, 1, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(1),
                                 nn.Sigmoid())
        self.relu = nn.ReLU(inplace=True)


class UNet_attention(UNet):
    """Attention U-Net of the reference (Model.py:299-391): UNet whose skip connections pass through attention gates,
    `x_l_attention = attenion_l(q = decoder input, x = skip)` (the misspelt attribute names are the reference's and fix the
    state_dict keys). Same constructor, RNG consumption (the gates keep torch's default init: no `.apply(weights_init)`,
    Model.py:325-341), 210 state_dict keys and forward(x) -> logits.
    Default width (initial_feature_map = 64, no dropout): the tensor-core engine - the U-Net body as in UNet, the gates as
    tcgen05 GEMMs (`up` and W_q composed into one ConvTranspose2d C_q -> C_h, W_x as a 1x1 GEMM) plus the bandwidth-bound
    kernels of csrc/gate.cu. Other variants, and `set_check_mode(True)`: the generic fp32 CUDA engine (csrc/generic_f32.cu,
    reference precision). H and W must be divisible by 16 (the reference's gate adds maps whose sizes only match then)."""

    def __init__(self, n_channels, n_classes, initial_feature_map=64, usa_cuda=True, dropout=False, dropout_p=0.5):
        nn.Module.__init__(self)
        self.usa_cuda = usa_cuda
        self.n_channels = {-2: 3, -1: 1}.get(n_channels, n_channels)  # Model.py:303-308
        self.n_classes = n_classes   # (the reference forgets this attribute; kept for the engine)
        self.initial_feature_map = initial_feature_map
        self.dropout = dropout
        self.dropout_p = dropout_p
        f = initial_feature_map

        def add(name, mod, init):
            setattr(self, name, mod)
            if init:
                mod.apply(self.weights_init)

        add("inc", DoubleConv(n_channels, f), True)   # the reference passes the RAW n_channels here (Model.py:314)
        for i in range(4):
            add(f"down{i + 1}", Down(f << i, f << (i + 1), dropout, dropout_p), True)
        for lvl in (4, 3, 2, 1):                      # attenion4 .. attenion1, default init (Model.py:325-341)
            add(f"attenion{lvl}", Attention_block(C_q=f << lvl, C_x=f << (lvl - 1), C_hidden=(f << (lvl - 1)) // 2), False)
        for i in range(4):
            add(f"up{i + 1}", Up(f << (4 - i), f << (3 - i), dropout, dropout_p), True)
        add("outc", OutConv(f, n_classes), True)
        self._engine = None
        self._generic = None
        self._check_fp32 = os.environ.get("B200UNET_CHECK_FP32", "0") not in ("", "0")
        self._cuda_graphs = False
        self._share_grads = False

    def _attention_gates(self):
        """Gate of decoder block j = 0..3 (up1..up4)."""
        return [self.attenion4, self.attenion3, self.attenion2, self.attenion1]

    def _fast_supported(self) -> bool:
        # the gate kernels take hidden widths 32..256 (csrc/gate.cu): base width 64
        return self.initial_feature_map == 64 and self.n_channels <= 7 and 1 <= self.n_classes <= ops.HEAD_MAX_CLASSES and not self.dropout

    def _engine_for(self, x):
        if x.dim() == 4 and (x.shape[2] % 16 or x.shape[3] % 16):
            raise ValueError("UNet_attention needs H and W divisible by 16 (its gates add a 2x-upsampled map to the skip)")
        return super()._engine_for(x)

    def refresh_operands(self, force: bool = True):
        if self._engine is not None and force:
            for g in self._engine.gates or ():
                g._ver = None
        return super().refresh_operands(force)

def preprocess(img_org, input_size=None, device=None) -> torch.Tensor:
    """`preprocess(img_org, input_size)` of test_mc3serousv5.py:100-127 / the z-normalisation of DataLoader.py:661-671 on
    the GPU: uint8 image(s) as cv2.imread returns them ([H,W,C] BGR, [H,W] grey, or a batch [N,H,W,C]) -> fp32 [N,C,H,W],
    each image and channel z-normalised with its own mean / population std, channels reversed to RGB.
    Resizing (scipy `zoom`, order 3) stays with the caller: a size mismatch with `input_size` raises."""
    if not torch.is_tensor(img_org):
        img_org = torch.from_numpy(img_org)
    if img_org.dtype != torch.uint8:
        raise TypeError(f"preprocess expects uint8 pixels (cv2.imread), got {img_org.dtype}")
    if img_org.dim() not in (2, 3, 4):
        raise ValueError(f"preprocess expects [H,W], [H,W,C] or [N,H,W,C], got {tuple(img_org.shape)}")
    hw = tuple(img_org.shape[:2]) if img_org.dim() < 4 else tuple(img_org.shape[1:3])
    if input_size is not None and tuple(input_size) != hw:
        raise ValueError(f"image is {hw}, input_size {tuple(input_size)}: resize (scipy zoom) before preprocess")
    if not img_org.is_cuda:
        dev = torch.device(device if device is not None else "cuda")
        img_org = (img_org.pin_memory() if torch.cuda.is_available() else img_org).to(dev, non_blocking=True)
    return ops.znorm_to_chw(img_org, reverse_channels=True)


def preprocess_crop(img_org, crop_size, device=None) -> torch.Tensor:
    """`preprocessCrop` of test.py:91-126 (image part) on the GPU: pad H and W up to multiples of `crop_size` with 255
    (split p//2 before, the rest after), then z-normalise the padded image like `preprocess` -> fp32 [1,C,Hp,Wp]."""
    if not torch.is_tensor(img_org):
        img_org = torch.from_numpy(img_org)
    if img_org.dtype != torch.uint8 or img_org.dim() not in (2, 3):
        raise TypeError("preprocess_crop expects one uint8 image [H,W] or [H,W,C]")
    if not img_org.is_cuda:
        img_org = img_org.to(torch.device(device if device is not None else "cuda"))
    if img_org.dim() == 2:
        img_org = img_org[:, :, None]
    ph, pw = (-img_org.shape[0]) % crop_size, (-img_org.shape[1]) % crop_size
    if ph or pw:
        padded = torch.full((img_org.shape[0] + ph, img_org.shape[1] + pw, img_org.shape[2]), 255, dtype=torch.uint8,
                            device=img_org.device)
        padded[ph // 2: ph // 2 + img_org.shape[0], pw // 2: pw // 2 + img_org.shape[1]] = img_org
        img_org = padded
    return ops.znorm_to_chw(img_org, reverse_channels=True)


def predict_tiled(net, img_org, crop_size, head="sigmoid", threshold=0.5, max_batch=64) -> torch.Tensor:
    """`test_single_crop` (test.py:420-447): pad + z-normalise the image (preprocess_crop), run every crop_size x crop_size
    crop through the network in eval mode and stitch the per-crop masks -> uint8 [Hp,Wp]. The reference loops over the
    crops one forward at a time; here they form batches (eval-mode BatchNorm makes crops independent of each other) and the
    mask comes from the fused head: head="sigmoid" (channel 0 >= threshold, test.py:436-440) or "mask" (softmax/argmax)."""
    if crop_size % 16:
        raise ValueError("predict_tiled: crop_size must be a multiple of 16")
    if net.training:
        raise RuntimeError("predict_tiled is an inference path: call net.eval() first (test.py:430)")
    x = preprocess_crop(img_org, crop_size, device=next(net.parameters()).device)
    _, c, hp, wp = x.shape
    nh, nw = hp // crop_size, wp // crop_size
    tiles = (x.view(c, nh, crop_size, nw, crop_size).permute(1, 3, 0, 2, 4).reshape(nh * nw, c, crop_size, crop_size)
             .contiguous())
    outs = []
    for i in range(0, nh * nw, max_batch):
        t = tiles[i:i + max_batch]
        outs.append(net.predict_binary(t, threshold) if head == "sigmoid" else net.predict(t))
    m = torch.cat(outs, 0)
    return m.view(nh, nw, crop_size, crop_size).permute(0, 2, 1, 3).reshape(hp, wp).contiguous()


def predict_mask(logits: torch.Tensor) -> torch.Tensor:
    """softmax(dim=1) -> argmax(dim=1) of test_mc3serousv5.py:880-881, fused."""
    return ops.softmax_argmax(logits.contiguous().float())
