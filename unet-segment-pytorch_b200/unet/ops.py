"""Autograd glue: each fused block of the network is one ``torch.autograd.Function``
whose forward and backward are sequences of C-ABI kernel launches (``kernels.py``).

Tensors crossing these functions are *logical NCHW, channels_last, bf16* — i.e.
physically NHWC bf16, the layout every kernel reads — so chaining blocks never
copies or transposes.  Parameters stay fp32 in the reference's layout and their
gradients are returned as fp32 tensors of the same shape.
"""
from __future__ import annotations

import torch

from . import kernels as K
from . import syncbn

BF16 = torch.bfloat16


# ---------------------------------------------------------------------------------------------
# Direct gradient accumulation.  When a sink is installed (BatchShardedTrainer does it for the
# duration of its step), a backward pass accumulates each parameter gradient straight into the
# existing ``param.grad`` buffer from inside the producing kernel and returns ``None`` for it, so
# autograd launches no per-parameter ``grad += g`` kernel (92 of them per step) and no zero fill for
# temporaries.  ``sink(param)`` is called once the gradient has been enqueued — the replacement
# for a post-accumulate-grad hook.  Without a sink gradients flow through autograd as usual.
GRAD_SINK = None


def _grad_targets(*params):
    """The .grad buffers of ``params`` if every one can be accumulated into in place, else None."""
    if GRAD_SINK is None:
        return None
    out = []
    for p in params:
        if not getattr(p, "is_leaf", False):      # a padded / derived view of a parameter: through autograd
            return None
        g = getattr(p, "grad", None)
        if (g is None or g.dtype != torch.float32 or not g.is_contiguous()
                or g.numel() != p.numel() or g.device != p.device):
            return None
        out.append(g)
    return out


def _grads_done(*params):
    for p in params:
        GRAD_SINK(p)


def _reduce_into(param, partial, cout, cin, taps, target):
    """Fold split-K partials into ``target`` (+=): right away, or — if the sink batches them —
    handed over to be folded together with the other layers of the same gradient bucket."""
    defer = getattr(GRAD_SINK, "defer_reduce", None)
    if defer is not None:
        defer(param, (partial, cout, cin, taps, target))
    else:
        K.wgrad_reduce(partial, cout, cin, taps, target, accumulate=True)
        GRAD_SINK(param)


# Weight gradients off the critical path.  In backward a layer's data gradient feeds the next layer's BatchNorm
# backward, its weight gradient feeds nothing until the bucket fold — yet both are tensor-pipe kernels that were
# queued one behind the other in front of the bandwidth-bound BatchNorm passes.  With a side stream installed
# (BatchShardedTrainer does it together with the sink) the weight-gradient GEMM of layer L runs next to the
# BatchNorm-backward reduce / apply passes of layer L-1: the data gradient is queued first on the main stream,
# the weight gradient forks behind the same dy, and the main stream joins again before the next fork and before
# any fold of the partial tiles.  Inside a CUDA-graph capture the fork and join become graph edges.
# Tensors the side stream reads (dy and the saved activations) are kept referenced until the join, because the
# caching allocator reuses a freed block in main-stream order only.
class SideStream:
    def __init__(self, device):
        self.stream = torch.cuda.Stream(device=device)
        self._keep = None

    def run(self, fn, *keep):
        main = torch.cuda.current_stream(self.stream.device)
        self.join()
        self.stream.wait_stream(main)
        with torch.cuda.stream(self.stream):
            out = fn()
        self._keep = (keep, out)
        return out

    def join(self):
        if self._keep is not None:
            torch.cuda.current_stream(self.stream.device).wait_stream(self.stream)
            self._keep = None


WGRAD_SIDE = None


def wgrad_join():
    """Main stream waits for the weight gradients still running on the side stream (before their partial tiles
    are folded, and at the end of backward)."""
    if WGRAD_SIDE is not None:
        WGRAD_SIDE.join()


# Weight packs prepared for the current step by a ``kernels.WeightPacker`` (installed by
# BatchShardedTrainer after it has rebuilt them in one launch); None -> pack per call.
PACKS = None


def _packs(weight, want_dgrad):
    if PACKS is not None:
        hit = PACKS.get(weight)
        if hit is not None:
            return hit
    return K.pack_conv_weight(weight, True, want_dgrad)


def to_nhwc(x: torch.Tensor) -> torch.Tensor:
    """Logical NCHW tensor -> dense NHWC bf16 view (no copy if already channels_last bf16)."""
    if not x.is_cuda:
        raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback); "
                           "move the model and its inputs to a B200 with .to('cuda')")
    if x.dtype != BF16:
        x = x.to(BF16)
    return x.permute(0, 2, 3, 1).contiguous()


def from_nhwc(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 3, 1, 2)


def _bn_train_coeffs(partials, count, bn):
    """Batch statistics -> (scale, shift, mean, invstd); running buffers updated like
    nn.BatchNorm2d in train mode (layers.py:33).  An nn.SyncBatchNorm that synchronises sums
    the statistics and pixel counts of every rank of its group first (unet.syncbn)."""
    if bn.momentum is None:
        raise NotImplementedError("BatchNorm momentum=None (cumulative average) is not supported")
    group = syncbn.group_of(bn)
    if group is not None:
        partials, count = syncbn.exchange(partials, count, group)
    track = bn.track_running_stats and bn.running_mean is not None
    return K.bn_finalize(partials, count, bn.weight, bn.bias,
                         bn.running_mean if track else None, bn.running_var if track else None,
                         bn.num_batches_tracked if track else None, float(bn.momentum), float(bn.eps))


def _bn_frozen_coeffs(bn):
    """Eval mode: normalise with the running statistics."""
    scale, shift = K.bn_eval_coeffs(bn.weight, bn.bias, bn.running_mean, bn.running_var, float(bn.eps))
    invstd = torch.rsqrt(bn.running_var + bn.eps)
    return scale, shift, bn.running_mean, invstd


def _use_batch_stats(bn) -> bool:
    return bn.training or bn.running_mean is None


class ConvBnRelu(torch.autograd.Function):
    """conv3x3(pad 1, no bias) over one or two (virtually concatenated) inputs -> BatchNorm ->
    ReLU, optionally also returning the 2x2 max-pooled activation (DoubleConv / Down / the
    concat in Up, layers.py:31-38, :56, :105)."""

    @staticmethod
    def forward(ctx, x0, x1, weight, gamma, beta, bn, pool):
        a0 = to_nhwc(x0)
        a1 = to_nhwc(x1) if x1 is not None else None
        n, h, w, _ = a0.shape
        taps = weight.shape[2] * weight.shape[3]
        need_grad = any(ctx.needs_input_grad)
        need_dx = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        wf, wd = _packs(weight, need_dx)
        batch = _use_batch_stats(bn)
        if not batch and not need_grad:
            # inference: BatchNorm folded into the conv epilogue, ReLU fused
            scale, shift = K.bn_eval_coeffs(gamma, beta, bn.running_mean, bn.running_var, float(bn.eps))
            a = K.conv_fwd(a0, wf, taps, x1=a1, scale=scale, shift=shift, relu=True)
            p = K.bn_act(a, None, None, relu=False, pool=True, write_act=False)[1] if pool else None
            return from_nhwc(a), (from_nhwc(p) if pool else None)
        if batch:
            y, st = K.conv_fwd(a0, wf, taps, x1=a1, stats=True)
            scale, shift, mean, invstd = _bn_train_coeffs(st, n * h * w, bn)
        else:
            y = K.conv_fwd(a0, wf, taps, x1=a1)
            scale, shift, mean, invstd = _bn_frozen_coeffs(bn)
        pidx = None
        if pool:
            a, p, pidx = K.bn_act(y, scale, shift, relu=True, pool=True, want_idx=True)
        else:
            a, p = K.bn_act(y, scale, shift, relu=True, pool=False)
        ctx.save_for_backward(a0, a1, y, scale, shift, mean, invstd, gamma, wd, pidx)
        ctx.meta = (weight.shape, batch, syncbn.group_of(bn) if batch else None)
        ctx.params = (weight, gamma, beta)
        return from_nhwc(a), (from_nhwc(p) if pool else None)

    @staticmethod
    def backward(ctx, dA, dP):
        a0, a1, y, scale, shift, mean, invstd, gamma, wd, pidx = ctx.saved_tensors
        wshape, batch, group = ctx.meta
        cout, cin, kh, kw = wshape
        taps = kh * kw
        dA_n = to_nhwc(dA) if dA is not None else None
        dP_n = to_nhwc(dP) if dP is not None else None
        p_w, p_gamma, p_beta = ctx.params
        bn_t = _grad_targets(p_gamma, p_beta) if ctx.needs_input_grad[3] and ctx.needs_input_grad[4] else None
        dy, dgamma, dbeta = _bn_backward(dA_n, dP_n, pidx, y, scale, shift, mean, invstd, gamma, batch,
                                         targets=bn_t, group=group)
        if bn_t is not None:
            _grads_done(p_gamma, p_beta)
        # data gradient first: it is what the next layer's backward waits for
        d0 = d1 = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            n, h, w, _ = a0.shape
            c0 = a0.shape[3]
            d0 = K.empty_nhwc(n, h, w, c0, dy.device)
            d1 = K.empty_nhwc(n, h, w, a1.shape[3], dy.device) if a1 is not None else None
            K.conv_fwd(dy, wd, taps, out=d0, out1=d1, split=c0)
            d0 = from_nhwc(d0)
            d1 = from_nhwc(d1) if d1 is not None else None
        gw = None
        if ctx.needs_input_grad[2]:
            w_t = _grad_targets(p_w)
            if w_t is not None and WGRAD_SIDE is not None and getattr(GRAD_SINK, "defer_reduce", None) is not None:
                part = WGRAD_SIDE.run(lambda: K.conv_wgrad(a0, dy, taps, x1=a1), a0, a1, dy)
            else:
                part = K.conv_wgrad(a0, dy, taps, x1=a1)
            if w_t is not None:
                _reduce_into(p_w, part, cout, cin, taps, w_t[0])
            else:
                gw = torch.empty(wshape, device=dy.device, dtype=torch.float32)
                K.wgrad_reduce(part, cout, cin, taps, gw)
        return d0, d1, gw, dgamma, dbeta, None, None


def _bn_backward(dA, dP, pidx, y, scale, shift, mean, invstd, gamma, batch, relu=True, targets=None, group=None):
    dg, db = targets if targets is not None else (None, None)
    return K.bn_backward(dA, dP, pidx, y, scale, shift, mean, invstd, gamma, relu=relu, frozen=not batch,
                         dgamma=dg, dbeta=db, exchange=syncbn.exchanger(group))


class ConvInBnRelu(torch.autograd.Function):
    """First stage: conv3x3 on the fp32 NCHW network input (Cin = n_channels) -> BN -> ReLU."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, bn):
        if not x.is_cuda:
            raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback)")
        x_dtype = x.dtype
        x = x.contiguous().float()
        n, _, h, w = x.shape
        batch = _use_batch_stats(bn)
        y, st = K.conv_in_fwd(x, weight, stats=batch)
        if batch:
            scale, shift, mean, invstd = _bn_train_coeffs(st, n * h * w, bn)
        else:
            scale, shift, mean, invstd = _bn_frozen_coeffs(bn)
        a, _ = K.bn_act(y, scale, shift, relu=True, pool=False)
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(x, y, scale, shift, mean, invstd, gamma,
                                  weight if ctx.needs_input_grad[0] else None)
            ctx.meta = (weight.shape, batch, x_dtype, syncbn.group_of(bn) if batch else None)
            ctx.params = (weight, gamma, beta)
        return from_nhwc(a)

    @staticmethod
    def backward(ctx, dA):
        x, y, scale, shift, mean, invstd, gamma, weight = ctx.saved_tensors
        wshape, batch, x_dtype, group = ctx.meta
        p_w, p_gamma, p_beta = ctx.params
        bn_t = _grad_targets(p_gamma, p_beta) if ctx.needs_input_grad[2] and ctx.needs_input_grad[3] else None
        dy, dgamma, dbeta = _bn_backward(to_nhwc(dA), None, None, y, scale, shift, mean, invstd, gamma, batch,
                                         targets=bn_t, group=group)
        if bn_t is not None:
            _grads_done(p_gamma, p_beta)
        dx = K.conv_in_dgrad(dy, weight.contiguous(), wshape[1]).to(x_dtype) if ctx.needs_input_grad[0] else None
        gw = None
        if ctx.needs_input_grad[1]:
            w_t = _grad_targets(p_w)
            if w_t is not None:
                K.conv_in_wgrad(x, dy, wshape[0], grad=w_t[0])
                _grads_done(p_w)
            else:
                gw = K.conv_in_wgrad(x, dy, wshape[0])
        return dx, gw, dgamma, dbeta, None


class Upsample2x(torch.autograd.Function):
    """nn.Upsample(2x, bilinear, align_corners=True) + F.pad to the skip size (layers.py:78,
    :98-102)."""

    @staticmethod
    def forward(ctx, x, out_h, out_w):
        a = to_nhwc(x)
        n, h, w, c = a.shape
        ctx.geom = (h, w, 2 * h, 2 * w)
        return from_nhwc(K.upsample(a, 2 * h, 2 * w, out_h, out_w))

    @staticmethod
    def backward(ctx, dout):
        h, w, hu, wu = ctx.geom
        return from_nhwc(K.upsample_bwd(to_nhwc(dout), h, w, hu, wu)), None, None


class ResizeLogits(torch.autograd.Function):
    """F.interpolate(logits, size, mode='bilinear', align_corners=True) of the deep-supervision heads
    (unet/models/unet.py:206-208): fp32 NCHW in and out."""

    @staticmethod
    def forward(ctx, x, out_h, out_w):
        x = x.contiguous()
        ctx.geom = (x.shape[2], x.shape[3])
        return K.resize_planes(x, out_h, out_w)

    @staticmethod
    def backward(ctx, dout):
        h, w = ctx.geom
        return K.resize_planes_bwd(dout.contiguous(), h, w), None, None


def resize_logits(x, size):
    if not x.is_cuda:
        raise RuntimeError("unet-b200 ops need CUDA tensors: there is no CPU fallback")
    return ResizeLogits.apply(x.float(), int(size[0]), int(size[1]))


def gate_groups(bn_g, bn_x, bn_p):
    """The groups the gate's BatchNorms synchronise over: (W_g and W_x together, psi).  The backward folds the
    statistics of W_g and W_x in one table, so the two must agree."""
    group_g, group_x = syncbn.group_of(bn_g), syncbn.group_of(bn_x)
    if group_g is not group_x:
        raise NotImplementedError("AttentionGate: W_g and W_x BatchNorms must both synchronise over the same "
                                  "process group or both not (convert them together with convert_sync_batchnorm)")
    return group_x, syncbn.group_of(bn_p)


class AttentionGateFn(torch.autograd.Function):
    """AttentionGate.forward (layers.py:171-192) as two tensor-core 1x1 projections plus three
    bandwidth-bound passes; see csrc/gate.cu."""

    @staticmethod
    def forward(ctx, g, x, w_g, w_x, w_psi, gam_g, bet_g, gam_x, bet_x, gam_p, bet_p, bn_g, bn_x, bn_p):
        gn, xn = to_nhwc(g), to_nhwc(x)
        n, h, w, cx = xn.shape
        count = n * h * w
        need_grad = any(ctx.needs_input_grad)
        wgf, wgd = _packs(w_g, need_grad)
        wxf, wxd = _packs(w_x, need_grad)
        wpsi = w_psi.reshape(-1)
        batch = _use_batch_stats(bn_x)
        q = K.conv_fwd(gn, wgf, 1)
        if batch:
            xp, st_x = K.conv_fwd(xn, wxf, 1, stats=True)
            sg, hg, mg, ig = _bn_train_coeffs(K.gate_upstats(q, h, w), count, bn_g)
            sx, hx, mx, ix = _bn_train_coeffs(st_x, count, bn_x)
        else:
            xp = K.conv_fwd(xn, wxf, 1)
            sg, hg, mg, ig = _bn_frozen_coeffs(bn_g)
            sx, hx, mx, ix = _bn_frozen_coeffs(bn_x)
        if not batch and not need_grad and cx == 2 * wpsi.numel():
            # inference: psi, sigmoid and the gating in one pass (csrc/gate.cu: gate_fused_eval_kernel)
            sp, hp, _, _ = _bn_frozen_coeffs(bn_p)
            return from_nhwc(K.gate_fused_eval(q, xp, xn, sg, hg, sx, hx, wpsi, sp, hp))
        psi, st_p = K.gate_psi(q, xp, sg, hg, sx, hx, wpsi, stats=batch)
        if batch:
            sp, hp, mp, ip = _bn_train_coeffs(st_p, count, bn_p)
        else:
            sp, hp, mp, ip = _bn_frozen_coeffs(bn_p)
        out, a = K.gate_apply(psi, sp, hp, xn, save_a=need_grad)
        if need_grad:
            ctx.save_for_backward(gn, xn, q, xp, psi, a, sg, hg, mg, ig, sx, hx, mx, ix, mp, ip, wgd, wxd,
                                  wpsi, gam_g, gam_x, gam_p)
            ctx.meta = (w_g.shape, w_x.shape, w_psi.shape, batch) + (gate_groups(bn_g, bn_x, bn_p) if batch else (None, None))
            ctx.params = (w_g, w_x, w_psi, gam_g, bet_g, gam_x, bet_x, gam_p, bet_p)
        return from_nhwc(out)

    @staticmethod
    def backward(ctx, dout):
        (gn, xn, q, xp, psi, a, sg, hg, mg, ig, sx, hx, mx, ix, mp, ip, wgd, wxd, wpsi, gam_g, gam_x,
         gam_p) = ctx.saved_tensors
        sh_g, sh_x, sh_p, batch, group_xg, group_p = ctx.meta
        n, h, w, cx = xn.shape
        _, hin, win, cg = gn.shape
        ci = q.shape[3]
        count = n * h * w
        d = to_nhwc(dout)
        p_wg, p_wx, p_wpsi, p_gg, p_bg, p_gx, p_bx, p_gp, p_bp = ctx.params
        direct = _grad_targets(*ctx.params) if all(ctx.needs_input_grad[2:11]) else None
        dx, dpsin, part = K.gate_bwd_a(d, xn, a, psi)
        if direct is not None:
            t_wg, t_wx, t_wpsi, t_gg, t_bg, t_gx, t_bx, t_gp, t_bp = direct
            _, _, coef_p = K.bn_bwd_finalize(part, count, gam_p, mp, ip, frozen=not batch, dgamma=t_gp, dbeta=t_bp)
        else:
            dgam_p, dbet_p, coef_p = K.bn_bwd_finalize(part, count, gam_p, mp, ip, frozen=not batch)
        if group_p is not None:
            coef_p = K.synced_coef(part, count, syncbn.exchanger(group_p), gam_p, mp, ip)
        ds, part2 = K.gate_bwd_s(dpsin, psi, coef_p, q, xp, sg, hg, sx, hx, wpsi)
        grads, coef = K.gate_bwd_finalize(part2, count, gam_x, mx, ix, gam_g, mg, ig, frozen=not batch,
                                          targets=[t_gx, t_bx, t_gg, t_bg, t_wpsi] if direct is not None else None,
                                          exchange=syncbn.exchanger(group_xg))
        dxp, dgup = K.gate_bwd_xg(ds, xp, q, coef)
        dq = K.upsample_bwd(dgup, hin, win, h, w)
        if direct is not None:
            _reduce_into(p_wx, K.conv_wgrad(xn, dxp, 1), ci, cx, 1, t_wx)
            _reduce_into(p_wg, K.conv_wgrad(gn, dq, 1), ci, cg, 1, t_wg)
        else:
            gw_x = torch.empty(sh_x, device=d.device, dtype=torch.float32)
            K.wgrad_reduce(K.conv_wgrad(xn, dxp, 1), ci, cx, 1, gw_x)
            gw_g = torch.empty(sh_g, device=d.device, dtype=torch.float32)
            K.wgrad_reduce(K.conv_wgrad(gn, dq, 1), ci, cg, 1, gw_g)
        K.conv_fwd(dxp, wxd, 1, out=dx, accumulate=True)
        dg = K.conv_fwd(dq, wgd, 1)
        if direct is not None:
            _grads_done(*ctx.params[2:])   # the two projection weights were reported by _reduce_into
            return (from_nhwc(dg), from_nhwc(dx)) + (None,) * 12
        return (from_nhwc(dg), from_nhwc(dx), gw_g, gw_x, grads[4].reshape(sh_p), grads[2], grads[3],
                grads[0], grads[1], dgam_p, dbet_p, None, None, None)


class OutConvFn(torch.autograd.Function):
    """OutConv: 1x1 conv with bias to fp32 NCHW logits (layers.py:120-123)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        a = to_nhwc(x)
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(a, weight)
            ctx.params = (weight, bias)
        return K.outc_fwd(a, weight.reshape(weight.shape[0], -1), bias)

    @staticmethod
    def backward(ctx, dlogits):
        a, weight = ctx.saved_tensors
        direct = _grad_targets(*ctx.params) if ctx.needs_input_grad[1] and ctx.needs_input_grad[2] else None
        da, dw, db = K.outc_bwd(dlogits.contiguous().float(), a, weight.reshape(weight.shape[0], -1),
                                need_da=ctx.needs_input_grad[0],
                                dw=direct[0] if direct is not None else None,
                                db=direct[1] if direct is not None else None)
        da = from_nhwc(da) if da is not None else None
        if direct is not None:
            _grads_done(*ctx.params)
            return da, None, None
        return da, dw.reshape(weight.shape), db


class SegStats(torch.autograd.Function):
    """Per-(image, class) pixel sums every reference loss is built from; see csrc/loss.cu.
    Returns (count, ce_sum, intersection, prob_sum), each (N, C) fp32."""

    @staticmethod
    def forward(ctx, logits, targets):
        if not logits.is_cuda:
            raise RuntimeError("unet-b200 losses run on CUDA tensors only (no CPU fallback)")
        logits = logits.contiguous().float()
        st = K.seg_stats(logits, targets)
        ctx.save_for_backward(logits, targets)
        cnt, ce, inter, psum = st.unbind(dim=1)
        ctx.mark_non_differentiable(cnt)
        return cnt, ce, inter, psum

    @staticmethod
    def backward(ctx, _dcnt, dce, dinter, dpsum):
        logits, targets = ctx.saved_tensors
        z = lambda t: t if t is not None else torch.zeros(logits.shape[:2], device=logits.device)
        coef = torch.stack([z(dce), z(dinter), z(dpsum)], dim=1).float()
        return K.seg_stats_bwd(logits, targets, coef), None


class DiceBCEFn(torch.autograd.Function):
    """DiceBCELoss (loss.py:153-191) end to end: statistics pass, one head launch for the value and
    the gradient table, one backward pass over the pixels."""

    @staticmethod
    def forward(ctx, logits, targets, ce_weight, dice_weight, class_weight, ce_smooth, dice_smooth, ignore_bg):
        if not logits.is_cuda:
            raise RuntimeError("unet-b200 losses run on CUDA tensors only (no CPU fallback)")
        logits = logits.contiguous().float()
        loss, coef = K.dice_bce_head(K.seg_stats(logits, targets), ce_weight, dice_weight, class_weight,
                                     ce_smooth, dice_smooth, ignore_bg)
        ctx.save_for_backward(logits, targets, coef)
        return loss

    @staticmethod
    def backward(ctx, gout):
        logits, targets, coef = ctx.saved_tensors
        return (K.seg_stats_bwd(logits, targets, coef, gscale=gout.contiguous().float()),) + (None,) * 7


class MaxPool2x2(torch.autograd.Function):
    """Standalone nn.MaxPool2d(2) (layers.py:56) for `Down` used outside the fused network."""

    @staticmethod
    def forward(ctx, x):
        a = to_nhwc(x)
        _, p, pidx = K.bn_act(a, None, None, relu=False, pool=True, write_act=False, want_idx=True)
        ctx.save_for_backward(a, pidx)
        return from_nhwc(p)

    @staticmethod
    def backward(ctx, dp):
        a, pidx = ctx.saved_tensors
        return from_nhwc(K.maxpool_bwd(to_nhwc(dp), pidx, a))


class ConvTranspose2x2(torch.autograd.Function):
    """nn.ConvTranspose2d(C, C/2, kernel_size=2, stride=2) + F.pad to the skip size (layers.py:81, :98-102,
    :217-221).  Because kernel == stride the output pixels do not overlap: a 1x1 convolution to 4*Cout
    channels on the tensor cores (bias in its epilogue) followed by a pixel shuffle; shuffle, padding, its
    transpose and the bias gradient are kernels of csrc/shuffle.cu — nothing on this path runs in ATen."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_h, out_w):
        a = to_nhwc(x)
        n, h, w, cin = a.shape
        cout = weight.shape[1]
        wf, wd, scale4, shift4 = K.pack_convt_weight(weight.contiguous(), bias)
        t = K.conv_fwd(a, wf, 1, scale=scale4, shift=shift4)
        out = K.shuffle2x2(t, cout, out_h, out_w)
        ctx.save_for_backward(a, wd)
        ctx.geom = (h, w, cin, cout, bias is not None)
        ctx.params = (weight, bias)
        return from_nhwc(out)

    @staticmethod
    def backward(ctx, dout):
        a, wd = ctx.saved_tensors
        h, w, cin, cout, has_bias = ctx.geom
        p_w, p_b = ctx.params
        need_w = ctx.needs_input_grad[1]
        need_b = has_bias and ctx.needs_input_grad[2]
        direct = _grad_targets(*([p_w] + ([p_b] if has_bias else []))) if need_w and (need_b or not has_bias) else None
        d = to_nhwc(dout)
        dt, gb = K.shuffle2x2_bwd(d, h, w, dbias=direct[1] if (direct is not None and has_bias) else None, want_bias=need_b)
        gw = None
        if need_w:
            part = K.conv_wgrad(a, dt, 1)
            if direct is not None:
                K.convt_wgrad_reduce(part, cin, cout, direct[0], accumulate=True)
            else:
                gw = torch.empty((cin, cout, 2, 2), device=d.device, dtype=torch.float32)
                K.convt_wgrad_reduce(part, cin, cout, gw)
        dx = from_nhwc(K.conv_fwd(dt, wd, 1)) if ctx.needs_input_grad[0] else None
        if direct is not None:
            _grads_done(*([p_w] + ([p_b] if has_bias else [])))
            return dx, None, None, None, None
        return dx, gw, gb, None, None


def conv_transpose2x2(x, weight, bias, out_h, out_w):
    if not x.is_cuda:
        raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback)")
    return ConvTranspose2x2.apply(x, weight, bias, int(out_h), int(out_w))
