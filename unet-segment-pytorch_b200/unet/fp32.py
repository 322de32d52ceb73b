"""fp32 / TF32 mode: ``unet.set_precision("tf32")``.

The default precision of the B200 path is bf16 operands with fp32 accumulation.  This module is
the higher-accuracy path of BASELINE configs[0] ("AttentionUNet fp32 forward") and of north_star's
"in fp32/TF32 mode, logits and gradients must match within 1e-3 relative error": activations and
gradients stay fp32 (NHWC), forward and data-gradient convolutions run on the tensor cores as
``kind::tf32`` with operands rounded to TF32 where they are produced, and everything around them is
plain fp32 kernels.

* inference (``model.eval()`` under ``torch.no_grad()``): BatchNorm folded into the conv epilogue with the
  running statistics (csrc/fp32_eval.cu);
* training: batch statistics, the autograd functions at the end of this file (csrc/fp32_train.cu).  The
  weight gradient runs on the bf16 tensor-core kernels with each fp32 operand split into hi + lo bf16
  halves (three launches, 2^-16 relative: ``kind::tf32`` has no MN-major operand mode).  This is the
  accuracy mode — what the reference's own fp32 training computes — not the fast one: train in bf16 for speed.

Reference semantics: unet/models/layers.py:16-255.
"""
from __future__ import annotations

import torch

from . import _C
from ._C import ptr, stream
from . import kernels as K

F32 = torch.float32
PRECISION = "bf16"


def set_precision(mode: str) -> None:
    """"bf16" (default: training and inference) or "tf32" (fp32 activations, inference only)."""
    global PRECISION
    if mode not in ("bf16", "tf32", "fp32"):
        raise ValueError("precision must be 'bf16' or 'tf32'")
    PRECISION = "tf32" if mode in ("tf32", "fp32") else "bf16"


def active() -> bool:
    return PRECISION == "tf32"


def _training_path(module, *tensors) -> bool:
    """Batch statistics or gradients needed -> the autograd functions below; else the folded eval kernels."""
    return module.training or (torch.is_grad_enabled() and (
        any(t is not None and t.requires_grad for t in tensors) or any(p.requires_grad for p in module.parameters())))


def _check(module, *tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback)")


def nhwc(x: torch.Tensor) -> torch.Tensor:
    """Logical NCHW -> dense NHWC fp32 (no copy if already channels_last fp32)."""
    return x.float().permute(0, 2, 3, 1).contiguous()


def nchw(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 3, 1, 2)


def _bn_coeffs(bn):
    return K.bn_eval_coeffs(bn.weight, bn.bias, bn.running_mean, bn.running_var, float(bn.eps))


def _pack(w):
    cout, cin, kh, kw = w.shape
    out = torch.empty((cout, kh * kw, cin), device=w.device, dtype=F32)
    _C.call("ub2_f32_pack_weight", ptr(w.contiguous()), ptr(out), cout, cin, kh * kw, stream())
    return out


def _pack3(w, dgrad=False):
    """OIHW fp32 -> the 3xTF32 pack (rows, taps, 3*K) = per tap [w_hi | w_hi | w_lo]; ``dgrad``: rows = Cin,
    K = Cout, taps flipped (the data gradient is the same kernel)."""
    cout, cin, kh, kw = w.shape
    rows, k = (cin, cout) if dgrad else (cout, cin)
    out = torch.empty((rows, kh * kw, 3 * k), device=w.device, dtype=F32)
    _C.call("ub2_f32_pack_weight3", ptr(w.contiguous()), ptr(out), cout, cin, kh * kw, int(dgrad), stream())
    return out


def split_tf32(x0, x1=None):
    """(N,H,W,C0 [+C1]) fp32 -> (N,H,W,2*(C0+C1)) = [hi(x0) | hi(x1) | lo(x0) | lo(x1)], two TF32 numbers per value."""
    n, h, w, c0, ld0 = K._nhwc32(x0)
    c1, ld1 = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1 = K._nhwc32(x1)
    out = torch.empty((n, h, w, 2 * (c0 + c1)), device=x0.device, dtype=F32)
    _C.call("ub2_f32_split_tf32", ptr(x0), ld0, c0, ptr(x1), ld1, c1, ptr(out), _C.c_longlong(n * h * w), stream(),
            work=(0.0, K._nbytes(x0, x1, out)))
    return out


def conv3(x0, x1, weight, dgrad=False):
    """3xTF32 convolution (forward, or data gradient with ``dgrad``) of fp32 NHWC operands, fp32 result:
    one tensor-core launch over K = [a_hi | a_lo | a_hi] against [w_hi | w_hi | w_lo]."""
    cout, cin, kh, kw = weight.shape
    rows = cin if dgrad else cout
    cat = split_tf32(x0, x1)
    half = cat.shape[3] // 2
    return conv_packed(cat, cat[..., :half], _pack3(weight, dgrad), rows, kh * kw, exact=True)


def conv_packed(x0, x1, pack, cout, taps, scale=None, shift=None, relu=False, exact=False):
    """x0 / x1: NHWC fp32 (channel stride may exceed the channel count); ``pack``: (Cout, taps, Cin) fp32."""
    n, h, w, c0, ld0 = K._nhwc32(x0)
    c1, ld1 = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1 = K._nhwc32(x1)
    assert pack.numel() == cout * taps * (c0 + c1)
    out = torch.empty((n, h, w, cout), device=x0.device, dtype=F32)
    _C.call("ub2_conv_fwd_tf32", ptr(x0), ld0, c0, ptr(x1), ld1, c1, ptr(pack), ptr(out), cout, n, h, w,
            cout, taps, ptr(scale), ptr(shift), int(relu), int(exact), stream(),
            work=(2.0 * n * h * w * cout * taps * (c0 + c1), K._nbytes(x0, x1, pack, out)))
    return out


def conv(x0, x1, weight, scale=None, shift=None, relu=False):
    """x0 / x1: NHWC fp32; returns NHWC fp32 (TF32 tensor-core convolution)."""
    cout, cin, kh, kw = weight.shape
    return conv_packed(x0, x1, _pack(weight), cout, kh * kw, scale, shift, relu)


def double_conv(module, x0, x1=None, pool_out=False):
    """DoubleConv (layers.py:16-41) on logical-NCHW inputs; returns (activation, pooled or None)."""
    _check(module, x0, x1)
    seq = module.double_conv
    if _training_path(module, x0, x1):
        cin = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
        if cin % 16 != 0:
            if x1 is not None:
                raise RuntimeError("concatenated inputs need channel counts that are multiples of 16")
            a = ConvInBnReluF32.apply(x0, seq[0].weight, seq[1].weight, seq[1].bias, seq[1])
        else:
            a, _ = ConvBnReluF32.apply(x0, x1, seq[0].weight, seq[1].weight, seq[1].bias, seq[1], False)
        return ConvBnReluF32.apply(a, None, seq[3].weight, seq[4].weight, seq[4].bias, seq[4], bool(pool_out))
    cin = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
    s1, h1 = _bn_coeffs(seq[1])
    if cin % 16 != 0:
        if x1 is not None:
            raise RuntimeError("concatenated inputs need channel counts that are multiples of 16")
        x = x0.contiguous().float()
        n, _, h, w = x.shape
        cout = seq[0].weight.shape[0]
        a = torch.empty((n, h, w, cout), device=x.device, dtype=F32)
        _C.call("ub2_f32_conv_in", ptr(x), ptr(seq[0].weight.contiguous()), ptr(s1), ptr(h1), ptr(a), n, cin, h, w,
                cout, stream())
    else:
        a = conv(nhwc(x0), nhwc(x1) if x1 is not None else None, seq[0].weight, s1, h1, relu=True)
    s2, h2 = _bn_coeffs(seq[4])
    a = conv(a, None, seq[3].weight, s2, h2, relu=True)
    p = maxpool_nhwc(a) if pool_out else None
    return nchw(a), (nchw(p) if p is not None else None)


def maxpool_nhwc(a):
    n, h, w, c = a.shape
    out = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_maxpool", ptr(a), ptr(out), n, h, w, c, stream())
    return out


def maxpool(x):
    if torch.is_grad_enabled() and x.requires_grad:
        return MaxPoolF32.apply(x)
    return nchw(maxpool_nhwc(nhwc(x)))


def upsample(x, out_h, out_w):
    """nn.Upsample(2x, bilinear, align_corners=True) + F.pad to (out_h, out_w) (layers.py:78, :98-102)."""
    if torch.is_grad_enabled() and x.requires_grad:
        return UpsampleF32.apply(x, int(out_h), int(out_w))
    a = nhwc(x)
    n, h, w, c = a.shape
    out = torch.empty((n, out_h, out_w, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_upsample", ptr(a), ptr(out), n, h, w, 2 * h, 2 * w, out_h, out_w, c, stream())
    return nchw(out)


def conv_transpose2x2(module, x, out_h, out_w):
    """nn.ConvTranspose2d(C, C/2, kernel_size=2, stride=2) + F.pad to (out_h, out_w) (layers.py:81, :98-102,
    :217-221): a 1x1 tensor-core convolution to 4*Cout channels with the bias in its epilogue, then the pixel
    shuffle of csrc/shuffle.cu."""
    _check(module, x)
    if _training_path(module, x):
        return ConvTranspose2x2F32.apply(x, module.weight, module.bias, int(out_h), int(out_w))
    w1, scale4, shift4 = pack_convt_weight(module.weight, module.bias)
    t = conv_packed(nhwc(x), None, _pack(w1), w1.shape[0], 1, scale4, shift4)
    return nchw(shuffle2x2(t, module.weight.shape[1], out_h, out_w))


def gate(module, g, x):
    """AttentionGate.forward (layers.py:171-192)."""
    _check(module, g, x)
    if _training_path(module, g, x):
        bg, bx, bp = module.W_g[1], module.W_x[1], module.psi[1]
        return AttentionGateF32.apply(g, x, module.W_g[0].weight, module.W_x[0].weight, module.psi[0].weight,
                                      bg.weight, bg.bias, bx.weight, bx.bias, bp.weight, bp.bias, bg, bx, bp)
    gn, xn = nhwc(g), nhwc(x)
    n, h, w, cx = xn.shape
    _, hin, win, _ = gn.shape
    q = conv(gn, None, module.W_g[0].weight)      # W_g at low resolution: commutes with the resampling
    xp = conv(xn, None, module.W_x[0].weight)
    sg, hg = _bn_coeffs(module.W_g[1])
    sx, hx = _bn_coeffs(module.W_x[1])
    sp, hp = _bn_coeffs(module.psi[1])
    ci = q.shape[3]
    out = torch.empty_like(xn)
    _C.call("ub2_f32_gate", ptr(q), ptr(xp), ptr(xn), ptr(sg), ptr(hg), ptr(sx), ptr(hx),
            ptr(module.psi[0].weight.reshape(-1).contiguous()), ptr(sp), ptr(hp), ptr(out), n, hin, win, h, w, ci,
            cx, stream())
    return nchw(out)


def outc(module, x):
    """OutConv (layers.py:109-123): fp32 NCHW logits."""
    _check(module, x)
    if _training_path(module, x):
        return OutConvF32.apply(x, module.conv.weight, module.conv.bias)
    a = nhwc(x)
    n, h, w, c = a.shape
    wt = module.conv.weight
    k = wt.shape[0]
    logits = torch.empty((n, k, h, w), device=a.device, dtype=F32)
    _C.call("ub2_f32_outc", ptr(a), ptr(wt.reshape(k, -1).contiguous()), ptr(module.conv.bias), ptr(logits), n, h, w,
            c, k, stream())
    return logits


# =============================================================================================
# Training: autograd functions on fp32 NHWC tensors (csrc/fp32_train.cu)
# =============================================================================================
F64 = torch.float64
BF16 = torch.bfloat16


def nhwc_view(x: torch.Tensor) -> torch.Tensor:
    """Logical NCHW -> (N,H,W,C) fp32 whose rows are dense in the channel stride: no copy for channels_last
    tensors and for channel slices of one (the two halves of a concat's gradient)."""
    if not x.is_cuda:
        raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback)")
    t = x.float().permute(0, 2, 3, 1)
    n, h, w, c = t.shape
    ld = t.stride(2)
    ok = (t.stride(3) == 1 and ld >= c and ld % 4 == 0 and (h == 1 or t.stride(1) == w * ld)
          and (n == 1 or t.stride(0) == h * w * ld) and w > 1)
    return t if ok else t.contiguous()


def _dense(t):
    return t if t.is_contiguous() else t.contiguous()


def channel_stats(x):
    """(rows, 2, C) fp64 per-block sums / sums of squares over the pixels of an NHWC fp32 tensor."""
    n, h, w, c, ld = K._nhwc32(x)
    rows = K._rows("ub2_f32_channel_rows", _C.c_longlong(n * h * w), c)
    part = torch.empty((rows, 2, c), device=x.device, dtype=F64)
    _C.call("ub2_f32_channel_stats", ptr(x), ld, _C.c_longlong(n * h * w), c, ptr(part), rows, stream(),
            work=(0.0, K._nbytes(x)))
    return part


def scalar_stats(x):
    n = x.numel()
    rows = K._rows("ub2_f32_scalar_rows", _C.c_longlong(n))
    part = torch.empty((rows, 2, 1), device=x.device, dtype=F64)
    _C.call("ub2_f32_scalar_stats", ptr(x), _C.c_longlong(n), ptr(part), rows, stream(), work=(0.0, K._nbytes(x)))
    return part


def affine_act(y, scale, shift, relu=True):
    n, h, w, c = y.shape
    out = torch.empty_like(y)
    _C.call("ub2_f32_affine_act", ptr(y), ptr(scale), ptr(shift), ptr(out), _C.c_longlong(n * h * w), c, int(relu), stream(),
            work=(0.0, K._nbytes(y, out)))
    return out


def maxpool_idx(a):
    n, h, w, c = a.shape
    p = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=F32)
    idx = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=torch.uint8)
    _C.call("ub2_f32_maxpool_idx", ptr(a), ptr(p), ptr(idx), n, h, w, c, stream(), work=(0.0, K._nbytes(a, p, idx)))
    return p, idx


def act_backward(dA, dP, idx, y, scale, shift, mean, invstd, gamma, batch, relu=True):
    """BatchNorm (+ReLU, + max-pool routing) backward: (dy, dgamma, dbeta)."""
    n, h, w, c = y.shape
    ld_da = K._nhwc32(dA)[4] if dA is not None else 0
    dP = _dense(dP) if dP is not None else None
    rows = K._rows("ub2_f32_channel_rows", _C.c_longlong(n * h * w), c)
    part = torch.empty((rows, 2, c), device=y.device, dtype=F64)
    _C.call("ub2_f32_act_bwd_reduce", ptr(dA), ld_da, ptr(dP), ptr(idx), ptr(y), ptr(scale), ptr(shift), ptr(part), rows,
            n, h, w, c, int(relu), stream(), work=(0.0, K._nbytes(dA, dP, idx, y)))
    dgamma, dbeta, coef = K.bn_bwd_finalize(part, n * h * w, gamma, mean, invstd, frozen=not batch)
    dy = torch.empty_like(y)
    _C.call("ub2_f32_act_bwd_apply", ptr(dA), ld_da, ptr(dP), ptr(idx), ptr(y), ptr(scale), ptr(shift), ptr(coef), ptr(dy),
            n, h, w, c, int(relu), stream(), work=(0.0, K._nbytes(dA, dP, idx, y, dy)))
    return dy, dgamma, dbeta


def upsample_nhwc(a, out_h, out_w, hu=None, wu=None):
    """bilinear (h,w) -> (hu,wu) (default 2x), centred in a zero (out_h,out_w) canvas (F.pad of layers.py:98-102)."""
    n, h, w, c = a.shape
    hu, wu = (2 * h if hu is None else hu), (2 * w if wu is None else wu)
    out = torch.empty((n, out_h, out_w, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_upsample_fwd", ptr(a), ptr(out), n, h, w, hu, wu, out_h, out_w, c, stream(),
            work=(0.0, K._nbytes(a, out)))
    return out


def upsample_bwd_nhwc(dout, hin, win, hu, wu):
    n, ho, wo, c, ld = K._nhwc32(dout)
    din = torch.empty((n, hin, win, c), device=dout.device, dtype=F32)
    _C.call("ub2_f32_upsample_bwd", ptr(dout), ld, ptr(din), n, hin, win, hu, wu, ho, wo, c, stream(),
            work=(0.0, K._nbytes(dout, din)))
    return din


def pack_convt_weight(weight, bias):
    """(Cin, Cout, 2, 2) fp32 parameter -> (the exact 1x1 weight (4*Cout, Cin, 1, 1) OIHW, row (i*2+j)*Cout + co;
    scale4 = ones, shift4 = bias tiled four times)."""
    cin, cout = weight.shape[0], weight.shape[1]
    w1 = torch.empty((4 * cout, cin, 1, 1), device=weight.device, dtype=F32)
    ss = torch.empty((2, 4 * cout), device=weight.device, dtype=F32)
    _C.call("ub2_f32_pack_convt_weight", ptr(weight.contiguous()), ptr(bias), ptr(w1), ptr(ss[0]), ptr(ss[1]), cin, cout,
            stream())
    return w1, ss[0], ss[1]


def shuffle2x2(t, cout, out_h, out_w):
    """t (N,h,w,4*Cout) fp32 -> (N,out_h,out_w,Cout): pixel shuffle of the transposed convolution + F.pad (zeros)."""
    n, h, w, c4, ld = K._nhwc32(t)
    assert c4 == 4 * cout
    out = torch.empty((n, out_h, out_w, cout), device=t.device, dtype=F32)
    _C.call("ub2_f32_shuffle2x2_fwd", ptr(t), ld, ptr(out), cout, n, h, w, cout, out_h, out_w, stream(),
            work=(0.0, K._nbytes(t, out)))
    return out


def shuffle2x2_bwd(dout, h, w, want_bias=True):
    """Transpose of shuffle2x2: dout (N,Ho,Wo,Cout), channel stride may exceed Cout -> (dt (N,h,w,4*Cout),
    bias gradient (Cout,) or None)."""
    n, ho, wo, cout, ld = K._nhwc32(dout)
    dt = torch.empty((n, h, w, 4 * cout), device=dout.device, dtype=F32)
    partials = db = None
    rows = 0
    if want_bias:
        rows = K._rows("ub2_f32_shuffle2x2_rows", n, h, w, cout, ho, wo)
        partials = torch.empty((rows, cout), device=dout.device, dtype=F64)
        db = torch.zeros((cout,), device=dout.device, dtype=F32)
    _C.call("ub2_f32_shuffle2x2_bwd", ptr(dout), ld, ptr(dt), 4 * cout, ptr(partials), rows, ptr(db), n, h, w, cout, ho, wo,
            stream(), work=(0.0, K._nbytes(dout, dt)))
    return dt, db


def split_bf16(x):
    """fp32 NHWC -> (hi, lo) bf16 NHWC with x = hi + lo to 2^-16 relative."""
    x = _dense(x)
    hi = torch.empty(x.shape, device=x.device, dtype=BF16)
    lo = torch.empty(x.shape, device=x.device, dtype=BF16)
    _C.call("ub2_f32_split_bf16", ptr(x), ptr(hi), ptr(lo), _C.c_longlong(x.numel()), stream(), work=(0.0, K._nbytes(x, hi, lo)))
    return hi, lo


def _hilo_wgrad(x0, x1, dy, taps, fold):
    """Weight gradient from fp32 operands: three bf16 tensor-core weight-gradient launches on the hi / lo halves
    (a_hi.dy_hi + a_lo.dy_hi + a_hi.dy_lo); ``fold(partial, accumulate)`` reduces each launch's split-K partials
    into the caller's fp32 gradient, the first one overwriting it, in this fixed order."""
    x0h, x0l = split_bf16(x0)
    x1h, x1l = split_bf16(x1) if x1 is not None else (None, None)
    dyh, dyl = split_bf16(dy)
    fold(K.conv_wgrad(x0h, dyh, taps, x1=x1h), False)
    fold(K.conv_wgrad(x0l, dyh, taps, x1=x1l), True)
    fold(K.conv_wgrad(x0h, dyl, taps, x1=x1h), True)


def weight_grad(x0, x1, dy, wshape):
    """dW (OIHW fp32) of a convolution from fp32 operands (see _hilo_wgrad)."""
    cout, cin, kh, kw = wshape
    taps = kh * kw
    gw = torch.empty(wshape, device=dy.device, dtype=F32)
    _hilo_wgrad(x0, x1, dy, taps, lambda part, acc: K.wgrad_reduce(part, cout, cin, taps, gw, accumulate=acc))
    return gw


def convt_weight_grad(a, dt, wshape):
    """dW (Cin, Cout, 2, 2) fp32 of the transposed convolution: the 1x1 weight gradient of a (N,h,w,Cin) against the
    shuffled gradient dt (N,h,w,4*Cout), folded into the ConvTranspose2d layout."""
    cin, cout = wshape[0], wshape[1]
    gw = torch.empty(wshape, device=dt.device, dtype=F32)
    _hilo_wgrad(a, None, dt, 1, lambda part, acc: K.convt_wgrad_reduce(part, cin, cout, gw, accumulate=acc))
    return gw


def _bn_coeffs_train(part, count, bn):
    from . import ops
    return ops._bn_train_coeffs(part, count, bn)


def _bn_stage(y, bn):
    """statistics (batch or running) -> (scale, shift, mean, invstd, batch?)"""
    from . import ops
    n, h, w, c = y.shape
    if ops._use_batch_stats(bn):
        return (*ops._bn_train_coeffs(channel_stats(y), n * h * w, bn), True)
    return (*ops._bn_frozen_coeffs(bn), False)


class ConvBnReluF32(torch.autograd.Function):
    """conv3x3 over one or two (virtually concatenated) inputs -> BatchNorm -> ReLU (+ 2x2 max-pooled copy):
    DoubleConv / Down / the concat in Up (layers.py:31-38, :56, :105) in fp32 / TF32."""

    @staticmethod
    def forward(ctx, x0, x1, weight, gamma, beta, bn, pool):
        a0 = nhwc_view(x0)
        a1 = nhwc_view(x1) if x1 is not None else None
        cout, cin, kh, kw = weight.shape
        y = conv3(a0, a1, weight)
        scale, shift, mean, invstd, batch = _bn_stage(y, bn)
        a = affine_act(y, scale, shift, relu=True)
        p, pidx = maxpool_idx(a) if pool else (None, None)
        ctx.save_for_backward(a0, a1, y, scale, shift, mean, invstd, gamma, weight, pidx)
        ctx.batch = batch
        return nchw(a), (nchw(p) if pool else None)

    @staticmethod
    def backward(ctx, dA, dP):
        a0, a1, y, scale, shift, mean, invstd, gamma, weight, pidx = ctx.saved_tensors
        cout, cin, kh, kw = weight.shape
        dA_n = nhwc_view(dA) if dA is not None else None
        dP_n = nhwc_view(dP) if dP is not None else None
        dy, dgamma, dbeta = act_backward(dA_n, dP_n, pidx, y, scale, shift, mean, invstd, gamma, ctx.batch)
        gw = weight_grad(a0, a1, dy, weight.shape) if ctx.needs_input_grad[2] else None
        d0 = d1 = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            c0 = a0.shape[3]
            dfull = conv3(dy, None, weight, dgrad=True)
            d0 = nchw(dfull[..., :c0])
            d1 = nchw(dfull[..., c0:]) if a1 is not None else None
        return d0, d1, gw, dgamma, dbeta, None, None


class ConvInBnReluF32(torch.autograd.Function):
    """First stage: conv3x3 on the fp32 NCHW network input (Cin = n_channels) -> BN -> ReLU, exact fp32."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, bn):
        if not x.is_cuda:
            raise RuntimeError("unet-b200 modules run on CUDA tensors only (no CPU fallback)")
        x_dtype = x.dtype
        x = x.contiguous().float()
        n, cin, h, w = x.shape
        cout = weight.shape[0]
        y = torch.empty((n, h, w, cout), device=x.device, dtype=F32)
        _C.call("ub2_f32_conv_in_raw", ptr(x), ptr(weight.contiguous()), ptr(y), n, cin, h, w, cout, stream())
        scale, shift, mean, invstd, batch = _bn_stage(y, bn)
        a = affine_act(y, scale, shift, relu=True)
        ctx.save_for_backward(x, y, scale, shift, mean, invstd, gamma,
                              weight if ctx.needs_input_grad[0] else None)
        ctx.meta = (weight.shape, batch, x_dtype)
        return nchw(a)

    @staticmethod
    def backward(ctx, dA):
        x, y, scale, shift, mean, invstd, gamma, weight = ctx.saved_tensors
        wshape, batch, x_dtype = ctx.meta
        dy, dgamma, dbeta = act_backward(nhwc_view(dA), None, None, y, scale, shift, mean, invstd, gamma, batch)
        dx = K.conv_in_dgrad(dy, weight.contiguous(), wshape[1]).to(x_dtype) if ctx.needs_input_grad[0] else None
        gw = None
        if ctx.needs_input_grad[1]:
            n, cin, h, w = x.shape
            cout = wshape[0]
            rows = K._rows("ub2_f32_channel_rows", _C.c_longlong(n * h * w), cout)
            part = torch.empty((rows, cin, 9, cout), device=x.device, dtype=F64)
            gw = torch.zeros(wshape, device=x.device, dtype=F32)
            _C.call("ub2_f32_conv_in_wgrad", ptr(x), ptr(dy), ptr(part), rows, ptr(gw), n, cin, h, w, cout, stream())
        return dx, gw, dgamma, dbeta, None


class MaxPoolF32(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        a = _dense(nhwc_view(x))
        p, idx = maxpool_idx(a)
        ctx.save_for_backward(idx)
        ctx.shape = a.shape
        return nchw(p)

    @staticmethod
    def backward(ctx, dp):
        (idx,) = ctx.saved_tensors
        n, h, w, c = ctx.shape
        # route through the BN-backward apply with identity coefficients (dy = routed gradient)
        dev = idx.device
        ones, zeros = torch.ones(c, device=dev), torch.zeros(c, device=dev)
        coef = torch.stack([ones, zeros, zeros])
        dummy_y = torch.zeros((n, h, w, c), device=dev, dtype=F32)
        dy = torch.empty((n, h, w, c), device=dev, dtype=F32)
        _C.call("ub2_f32_act_bwd_apply", ptr(None), 0, ptr(_dense(nhwc_view(dp))), ptr(idx), ptr(dummy_y), ptr(ones), ptr(zeros),
                ptr(coef), ptr(dy), n, h, w, c, 0, stream())
        return nchw(dy)


class UpsampleF32(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, out_h, out_w):
        a = _dense(nhwc_view(x))
        ctx.geom = (a.shape[1], a.shape[2])
        return nchw(upsample_nhwc(a, out_h, out_w))

    @staticmethod
    def backward(ctx, dout):
        h, w = ctx.geom
        return nchw(upsample_bwd_nhwc(nhwc_view(dout), h, w, 2 * h, 2 * w)), None, None


class ConvTranspose2x2F32(torch.autograd.Function):
    """nn.ConvTranspose2d(C, C/2, 2, stride 2) + F.pad in fp32 / TF32 training: the 1x1 convolution to 4*Cout
    channels as one 3xTF32 launch (bias in its epilogue) and the fp32 pixel shuffle; backward: the shuffle's
    transpose with the bias gradient, the hi/lo bf16 weight gradient and one 3xTF32 data-gradient launch."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_h, out_w):
        a = nhwc_view(x)
        cin, cout = weight.shape[0], weight.shape[1]
        w1, scale4, shift4 = pack_convt_weight(weight, bias)
        split = split_tf32(a)
        t = conv_packed(split, split[..., :cin], _pack3(w1), 4 * cout, 1, scale4, shift4, exact=True)
        ctx.save_for_backward(a, w1)
        ctx.meta = (weight.shape, bias is not None)
        return nchw(shuffle2x2(t, cout, out_h, out_w))

    @staticmethod
    def backward(ctx, dout):
        a, w1 = ctx.saved_tensors
        wshape, has_bias = ctx.meta
        need_x, need_w, need_b = ctx.needs_input_grad[:3]
        dt, db = shuffle2x2_bwd(nhwc_view(dout), a.shape[1], a.shape[2], want_bias=has_bias and need_b)
        gw = convt_weight_grad(a, dt, wshape) if need_w else None
        dx = nchw(conv3(dt, None, w1, dgrad=True)) if need_x else None
        return dx, gw, db, None, None


class AttentionGateF32(torch.autograd.Function):
    """AttentionGate.forward (layers.py:171-192) in fp32 / TF32: two tensor-core 1x1 projections (W_g at low
    resolution: it commutes with the bilinear resampling) and plain fp32 passes; up(q) is materialised."""

    @staticmethod
    def forward(ctx, g, x, w_g, w_x, w_psi, gam_g, bet_g, gam_x, bet_x, gam_p, bet_p, bn_g, bn_x, bn_p):
        from . import ops
        gn, xn = _dense(nhwc_view(g)), _dense(nhwc_view(x))
        n, h, w, cx = xn.shape
        ci = w_g.shape[0]
        count = n * h * w
        q = conv3(gn, None, w_g)
        xp = conv3(xn, None, w_x)
        u = upsample_nhwc(q, h, w, hu=h, wu=w)   # F.interpolate(g, size=x.size()) (layers.py:183)
        sg, hg, mg, ig, batch = _bn_stage(u, bn_g)
        sx, hx, mx, ix, _ = _bn_stage(xp, bn_x)
        wpsi = w_psi.reshape(-1).contiguous()
        psi = torch.empty((n, h, w), device=xn.device, dtype=F32)
        _C.call("ub2_f32_gate_psi", ptr(u), ptr(xp), ptr(sg), ptr(hg), ptr(sx), ptr(hx), ptr(wpsi), ptr(psi),
                _C.c_longlong(count), ci, stream(), work=(0.0, K._nbytes(u, xp, psi)))
        if batch:
            sp, hp, mp, ip = ops._bn_train_coeffs(scalar_stats(psi), count, bn_p)
        else:
            sp, hp, mp, ip = ops._bn_frozen_coeffs(bn_p)
        out = torch.empty_like(xn)
        a = torch.empty((n, h, w), device=xn.device, dtype=F32)
        _C.call("ub2_f32_gate_apply", ptr(psi), ptr(sp), ptr(hp), ptr(xn), ptr(out), ptr(a), _C.c_longlong(count), cx, stream(),
                work=(0.0, K._nbytes(psi, xn, out, a)))
        ctx.save_for_backward(gn, xn, u, xp, psi, a, sg, hg, mg, ig, sx, hx, mx, ix, mp, ip, wpsi, gam_g, gam_x, gam_p,
                              w_g, w_x)
        ctx.meta = (w_psi.shape, batch)
        return nchw(out)

    @staticmethod
    def backward(ctx, dout):
        (gn, xn, u, xp, psi, a, sg, hg, mg, ig, sx, hx, mx, ix, mp, ip, wpsi, gam_g, gam_x, gam_p, w_g,
         w_x) = ctx.saved_tensors
        sh_p, batch = ctx.meta
        n, h, w, cx = xn.shape
        _, hin, win, cg = gn.shape
        ci = u.shape[3]
        count = n * h * w
        d = nhwc_view(dout)
        ld_do = K._nhwc32(d)[4]
        rows = K._rows("ub2_f32_gate_rows", _C.c_longlong(count))
        dx = torch.empty_like(xn)
        dpsin = torch.empty((n, h, w), device=xn.device, dtype=F32)
        part = torch.empty((rows, 2, 1), device=xn.device, dtype=F64)
        _C.call("ub2_f32_gate_bwd_a", ptr(d), ld_do, ptr(xn), ptr(a), ptr(psi), ptr(dx), ptr(dpsin), ptr(part), rows,
                _C.c_longlong(count), cx, stream(), work=(0.0, K._nbytes(d, xn, a, psi, dx, dpsin)))
        dgam_p, dbet_p, coef_p = K.bn_bwd_finalize(part, count, gam_p, mp, ip, frozen=not batch)
        ds = torch.empty_like(xp)
        part2 = torch.empty((rows, 4, ci), device=xn.device, dtype=F64)
        _C.call("ub2_f32_gate_bwd_s", ptr(dpsin), ptr(psi), ptr(coef_p), ptr(u), ptr(xp), ptr(sg), ptr(hg), ptr(sx), ptr(hx),
                ptr(wpsi), ptr(ds), ptr(part2), rows, _C.c_longlong(count), ci, stream(),
                work=(0.0, K._nbytes(dpsin, psi, u, xp, ds)))
        grads, coef = K.gate_bwd_finalize(part2, count, gam_x, mx, ix, gam_g, mg, ig, frozen=not batch)
        dxp = torch.empty_like(xp)
        du = torch.empty_like(xp)
        _C.call("ub2_f32_gate_bwd_xg", ptr(ds), ptr(xp), ptr(u), ptr(coef), ptr(dxp), ptr(du), _C.c_longlong(count), ci,
                stream(), work=(0.0, K._nbytes(ds, xp, u, dxp, du)))
        dq = upsample_bwd_nhwc(du, hin, win, h, w)
        gw_x = weight_grad(xn, None, dxp, w_x.shape)
        gw_g = weight_grad(gn, None, dq, w_g.shape)
        dx = dx + conv3(dxp, None, w_x, dgrad=True)
        dg = conv3(dq, None, w_g, dgrad=True)
        # grads rows: dgamma_x, dbeta_x, dgamma_g, dbeta_g, dwpsi
        return (nchw(dg), nchw(dx), gw_g, gw_x, grads[4].reshape(sh_p), grads[2], grads[3], grads[0], grads[1],
                dgam_p, dbet_p, None, None, None)


class OutConvF32(torch.autograd.Function):
    """OutConv (layers.py:120-123): 1x1 conv with bias to fp32 NCHW logits, exact fp32."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        a = _dense(nhwc_view(x))
        n, h, w, c = a.shape
        k = weight.shape[0]
        logits = torch.empty((n, k, h, w), device=a.device, dtype=F32)
        _C.call("ub2_f32_outc", ptr(a), ptr(weight.reshape(k, -1).contiguous()), ptr(bias), ptr(logits), n, h, w, c, k, stream(),
                work=(0.0, K._nbytes(a, logits)))
        ctx.save_for_backward(a, weight)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        a, weight = ctx.saved_tensors
        n, h, w, c = a.shape
        k = weight.shape[0]
        dl = dlogits.contiguous().float()
        rows = K._rows("ub2_f32_outc_rows", n, h, w)
        part = torch.empty((rows, k * c + k), device=a.device, dtype=F64)
        da = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        dw = torch.zeros(weight.shape, device=a.device, dtype=F32)
        db = torch.zeros((k,), device=a.device, dtype=F32)
        _C.call("ub2_f32_outc_bwd", ptr(dl), ptr(a), ptr(weight.reshape(k, -1).contiguous()), ptr(da), ptr(part), rows, ptr(dw),
                ptr(db), n, h, w, c, k, stream(), work=(0.0, K._nbytes(dl, a, da)))
        return (nchw(da) if da is not None else None), dw, db
