"""Typed Python wrappers over the C ABI (one function per entry point family): the only module of
the package that launches (``_C.call``).

All tensors are CUDA tensors; activations are NHWC bf16 ``(N, H, W, C)`` views (fp32 in the fp32 /
TF32 section at the end) that are dense in their last dimension.  These wrappers only allocate outputs /
workspaces with torch and pass raw pointers through ctypes; nothing here
computes on the host and nothing synchronises the device, so a whole training
step can be captured into a CUDA graph.
"""
from __future__ import annotations

import ctypes

import torch

from . import _C
from ._C import byref, c_int, ptr, stream

BF16 = torch.bfloat16
F32 = torch.float32
F64 = torch.float64

_SMS = None


def _nbytes(*tensors) -> int:
    """Algorithmic bytes of a bandwidth-bound call: every tensor it reads or writes, touched once."""
    return sum(t.numel() * t.element_size() for t in tensors if t is not None)


def num_sms() -> int:
    global _SMS
    if _SMS is None:
        _SMS = int(_C.lib().ub2_num_sms())
    return _SMS


def last_conv_variant() -> int:
    """Kernel the dispatcher picked for this thread's last conv_fwd / conv_wgrad (see unetb200.h)."""
    return int(_C.lib().ub2_last_conv_variant())


def _nhwc(t: torch.Tensor):
    assert t.dim() == 4 and t.dtype == BF16 and t.stride(3) == 1, "expected NHWC bf16"
    n, h, w, c = t.shape
    ld = t.stride(2) if w > 1 else c
    if h > 1:
        assert t.stride(1) == w * ld, "expected dense NHWC rows"
    if n > 1:
        assert t.stride(0) == h * w * ld, "expected dense NHWC images"
    return n, h, w, c, ld


def _nhwc32(t: torch.Tensor, dense=False):
    """fp32 / TF32 mode: (N,H,W,C) fp32 whose channel stride may exceed C (a channel slice); ``dense``: the
    entry point takes no channel stride, so the stride must be C."""
    assert t.dim() == 4 and t.dtype == F32 and t.stride(3) == 1, "expected NHWC fp32"
    assert not dense or t.is_contiguous(), "expected dense NHWC fp32"
    n, h, w, c = t.shape
    # the stride between consecutive pixels: across a row, or (W = 1) down the rows, or (H = W = 1) across images
    ld = t.stride(2) if w > 1 else t.stride(1) if h > 1 else t.stride(0) if n > 1 else c
    if h > 1:
        assert t.stride(1) == w * ld, "expected dense NHWC rows"
    if n > 1:
        assert t.stride(0) == h * w * ld, "expected dense NHWC images"
    return n, h, w, c, ld


def empty_nhwc(n, h, w, c, device):
    return torch.empty((n, h, w, c), device=device, dtype=BF16)


def _rows(name, *args) -> int:
    r = int(getattr(_C.lib(), name)(*args))
    if r <= 0:
        _C.check(r if r < 0 else -1, name)
    return r


# --------------------------------------------------------------------------- convolution
def conv_fwd(x0, wgt, taps, x1=None, out=None, out1=None, split=0, scale=None, shift=None,
             relu=False, accumulate=False, stats=False, bn_override=0, grid_override=0):
    """Implicit-GEMM conv (3x3 pad 1 or 1x1). ``wgt``: (Cout, taps, C0+C1) bf16.

    Returns ``out`` or ``(out, stats_partials)`` where stats_partials is a
    (rows, 2, Cout) float64 tensor of per-CTA sums / sums of squares.
    """
    n, h, w, c0, ld0_in = _nhwc(x0)
    c1, ld1_in = 0, 0
    if x1 is not None:
        n1, h1, w1, c1, ld1_in = _nhwc(x1)
        assert (n1, h1, w1) == (n, h, w)
    cout = wgt.shape[0]
    assert wgt.dtype == BF16 and wgt.is_contiguous() and wgt.numel() == cout * taps * (c0 + c1)
    if out is None:
        out = empty_nhwc(n, h, w, cout if out1 is None else split, x0.device)
    _, _, _, _, ldo0 = _nhwc(out)
    ldo1 = 0
    if out1 is not None:
        _, _, _, _, ldo1 = _nhwc(out1)
    st = None
    rows = 0
    if stats:
        rows = num_sms()
        st = torch.empty((rows, 2, cout), device=x0.device, dtype=F64)
    used = c_int(0)
    _C.call("ub2_conv_fwd", ptr(x0), ld0_in, c0, ptr(x1), ld1_in, c1, ptr(wgt), ptr(out), ldo0,
            ptr(out1), ldo1, split, n, h, w, cout, taps, ptr(scale), ptr(shift), int(relu),
            int(accumulate), ptr(st), rows, byref(used), bn_override, grid_override, stream(),
            work=(2.0 * n * h * w * cout * taps * (c0 + c1), _nbytes(x0, x1, wgt, out, out1)))
    if stats:
        return out, st[: used.value]
    return out


def conv_wgrad(x0, dy, taps, x1=None, splits_override=0):
    """Split-K partial weight gradients: (splits, taps*(C0+C1), Cout) fp32."""
    n, h, w, c0, ld0_in = _nhwc(x0)
    c1, ld1_in = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1_in = _nhwc(x1)
    n2, h2, w2, cout, ld_dy = _nhwc(dy)
    assert (n2, h2, w2) == (n, h, w)
    mtot = taps * (c0 + c1)
    max_splits = max(1, min(2 * num_sms(), (96 << 20) // (mtot * cout * 4)))
    partial = torch.empty((max_splits, mtot, cout), device=x0.device, dtype=F32)
    used = c_int(0)
    _C.call("ub2_conv_wgrad", ptr(x0), ld0_in, c0, ptr(x1), ld1_in, c1, ptr(dy), ld_dy,
            ptr(partial), max_splits, byref(used), n, h, w, cout, taps, splits_override, stream(),
            work=(2.0 * n * h * w * cout * mtot, _nbytes(x0, x1, dy) + 4 * mtot * cout))
    return partial[: used.value]


def wgrad_reduce(partial, cout, cin, taps, grad, accumulate=False):
    """grad (Cout,Cin,k,k) fp32 = (or +=) sum over splits of partial (splits, taps*Cin, Cout).
    ``partial`` is consumed (used as scratch)."""
    assert grad.dtype == F32 and grad.is_contiguous() and partial.is_contiguous()
    _C.call("ub2_wgrad_reduce", ptr(partial), partial.shape[0], cout, cin, taps, ptr(grad), int(accumulate),
            stream())
    return grad


class _ReduceItem(ctypes.Structure):
    _fields_ = [("partial", ctypes.c_void_p), ("grad", ctypes.c_void_p), ("splits", ctypes.c_int),
                ("Cout", ctypes.c_int), ("Cin", ctypes.c_int), ("taps", ctypes.c_int)]


def wgrad_reduce_multi(items, accumulate=True):
    """Fold the split-K partials of several layers in one or two launches.
    ``items``: (partial, cout, cin, taps, grad) tuples; see ``wgrad_reduce``."""
    for i in range(0, len(items), 32):
        chunk = items[i:i + 32]
        arr = (_ReduceItem * len(chunk))()
        for j, (partial, cout, cin, taps, grad) in enumerate(chunk):
            assert grad.dtype == F32 and grad.is_contiguous() and partial.is_contiguous()
            arr[j] = _ReduceItem(partial.data_ptr(), grad.data_ptr(), partial.shape[0], cout, cin, taps)
        _C.call("ub2_wgrad_reduce_multi", arr, len(chunk), int(accumulate), stream())


def pack_conv_weight(w, want_fwd=True, want_dgrad=True, out_scale=None):
    """OIHW fp32 parameter -> (fwd pack (Cout,taps,Cin), dgrad pack (Cin,taps,Cout)) bf16."""
    cout, cin, kh, kw = w.shape
    taps = kh * kw
    assert w.dtype == F32 and w.is_contiguous()
    fwd = torch.empty((cout, taps, cin), device=w.device, dtype=BF16) if want_fwd else None
    dg = torch.empty((cin, taps, cout), device=w.device, dtype=BF16) if want_dgrad else None
    _C.call("ub2_pack_conv_weight", ptr(w), ptr(fwd), ptr(dg), cout, cin, taps, ptr(out_scale), stream())
    return fwd, dg


class WeightPacker:
    """bf16 packs of many conv weights rebuilt by ONE launch (``ub2_pack_conv_weights_multi``).

    The packs only change when the optimizer steps, so a training step rebuilds them once at its
    start instead of launching a small kernel per layer inside forward.  ``get(w)`` returns the
    (forward, data-gradient) packs of a registered weight or None."""

    def __init__(self, weights):
        self.entries = {}
        desc, blocks = [], []
        for w in weights:
            cout, cin, kh, kw = w.shape
            taps = kh * kw
            if not (w.is_cuda and w.dtype == F32 and w.is_contiguous() and cout % 8 == 0 and cin % 8 == 0
                    and taps in (1, 9)) or id(w) in self.entries:
                continue
            fwd = torch.empty((cout, taps, cin), device=w.device, dtype=BF16)
            dg = torch.empty((cin, taps, cout), device=w.device, dtype=BF16)
            t = len(desc)
            desc.append([w.data_ptr(), fwd.data_ptr(), dg.data_ptr(), cout, cin, taps])
            # 4th field: a tile that reaches past Cin or Cout (channel counts not multiples of 16) -> edge path
            blocks += [[t, ci, co, int(16 * ci + 16 > cin or 16 * co + 16 > cout)]
                       for co in range((cout + 15) // 16) for ci in range((cin + 15) // 16)]
            self.entries[id(w)] = (w, w.data_ptr(), fwd, dg)
        self.nblocks = len(blocks)
        if self.nblocks:
            dev = next(iter(self.entries.values()))[0].device
            self.desc = torch.tensor(desc, dtype=torch.int64).to(dev)
            self.blocks = torch.tensor(blocks, dtype=torch.int32).to(dev)

    def run(self):
        if self.nblocks:
            _C.call("ub2_pack_conv_weights_multi", ptr(self.desc), ptr(self.blocks), self.nblocks, stream())

    def get(self, w):
        e = self.entries.get(id(w))
        if e is None or e[0] is not w or e[1] != w.data_ptr():
            return None
        return e[2], e[3]


# --------------------------------------------------------------------------- batch norm
def bn_finalize(partials, count, gamma, beta, running_mean, running_var, nbt, momentum, eps):
    """Per-CTA sums -> (scale, shift, mean, invstd); updates the running buffers in place."""
    rows, _, c = partials.shape
    dev = partials.device
    out = torch.empty((4, c), device=dev, dtype=F32)
    _C.call("ub2_bn_finalize", ptr(partials), rows, c, count, ptr(gamma), ptr(beta),
            ptr(running_mean), ptr(running_var), ptr(nbt), momentum, eps,
            ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(out[3]), stream())
    return out[0], out[1], out[2], out[3]


def bn_eval_coeffs(gamma, beta, running_mean, running_var, eps):
    c = running_mean.numel()
    out = torch.empty((2, c), device=running_mean.device, dtype=F32)
    _C.call("ub2_bn_eval_coeffs", ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
            eps, c, ptr(out[0]), ptr(out[1]), stream())
    return out[0], out[1]


def bn_act(y, scale, shift, relu=True, pool=False, write_act=True, want_idx=False):
    """a = relu(scale*y+shift), optionally its 2x2 max-pooled copy and the uint8 window position of
    each maximum (saved for the backward pass)."""
    n, h, w, c, ld = _nhwc(y)
    a = empty_nhwc(n, h, w, c, y.device) if write_act else None
    p = empty_nhwc(n, h // 2, w // 2, c, y.device) if pool else None
    idx = torch.empty((n, h // 2, w // 2, c), device=y.device, dtype=torch.uint8) if pool and want_idx else None
    _C.call("ub2_bn_act", ptr(y), ld, ptr(scale), ptr(shift), ptr(a), c, ptr(p), c, ptr(idx), n, h, w, c,
            int(relu), stream(), work=(0.0, _nbytes(y, a, p, idx)))
    if want_idx:
        return a, p, idx
    return a, p


def bn_backward(dA, dP, pidx, y, scale, shift, mean, invstd, gamma, relu=True, frozen=False,
                dgamma=None, dbeta=None, exchange=None):
    """BatchNorm(+ReLU, + max-pool routing) backward: returns (dy bf16, dgamma, dbeta).
    ``frozen``: statistics were the running buffers (eval-mode backward), no mean terms.
    ``dgamma`` / ``dbeta``: existing fp32 gradient buffers to accumulate into (then None is
    returned in their place).  ``exchange``: SyncBatchNorm (see ``synced_coef``)."""
    n, h, w, c, ld_y = _nhwc(y)
    ld_da = _nhwc(dA)[4] if dA is not None else 0
    ld_dp = _nhwc(dP)[4] if dP is not None else 0
    rows = _rows("ub2_bn_bwd_rows", n, h, w, c, int(dP is not None))
    dev = y.device
    partials = torch.empty((rows, 2, c), device=dev, dtype=F64)
    _C.call("ub2_bn_bwd_reduce", ptr(dA), ld_da, ptr(dP), ld_dp, ptr(pidx), ptr(y), ld_y, ptr(scale),
            ptr(shift), ptr(partials), rows, n, h, w, c, int(relu), stream(), work=(0.0, _nbytes(dA, dP, pidx, y)))
    dgamma, dbeta, coef = bn_bwd_finalize(partials, n * h * w, gamma, mean, invstd, frozen, dgamma, dbeta)
    if exchange is not None:
        coef = synced_coef(partials, n * h * w, exchange, gamma, mean, invstd, frozen)
    dy = empty_nhwc(n, h, w, c, dev)
    _C.call("ub2_bn_bwd_apply", ptr(dA), ld_da, ptr(dP), ld_dp, ptr(pidx), ptr(y), ld_y, ptr(scale),
            ptr(shift), ptr(coef), ptr(dy), c, n, h, w, c, int(relu), stream(),
            work=(0.0, _nbytes(dA, dP, pidx, y, dy)))
    return dy, dgamma, dbeta


def bn_bwd_finalize(partials, count, gamma, mean, invstd, frozen=False, dgamma=None, dbeta=None, grads=True):
    """(sum g, sum g*y) rows -> (dgamma, dbeta, coef[3,C]) with dy = coef0*g + coef1*y + coef2.
    The kernel accumulates (+=): into fresh zeros, or into the given ``dgamma`` / ``dbeta``;
    ``grads=False``: coefficients only (no gradient is written, None is returned for both)."""
    rows, _, c = partials.shape
    direct = dgamma is not None and dbeta is not None
    if not grads:
        dgamma = dbeta = None
        direct = True
    elif not direct:
        grads = torch.zeros((2, c), device=partials.device, dtype=F32)
        dgamma, dbeta = grads[0], grads[1]
    coef = torch.empty((3, c), device=partials.device, dtype=F32)
    _C.call("ub2_bn_bwd_finalize", ptr(partials), rows, c, count, ptr(gamma), ptr(mean),
            ptr(invstd), int(frozen), ptr(dgamma), ptr(dbeta), ptr(coef), stream())
    if direct:
        return None, None, coef
    return dgamma, dbeta, coef


def synced_coef(partials, count, exchange, gamma, mean, invstd, frozen=False):
    """SyncBatchNorm backward: the apply coefficients of one BatchNorm from the (sum g, sum g*y) rows of every
    rank.  ``exchange(partials, count)`` returns the rows summed over the ranks and the pixel count over the
    ranks (unet.syncbn.exchange); it sums ``partials`` in place when the ranks' row counts agree.  The caller has
    already finalized ``partials`` into dgamma / dbeta: those stay the LOCAL sums, which the trainer's gradient
    all-reduce then adds up over the ranks (as DDP does with nn.SyncBatchNorm)."""
    partials, count = exchange(partials, count)
    return bn_bwd_finalize(partials, count, gamma, mean, invstd, frozen, grads=False)[2]


def maxpool_bwd(dP, pidx, a):
    """Route the pooled gradient to the saved window positions (no BN, no ReLU)."""
    n, h, w, c, ld = _nhwc(a)
    dev = a.device
    ident = torch.zeros((5, c), device=dev, dtype=F32)
    ident[0].fill_(1.0)   # scale = 1
    ident[2].fill_(1.0)   # coef A = 1 (B = C = 0, shift = 0)
    dy = empty_nhwc(n, h, w, c, dev)
    _C.call("ub2_bn_bwd_apply", ptr(None), 0, ptr(dP), _nhwc(dP)[4], ptr(pidx), ptr(a), ld, ptr(ident[0]),
            ptr(ident[1]), ptr(ident[2]), ptr(dy), c, n, h, w, c, 0, stream())
    return dy


# --------------------------------------------------------------------------- resampling
def upsample(x, hu, wu, ho, wo):
    n, hin, win, c, ld = _nhwc(x)
    out = empty_nhwc(n, ho, wo, c, x.device)
    _C.call("ub2_upsample_fwd", ptr(x), ld, ptr(out), c, n, hin, win, hu, wu, ho, wo, c, stream(),
            work=(0.0, _nbytes(x, out)))
    return out


def upsample_bwd(dout, hin, win, hu, wu, into=None):
    n, ho, wo, c, ld = _nhwc(dout)
    acc = into is not None
    din = into if acc else empty_nhwc(n, hin, win, c, dout.device)
    _C.call("ub2_upsample_bwd", ptr(dout), ld, ptr(din), _nhwc(din)[4], int(acc), n, hin, win, hu, wu,
            ho, wo, c, stream(), work=(0.0, _nbytes(dout, din) * (2 if acc else 1) - (_nbytes(dout) if acc else 0)))
    return din


# --------------------------------------------------------------------------- attention gate
def gate_rows(n, h, w, c):
    return _rows("ub2_gate_rows", n, h, w, c)


def gate_strip_rows(n, h, w, c):
    return _rows("ub2_gate_strip_rows", n, h, w, c)


def gate_upstats(q, h, w):
    n, hin, win, ci, ld = _nhwc(q)
    rows = gate_strip_rows(n, h, w, ci)
    partials = torch.empty((rows, 2, ci), device=q.device, dtype=F64)
    _C.call("ub2_gate_upstats", ptr(q), ld, n, hin, win, h, w, ci, ptr(partials), rows, stream(),
            work=(0.0, _nbytes(q)))
    return partials


def gate_psi(q, xp, sg, hg, sx, hx, wpsi, stats=True):
    n, hin, win, ci, ld_q = _nhwc(q)
    _, h, w, _, ld_xp = _nhwc(xp)
    psi = torch.empty((n, h, w), device=q.device, dtype=F32)
    rows = gate_strip_rows(n, h, w, ci)
    partials = torch.empty((rows, 2, 1), device=q.device, dtype=F64) if stats else None
    _C.call("ub2_gate_psi", ptr(q), ld_q, ptr(xp), ld_xp, ptr(sg), ptr(hg), ptr(sx), ptr(hx), ptr(wpsi),
            ptr(psi), ptr(partials), rows, n, hin, win, h, w, ci, stream(), work=(0.0, _nbytes(q, xp, psi)))
    return psi, partials


def gate_fused_eval(q, xp, x, sg, hg, sx, hx, wpsi, spsi, hpsi):
    """Inference: out = x * sigmoid(BN_psi(w_psi . relu(BN_g(up q) + BN_x(xp)))) in one pass (Cx == 2*Ci)."""
    n, hin, win, ci, ld_q = _nhwc(q)
    _, h, w, _, ld_xp = _nhwc(xp)
    _, _, _, cx, ld_x = _nhwc(x)
    out = empty_nhwc(n, h, w, cx, x.device)
    _C.call("ub2_gate_fused_eval", ptr(q), ld_q, ptr(xp), ld_xp, ptr(x), ld_x, ptr(sg), ptr(hg), ptr(sx), ptr(hx), ptr(wpsi),
            ptr(spsi), ptr(hpsi), ptr(out), cx, n, hin, win, h, w, ci, cx, stream(), work=(0.0, _nbytes(q, xp, x, out)))
    return out


def gate_apply(psi, spsi, hpsi, x, save_a=True):
    n, h, w, cx, ld = _nhwc(x)
    out = empty_nhwc(n, h, w, cx, x.device)
    a = torch.empty((n, h, w), device=x.device, dtype=F32) if save_a else None
    _C.call("ub2_gate_apply", ptr(psi), ptr(spsi), ptr(hpsi), ptr(x), ld, ptr(out), cx, ptr(a), n, h, w,
            cx, stream(), work=(0.0, _nbytes(psi, x, out, a)))
    return out, a


def gate_bwd_a(dout, x, a, psi):
    n, h, w, cx, ld_x = _nhwc(x)
    ld_do = _nhwc(dout)[4]
    dx = empty_nhwc(n, h, w, cx, x.device)
    dpsin = torch.empty((n, h, w), device=x.device, dtype=F32)
    rows = gate_rows(n, h, w, cx)
    partials = torch.empty((rows, 2, 1), device=x.device, dtype=F64)
    _C.call("ub2_gate_bwd_a", ptr(dout), ld_do, ptr(x), ld_x, ptr(a), ptr(psi), ptr(dx), cx, ptr(dpsin),
            ptr(partials), rows, n, h, w, cx, stream(), work=(0.0, _nbytes(dout, x, a, psi, dx, dpsin)))
    return dx, dpsin, partials


def gate_bwd_s(dpsin, psi, coef_psi, q, xp, sg, hg, sx, hx, wpsi):
    n, hin, win, ci, ld_q = _nhwc(q)
    _, h, w, _, ld_xp = _nhwc(xp)
    ds = empty_nhwc(n, h, w, ci, q.device)
    rows = gate_strip_rows(n, h, w, ci)
    partials = torch.empty((rows, 4, ci), device=q.device, dtype=F64)
    _C.call("ub2_gate_bwd_s", ptr(dpsin), ptr(psi), ptr(coef_psi), ptr(q), ld_q, ptr(xp), ld_xp, ptr(sg),
            ptr(hg), ptr(sx), ptr(hx), ptr(wpsi), ptr(ds), ci, ptr(partials), rows, n, hin, win, h, w, ci,
            stream(), work=(0.0, _nbytes(dpsin, psi, q, xp, ds)))
    return ds, partials


def gate_bwd_finalize(partials, count, gamma_x, mean_x, invstd_x, gamma_g, mean_g, invstd_g, frozen=False,
                      targets=None, exchange=None):
    """``targets``: five existing fp32 buffers (dgamma_x, dbeta_x, dgamma_g, dbeta_g, dwpsi) to
    accumulate into instead of fresh zeros.  ``exchange``: SyncBatchNorm — the gradients come from this
    rank's rows, the coefficients from the rows of every rank (see ``synced_coef``)."""
    rows, _, ci = partials.shape
    grads = targets if targets is not None else torch.zeros((5, ci), device=partials.device, dtype=F32)
    coef = torch.empty((6, ci), device=partials.device, dtype=F32)
    _C.call("ub2_gate_bwd_finalize", ptr(partials), rows, ci, count, ptr(gamma_x),
            ptr(mean_x), ptr(invstd_x), ptr(gamma_g), ptr(mean_g), ptr(invstd_g), int(frozen), ptr(grads[0]),
            ptr(grads[1]),
            ptr(grads[2]), ptr(grads[3]), ptr(grads[4]), ptr(coef), stream())
    if exchange is not None:
        partials, count = exchange(partials, count)
        rows = partials.shape[0]
        _C.call("ub2_gate_bwd_finalize", ptr(partials), rows, ci, count, ptr(gamma_x),
                ptr(mean_x), ptr(invstd_x), ptr(gamma_g), ptr(mean_g), ptr(invstd_g), int(frozen), ptr(None),
                ptr(None), ptr(None), ptr(None), ptr(None), ptr(coef), stream())
    # dgamma_x, dbeta_x, dgamma_g, dbeta_g, dwpsi
    return grads, coef


def gate_bwd_xg(ds, xp, q, coef):
    n, hin, win, ci, ld_q = _nhwc(q)
    _, h, w, _, ld_xp = _nhwc(xp)
    dxp = empty_nhwc(n, h, w, ci, q.device)
    dgup = empty_nhwc(n, h, w, ci, q.device)
    _C.call("ub2_gate_bwd_xg", ptr(ds), _nhwc(ds)[4], ptr(xp), ld_xp, ptr(q), ld_q, ptr(coef), ptr(dxp), ci,
            ptr(dgup), ci, n, hin, win, h, w, ci, stream(), work=(0.0, _nbytes(ds, xp, q, dxp, dgup)))
    return dxp, dgup


# --------------------------------------------------------------------------- network ends
def conv_in_fwd(x, w, stats=True):
    """First conv: x (N,Cin,H,W) fp32 NCHW, w (Cout,Cin,3,3) fp32 -> NHWC bf16 (+ stat rows)."""
    assert x.dtype == F32 and x.is_contiguous() and w.dtype == F32 and w.is_contiguous()
    n, cin, h, wd = x.shape
    cout = w.shape[0]
    y = empty_nhwc(n, h, wd, cout, x.device)
    rows = _rows("ub2_conv_in_rows", n, h, wd, cout)
    partials = torch.empty((rows, 2, cout), device=x.device, dtype=F64) if stats else None
    _C.call("ub2_conv_in_fwd", ptr(x), ptr(w), ptr(y), cout, ptr(partials), rows, n, cin, h, wd, cout,
            stream(), work=(2.0 * n * h * wd * cout * 9 * cin, _nbytes(x, y)))
    return y, partials


def conv_in_wgrad(x, dy, cout, grad=None):
    """``grad``: existing (Cout,Cin,3,3) fp32 buffer to accumulate into (default: fresh zeros)."""
    n, cin, h, wd = x.shape
    rows = _rows("ub2_conv_in_rows", n, h, wd, cout)
    partials = torch.empty((rows, cin, 9, cout), device=x.device, dtype=F64)
    if grad is None:
        grad = torch.zeros((cout, cin, 3, 3), device=x.device, dtype=F32)
    _C.call("ub2_conv_in_wgrad", ptr(x), ptr(dy), _nhwc(dy)[4], ptr(partials), rows, ptr(grad), n, cin,
            h, wd, cout, stream(), work=(2.0 * n * h * wd * cout * 9 * cin, _nbytes(x, dy)))
    return grad


def conv_in_dgrad(dy, w, cin):
    """First conv's data gradient: dy (N,H,W,Cout) NHWC bf16 or fp32 (the fp32 / TF32 mode), w (Cout,Cin,3,3)
    fp32 -> dx (N,Cin,H,W) fp32 NCHW."""
    assert w.dtype == F32 and w.is_contiguous()
    if dy.dtype == F32:
        n, h, wd, cout, ld = _nhwc32(dy)
        name = "ub2_f32_conv_in_dgrad"
    else:
        n, h, wd, cout, ld = _nhwc(dy)
        name = "ub2_conv_in_dgrad"
    dx = torch.empty((n, cin, h, wd), device=dy.device, dtype=F32)
    _C.call(name, ptr(dy), ld, ptr(w), ptr(dx), n, cin, h, wd, cout, stream(),
            work=(2.0 * n * h * wd * cout * 9 * cin, _nbytes(dy, dx)))
    return dx


def outc_fwd(a, w, bias):
    n, h, wd, c, ld = _nhwc(a)
    k = w.shape[0]
    logits = torch.empty((n, k, h, wd), device=a.device, dtype=F32)
    _C.call("ub2_outc_fwd", ptr(a), ld, ptr(w), ptr(bias), ptr(logits), n, h, wd, c, k, stream(),
            work=(0.0, _nbytes(a, logits)))
    return logits


def outc_bwd(dlogits, a, w, need_da=True, dw=None, db=None):
    """``dw`` / ``db``: existing fp32 gradient buffers to accumulate into (default: fresh zeros)."""
    n, h, wd, c, ld = _nhwc(a)
    k = w.shape[0]
    assert dlogits.dtype == F32 and dlogits.is_contiguous()
    rows = _rows("ub2_outc_rows", n, h, wd, c)
    partials = torch.empty((rows, k * c + k), device=a.device, dtype=F64)
    da = empty_nhwc(n, h, wd, c, a.device) if need_da else None
    if dw is None:
        dw = torch.zeros((k, c, 1, 1), device=a.device, dtype=F32)
    if db is None:
        db = torch.zeros((k,), device=a.device, dtype=F32)
    _C.call("ub2_outc_bwd", ptr(dlogits), ptr(a), ld, ptr(w), ptr(da), c, ptr(partials), rows, ptr(dw),
            ptr(db), n, h, wd, c, k, stream(), work=(0.0, _nbytes(dlogits, a, da)))
    return da, dw, db


# --------------------------------------------------------------------------- loss / metrics
def seg_stats(logits, targets):
    """(N,4,C) fp32: per image and class {count, CE sum, intersection, prob sum}."""
    assert logits.dtype == F32 and logits.is_contiguous() and targets.dtype == torch.int64
    n, c, h, w = logits.shape
    targets = targets.contiguous()
    blocks = _rows("ub2_seg_stats_blocks", n, h * w)
    partials = torch.empty((n, blocks, c, 4), device=logits.device, dtype=F64)
    stats = torch.empty((n, 4, c), device=logits.device, dtype=F32)
    _C.call("ub2_seg_stats", ptr(logits), ptr(targets), n, c, h * w, ptr(partials), blocks,
            ptr(stats), stream(), work=(0.0, _nbytes(logits, targets)))
    return stats


def seg_stats_bwd(logits, targets, coef, gscale=None):
    """coef (N,3,C) fp32 = {dL/dCE, dL/dI, dL/dP} (times the device scalar ``gscale`` if given);
    returns dL/dlogits (N,C,H,W) fp32."""
    n, c, h, w = logits.shape
    coef = coef.contiguous()
    assert coef.dtype == F32 and coef.shape == (n, 3, c)
    assert gscale is None or (gscale.dtype == F32 and gscale.numel() == 1)
    dl = torch.empty_like(logits)
    _C.call("ub2_seg_stats_bwd", ptr(logits), ptr(targets.contiguous()), ptr(coef), ptr(gscale), n, c,
            h * w, ptr(dl), stream(), work=(0.0, _nbytes(logits, targets, dl)))
    return dl


def dice_bce_head(stats, ce_weight, dice_weight, class_weight, ce_smooth, dice_smooth, ignore_background):
    """stats (N,4,C) -> (loss 0-dim fp32, coef (N,3,C) fp32)."""
    n, _, c = stats.shape
    loss = torch.empty((1,), device=stats.device, dtype=F32)
    coef = torch.empty((n, 3, c), device=stats.device, dtype=F32)
    _C.call("ub2_dice_bce_head", ptr(stats), n, c, ce_weight, dice_weight, class_weight,
            ce_smooth, dice_smooth, int(ignore_background), ptr(loss), ptr(coef), stream())
    return loss[0], coef


def confusion(pred, target, num_classes, cm, ignore_index=None, threshold=None, mask_out=None):
    """cm ((C+1),(C+1)) int64 += histogram of (target, prediction)."""
    target = target.contiguous()
    assert target.dtype == torch.int64 and cm.dtype == torch.int64 and cm.is_contiguous()
    if pred.dim() == 4:
        assert pred.dtype == F32 and pred.is_contiguous()
        n, c, h, w = pred.shape
        assert c == num_classes
        mode = 2 if threshold is not None else 0
    else:
        pred = pred.contiguous()
        assert pred.dtype == torch.int64
        n, h, w = pred.shape
        mode = 1
    _C.call("ub2_confusion", ptr(pred), ptr(target), mode, n, num_classes, h * w,
            ignore_index if ignore_index is not None else 0,
            int(ignore_index is not None), threshold if threshold is not None else 0.5, ptr(cm),
            ptr(mask_out), stream(), work=(0.0, _nbytes(pred, target, mask_out)))
    return cm


# --------------------------------------------------------------------------- either side of the forward
def prepare_batch(images, labels=None, flags=None, mean=0.5, std=0.5, x=None, targets=None):
    """uint8 slices (N,H,W) -> x fp32 (N,1,H,W) = ((px/255)-mean)/std and targets int64 (N,H,W) =
    label > 127, optionally flipped per image (flags uint8 (N): bit 0 horizontal, bit 1 vertical)."""
    assert images.dtype == torch.uint8 and images.dim() == 3 and images.is_contiguous()
    n, h, w = images.shape
    if x is None:
        x = torch.empty((n, 1, h, w), device=images.device, dtype=F32)
    assert x.dtype == F32 and x.is_contiguous() and x.numel() == n * h * w
    if labels is not None:
        assert labels.dtype == torch.uint8 and labels.shape == images.shape and labels.is_contiguous()
        if targets is None:
            targets = torch.empty((n, h, w), device=images.device, dtype=torch.int64)
        assert targets.dtype == torch.int64 and targets.is_contiguous() and targets.numel() == n * h * w
    else:
        targets = None
    if flags is not None:
        assert flags.dtype == torch.uint8 and flags.numel() == n and flags.is_contiguous()
    _C.call("ub2_prepare_batch", ptr(images), ptr(labels), ptr(flags), n, h, w, mean, std,
            ptr(x), ptr(targets), stream())
    return x, targets


def predict_mask(logits, threshold=0.5, mask=None, positives=None):
    """logits fp32 (N,2,H,W) -> (mask uint8 (N,H,W) in {0,255}, positives int32 (N))."""
    assert logits.dim() == 4 and logits.dtype == F32 and logits.is_contiguous()
    n, c, h, w = logits.shape
    if mask is None:
        mask = torch.empty((n, h, w), device=logits.device, dtype=torch.uint8)
    if positives is None:
        positives = torch.empty((n,), device=logits.device, dtype=torch.int32)
    assert mask.dtype == torch.uint8 and mask.is_contiguous() and mask.numel() == n * h * w
    assert positives.dtype == torch.int32 and positives.numel() == n
    _C.call("ub2_predict_mask", ptr(logits), n, c, h * w, threshold, ptr(mask), ptr(positives),
            stream())
    return mask, positives


# --------------------------------------------------------------------------- optimizer tail
def grad_sumsq(ptrs, numel, chunks, nchunks, t, partial, step):
    """Per-chunk fp64 sums of squared gradients (FusedAdamW's device tables, see unetb200.h); step += 1."""
    _C.call("ub2_grad_sumsq", ptr(ptrs), ptr(numel), ptr(chunks), nchunks, t, ptr(partial), ptr(step), stream())


def adamw_step(ptrs, numel, group, chunks, nchunks, t, partial, hyper, step, total_norm, write_grads):
    """Gradient-norm clipping + AdamW update in place from grad_sumsq's partials."""
    _C.call("ub2_adamw_step", ptr(ptrs), ptr(numel), ptr(group), ptr(chunks), nchunks, t, ptr(partial), ptr(hyper),
            ptr(step), ptr(total_norm), int(write_grads), stream())


def ema_update(desc, chunks, nchunks, decay):
    """ModelEMA.update over the (T,4) int64 table ``desc`` with the device scalar ``decay``."""
    _C.call("ub2_ema_update", ptr(desc), ptr(chunks), nchunks, ptr(decay), stream())


# --------------------------------------------------------------------------- ConvTranspose2d(k = 2, s = 2)
def pack_convt_weight(w, bias):
    """(Cin, Cout, 2, 2) fp32 -> (fwd pack (4*Cout, 1, Cin), dgrad pack (Cin, 1, 4*Cout), scale4, shift4)."""
    cin, cout = w.shape[0], w.shape[1]
    assert w.dtype == F32 and w.is_contiguous() and w.shape[2:] == (2, 2)
    fwd = torch.empty((4 * cout, 1, cin), device=w.device, dtype=BF16)
    dg = torch.empty((cin, 1, 4 * cout), device=w.device, dtype=BF16)
    ss = torch.empty((2, 4 * cout), device=w.device, dtype=F32)
    _C.call("ub2_pack_convt_weight", ptr(w), ptr(bias), ptr(fwd), ptr(dg), ptr(ss[0]), ptr(ss[1]), cin, cout, stream())
    return fwd, dg, ss[0], ss[1]


def shuffle2x2(t, cout, ho, wo):
    """t (N,h,w,4*Cout) -> (N,ho,wo,Cout): pixel shuffle of the transposed convolution + F.pad (zeros)."""
    n, h, w, c4, ld = _nhwc(t)
    assert c4 == 4 * cout
    out = empty_nhwc(n, ho, wo, cout, t.device)
    _C.call("ub2_shuffle2x2_fwd", ptr(t), ld, ptr(out), cout, n, h, w, cout, ho, wo, stream(), work=(0.0, _nbytes(t, out)))
    return out


def shuffle2x2_bwd(dout, h, w, dbias=None, want_bias=True):
    """Transpose of shuffle2x2: (N,ho,wo,Cout) -> dt (N,h,w,4*Cout); the bias gradient (sum of the gathered
    gradient per channel) is accumulated into ``dbias`` (fresh zeros by default)."""
    n, ho, wo, cout, ld = _nhwc(dout)
    dt = empty_nhwc(n, h, w, 4 * cout, dout.device)
    partials = None
    rows = 0
    if want_bias:
        rows = _rows("ub2_shuffle2x2_rows", n, h, w, cout, ho, wo)
        partials = torch.empty((rows, cout), device=dout.device, dtype=F64)
        if dbias is None:
            dbias = torch.zeros((cout,), device=dout.device, dtype=F32)
    _C.call("ub2_shuffle2x2_bwd", ptr(dout), ld, ptr(dt), 4 * cout, ptr(partials), rows, ptr(dbias if want_bias else None),
            n, h, w, cout, ho, wo, stream(), work=(0.0, _nbytes(dout, dt)))
    return dt, (dbias if want_bias else None)


def convt_wgrad_reduce(partial, cin, cout, grad, accumulate=False):
    """grad (Cin,Cout,2,2) fp32 = (or +=) sum over splits of partial (splits, Cin, 4*Cout)."""
    assert grad.dtype == F32 and grad.is_contiguous() and partial.is_contiguous()
    _C.call("ub2_convt_wgrad_reduce", ptr(partial), partial.shape[0], cin, cout, ptr(grad), int(accumulate), stream())
    return grad


def resize_planes(x, ho, wo):
    """fp32 (N,C,h,w) -> (N,C,ho,wo), bilinear, align_corners=True (the deep-supervision resize)."""
    assert x.dim() == 4 and x.dtype == F32 and x.is_contiguous()
    n, c, h, w = x.shape
    out = torch.empty((n, c, ho, wo), device=x.device, dtype=F32)
    _C.call("ub2_resize_planes_fwd", ptr(x), ptr(out), n * c, h, w, ho, wo, stream())
    return out


def resize_planes_bwd(dout, h, w):
    """Transpose of resize_planes: fp32 (N,C,ho,wo) -> (N,C,h,w)."""
    assert dout.dim() == 4 and dout.dtype == F32 and dout.is_contiguous()
    n, c, ho, wo = dout.shape
    din = torch.empty((n, c, h, w), device=dout.device, dtype=F32)
    _C.call("ub2_resize_planes_bwd", ptr(dout), ptr(din), n * c, h, w, ho, wo, stream())
    return din


# --------------------------------------------------------------------------- fp32 / TF32 mode
# fp32 NHWC activations and gradients (unet/fp32.py); reductions write the fp64 rows that bn_finalize,
# bn_bwd_finalize and gate_bwd_finalize above fold.
def conv_fwd_tf32(x0, x1, pack, cout, taps, scale=None, shift=None, relu=False, exact=False):
    """x0 / x1: NHWC fp32 (channel stride may exceed the channel count); ``pack``: (Cout, taps, Cin) fp32."""
    n, h, w, c0, ld0 = _nhwc32(x0)
    c1, ld1 = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1 = _nhwc32(x1)
    assert pack.is_contiguous() and pack.numel() == cout * taps * (c0 + c1)
    out = torch.empty((n, h, w, cout), device=x0.device, dtype=F32)
    _C.call("ub2_conv_fwd_tf32", ptr(x0), ld0, c0, ptr(x1), ld1, c1, ptr(pack), ptr(out), cout, n, h, w,
            cout, taps, ptr(scale), ptr(shift), int(relu), int(exact), stream(),
            work=(2.0 * n * h * w * cout * taps * (c0 + c1), _nbytes(x0, x1, pack, out)))
    return out


def f32_pack_weight(w):
    """OIHW fp32 -> the TF32 pack (Cout, taps, Cin)."""
    cout, cin, kh, kw = w.shape
    out = torch.empty((cout, kh * kw, cin), device=w.device, dtype=F32)
    _C.call("ub2_f32_pack_weight", ptr(w.contiguous()), ptr(out), cout, cin, kh * kw, stream())
    return out


def f32_pack_weight3(w, dgrad=False):
    """OIHW fp32 -> the 3xTF32 pack (rows, taps, 3*K) = per tap [w_hi | w_hi | w_lo]; ``dgrad``: rows = Cin,
    K = Cout, taps flipped (the data gradient is the same kernel)."""
    cout, cin, kh, kw = w.shape
    rows, k = (cin, cout) if dgrad else (cout, cin)
    out = torch.empty((rows, kh * kw, 3 * k), device=w.device, dtype=F32)
    _C.call("ub2_f32_pack_weight3", ptr(w.contiguous()), ptr(out), cout, cin, kh * kw, int(dgrad), stream())
    return out


def f32_split_tf32(x0, x1=None):
    """(N,H,W,C0 [+C1]) fp32 -> (N,H,W,2*(C0+C1)) = [hi(x0) | hi(x1) | lo(x0) | lo(x1)], two TF32 numbers per value."""
    n, h, w, c0, ld0 = _nhwc32(x0)
    c1, ld1 = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1 = _nhwc32(x1)
    out = torch.empty((n, h, w, 2 * (c0 + c1)), device=x0.device, dtype=F32)
    _C.call("ub2_f32_split_tf32", ptr(x0), ld0, c0, ptr(x1), ld1, c1, ptr(out), n * h * w, stream(),
            work=(0.0, _nbytes(x0, x1, out)))
    return out


def f32_split_bf16(x):
    """dense fp32 NHWC -> (hi, lo) bf16 NHWC with x = hi + lo to 2^-16 relative."""
    _nhwc32(x, dense=True)
    hi = torch.empty(x.shape, device=x.device, dtype=BF16)
    lo = torch.empty(x.shape, device=x.device, dtype=BF16)
    _C.call("ub2_f32_split_bf16", ptr(x), ptr(hi), ptr(lo), x.numel(), stream(), work=(0.0, _nbytes(x, hi, lo)))
    return hi, lo


def f32_conv_in(x, w, scale, shift):
    """Inference: first conv + folded BN + ReLU, x (N,Cin,H,W) fp32 NCHW -> (N,H,W,Cout) fp32."""
    assert x.dtype == F32 and x.is_contiguous()
    n, cin, h, wd = x.shape
    cout = w.shape[0]
    out = torch.empty((n, h, wd, cout), device=x.device, dtype=F32)
    _C.call("ub2_f32_conv_in", ptr(x), ptr(w.contiguous()), ptr(scale), ptr(shift), ptr(out), n, cin, h, wd, cout,
            stream())
    return out


def f32_conv_in_raw(x, w):
    """First conv without BatchNorm (training): x (N,Cin,H,W) fp32 NCHW -> y (N,H,W,Cout) fp32."""
    assert x.dtype == F32 and x.is_contiguous()
    n, cin, h, wd = x.shape
    cout = w.shape[0]
    y = torch.empty((n, h, wd, cout), device=x.device, dtype=F32)
    _C.call("ub2_f32_conv_in_raw", ptr(x), ptr(w.contiguous()), ptr(y), n, cin, h, wd, cout, stream())
    return y


def f32_conv_in_wgrad(x, dy, wshape):
    """Weight gradient (Cout,Cin,3,3) fp32 of f32_conv_in_raw from x NCHW and dy (N,H,W,Cout) fp32."""
    assert x.dtype == F32 and x.is_contiguous()
    _nhwc32(dy, dense=True)
    n, cin, h, wd = x.shape
    cout = wshape[0]
    rows = _rows("ub2_f32_channel_rows", n * h * wd, cout)
    part = torch.empty((rows, cin, 9, cout), device=x.device, dtype=F64)
    gw = torch.zeros(wshape, device=x.device, dtype=F32)
    _C.call("ub2_f32_conv_in_wgrad", ptr(x), ptr(dy), ptr(part), rows, ptr(gw), n, cin, h, wd, cout, stream())
    return gw


def f32_maxpool(a):
    """Inference: 2x2 max-pool of a dense NHWC fp32 tensor."""
    n, h, w, c, _ = _nhwc32(a, dense=True)
    out = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_maxpool", ptr(a), ptr(out), n, h, w, c, stream())
    return out


def f32_maxpool_idx(a):
    """2x2 max-pool of a dense NHWC fp32 tensor and the uint8 window position of each maximum."""
    n, h, w, c, _ = _nhwc32(a, dense=True)
    p = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=F32)
    idx = torch.empty((n, h // 2, w // 2, c), device=a.device, dtype=torch.uint8)
    _C.call("ub2_f32_maxpool_idx", ptr(a), ptr(p), ptr(idx), n, h, w, c, stream(), work=(0.0, _nbytes(a, p, idx)))
    return p, idx


def f32_maxpool_bwd(dP, idx, shape):
    """Route the pooled gradient to the saved window positions: the act_bwd apply pass with identity coefficients
    (dy = routed gradient) onto an (N,H,W,C) = ``shape`` fp32 tensor."""
    n, h, w, c = shape
    _nhwc32(dP, dense=True)
    dev = idx.device
    ones, zeros = torch.ones(c, device=dev), torch.zeros(c, device=dev)
    coef = torch.stack([ones, zeros, zeros])
    dummy_y = torch.zeros((n, h, w, c), device=dev, dtype=F32)
    dy = torch.empty((n, h, w, c), device=dev, dtype=F32)
    _C.call("ub2_f32_act_bwd_apply", None, 0, ptr(dP), ptr(idx), ptr(dummy_y), ptr(ones), ptr(zeros),
            ptr(coef), ptr(dy), n, h, w, c, 0, stream())
    return dy


def f32_upsample(a, out_h, out_w):
    """Inference: bilinear 2x (align_corners=True) of a dense NHWC fp32 tensor, centred in (out_h, out_w)."""
    n, h, w, c, _ = _nhwc32(a, dense=True)
    out = torch.empty((n, out_h, out_w, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_upsample", ptr(a), ptr(out), n, h, w, 2 * h, 2 * w, out_h, out_w, c, stream())
    return out


def f32_upsample_fwd(a, out_h, out_w, hu=None, wu=None):
    """bilinear (h,w) -> (hu,wu) (default 2x), centred in a zero (out_h,out_w) canvas (F.pad of layers.py:98-102)."""
    n, h, w, c, _ = _nhwc32(a, dense=True)
    hu, wu = (2 * h if hu is None else hu), (2 * w if wu is None else wu)
    out = torch.empty((n, out_h, out_w, c), device=a.device, dtype=F32)
    _C.call("ub2_f32_upsample_fwd", ptr(a), ptr(out), n, h, w, hu, wu, out_h, out_w, c, stream(),
            work=(0.0, _nbytes(a, out)))
    return out


def f32_upsample_bwd(dout, hin, win, hu, wu):
    n, ho, wo, c, ld = _nhwc32(dout)
    din = torch.empty((n, hin, win, c), device=dout.device, dtype=F32)
    _C.call("ub2_f32_upsample_bwd", ptr(dout), ld, ptr(din), n, hin, win, hu, wu, ho, wo, c, stream(),
            work=(0.0, _nbytes(dout, din)))
    return din


def f32_channel_stats(x):
    """(rows, 2, C) fp64 per-block sums / sums of squares over the pixels of an NHWC fp32 tensor."""
    n, h, w, c, ld = _nhwc32(x)
    rows = _rows("ub2_f32_channel_rows", n * h * w, c)
    part = torch.empty((rows, 2, c), device=x.device, dtype=F64)
    _C.call("ub2_f32_channel_stats", ptr(x), ld, n * h * w, c, ptr(part), rows, stream(), work=(0.0, _nbytes(x)))
    return part


def f32_scalar_stats(x):
    """(rows, 2, 1) fp64 per-block sum / sum of squares of a dense fp32 tensor."""
    assert x.dtype == F32 and x.is_contiguous()
    n = x.numel()
    rows = _rows("ub2_f32_scalar_rows", n)
    part = torch.empty((rows, 2, 1), device=x.device, dtype=F64)
    _C.call("ub2_f32_scalar_stats", ptr(x), n, ptr(part), rows, stream(), work=(0.0, _nbytes(x)))
    return part


def f32_affine_act(y, scale, shift, relu=True):
    """relu?(scale*y + shift) per channel of a dense NHWC fp32 tensor."""
    n, h, w, c, _ = _nhwc32(y, dense=True)
    out = torch.empty_like(y)
    _C.call("ub2_f32_affine_act", ptr(y), ptr(scale), ptr(shift), ptr(out), n * h * w, c, int(relu), stream(),
            work=(0.0, _nbytes(y, out)))
    return out


def f32_act_bwd(dA, dP, idx, y, scale, shift, mean, invstd, gamma, batch, relu=True, exchange=None):
    """BatchNorm (+ReLU, + max-pool routing) backward: (dy, dgamma, dbeta).  dA may be a channel slice; dP, y dense.
    ``exchange``: SyncBatchNorm (see ``synced_coef``)."""
    n, h, w, c, _ = _nhwc32(y, dense=True)
    ld_da = _nhwc32(dA)[4] if dA is not None else 0
    if dP is not None:
        _nhwc32(dP, dense=True)
    rows = _rows("ub2_f32_channel_rows", n * h * w, c)
    part = torch.empty((rows, 2, c), device=y.device, dtype=F64)
    _C.call("ub2_f32_act_bwd_reduce", ptr(dA), ld_da, ptr(dP), ptr(idx), ptr(y), ptr(scale), ptr(shift), ptr(part),
            rows, n, h, w, c, int(relu), stream(), work=(0.0, _nbytes(dA, dP, idx, y)))
    dgamma, dbeta, coef = bn_bwd_finalize(part, n * h * w, gamma, mean, invstd, frozen=not batch)
    if exchange is not None:
        coef = synced_coef(part, n * h * w, exchange, gamma, mean, invstd, frozen=not batch)
    dy = torch.empty_like(y)
    _C.call("ub2_f32_act_bwd_apply", ptr(dA), ld_da, ptr(dP), ptr(idx), ptr(y), ptr(scale), ptr(shift), ptr(coef),
            ptr(dy), n, h, w, c, int(relu), stream(), work=(0.0, _nbytes(dA, dP, idx, y, dy)))
    return dy, dgamma, dbeta


def f32_gate(q, xp, x, sg, hg, sx, hx, wpsi, spsi, hpsi):
    """Inference: out = x * sigmoid(BN_psi(w_psi . relu(BN_g(up q) + BN_x(xp)))), q at the gating resolution."""
    _, hin, win, ci, _ = _nhwc32(q, dense=True)
    _nhwc32(xp, dense=True)
    n, h, w, cx, _ = _nhwc32(x, dense=True)
    out = torch.empty_like(x)
    _C.call("ub2_f32_gate", ptr(q), ptr(xp), ptr(x), ptr(sg), ptr(hg), ptr(sx), ptr(hx), ptr(wpsi), ptr(spsi),
            ptr(hpsi), ptr(out), n, hin, win, h, w, ci, cx, stream())
    return out


def f32_gate_psi(u, xp, sg, hg, sx, hx, wpsi):
    """psi_raw (N,H,W) = w_psi . relu(BN_g(u) + BN_x(xp)), u = up(q) and xp dense NHWC fp32."""
    n, h, w, ci, _ = _nhwc32(u, dense=True)
    _nhwc32(xp, dense=True)
    psi = torch.empty((n, h, w), device=u.device, dtype=F32)
    _C.call("ub2_f32_gate_psi", ptr(u), ptr(xp), ptr(sg), ptr(hg), ptr(sx), ptr(hx), ptr(wpsi), ptr(psi),
            n * h * w, ci, stream(), work=(0.0, _nbytes(u, xp, psi)))
    return psi


def f32_gate_apply(psi, spsi, hpsi, x):
    """a = sigmoid(BN_psi(psi_raw)), out = x * a: returns (out, a)."""
    n, h, w, cx, _ = _nhwc32(x, dense=True)
    assert psi.is_contiguous()
    out = torch.empty_like(x)
    a = torch.empty((n, h, w), device=x.device, dtype=F32)
    _C.call("ub2_f32_gate_apply", ptr(psi), ptr(spsi), ptr(hpsi), ptr(x), ptr(out), ptr(a), n * h * w, cx, stream(),
            work=(0.0, _nbytes(psi, x, out, a)))
    return out, a


def f32_gate_bwd_a(dout, x, a, psi):
    """(dx, dpsin, (rows, 2, 1) partials); dout may be a channel slice."""
    ld_do = _nhwc32(dout)[4]
    n, h, w, cx, _ = _nhwc32(x, dense=True)
    assert a.is_contiguous() and psi.is_contiguous()
    rows = _rows("ub2_f32_gate_rows", n * h * w)
    dx = torch.empty_like(x)
    dpsin = torch.empty((n, h, w), device=x.device, dtype=F32)
    part = torch.empty((rows, 2, 1), device=x.device, dtype=F64)
    _C.call("ub2_f32_gate_bwd_a", ptr(dout), ld_do, ptr(x), ptr(a), ptr(psi), ptr(dx), ptr(dpsin), ptr(part), rows,
            n * h * w, cx, stream(), work=(0.0, _nbytes(dout, x, a, psi, dx, dpsin)))
    return dx, dpsin, part


def f32_gate_bwd_s(dpsin, psi, coef_psi, u, xp, sg, hg, sx, hx, wpsi):
    """(ds, (rows, 4, Ci) partials)."""
    n, h, w, ci, _ = _nhwc32(u, dense=True)
    _nhwc32(xp, dense=True)
    assert dpsin.is_contiguous() and psi.is_contiguous()
    rows = _rows("ub2_f32_gate_rows", n * h * w)
    ds = torch.empty_like(xp)
    part = torch.empty((rows, 4, ci), device=u.device, dtype=F64)
    _C.call("ub2_f32_gate_bwd_s", ptr(dpsin), ptr(psi), ptr(coef_psi), ptr(u), ptr(xp), ptr(sg), ptr(hg), ptr(sx),
            ptr(hx), ptr(wpsi), ptr(ds), ptr(part), rows, n * h * w, ci, stream(),
            work=(0.0, _nbytes(dpsin, psi, u, xp, ds)))
    return ds, part


def f32_gate_bwd_xg(ds, xp, u, coef):
    """(dxp, du): the gradients of BN_x(xp) and BN_g(u)."""
    n, h, w, ci, _ = _nhwc32(u, dense=True)
    _nhwc32(ds, dense=True)
    _nhwc32(xp, dense=True)
    dxp = torch.empty_like(xp)
    du = torch.empty_like(xp)
    _C.call("ub2_f32_gate_bwd_xg", ptr(ds), ptr(xp), ptr(u), ptr(coef), ptr(dxp), ptr(du), n * h * w, ci, stream(),
            work=(0.0, _nbytes(ds, xp, u, dxp, du)))
    return dxp, du


def f32_outc(a, w, bias, claim_work=True):
    """OutConv: dense NHWC fp32 a, w (K,C,1,1) -> fp32 NCHW logits.  ``claim_work=False``: no roofline claim (the
    inference path)."""
    n, h, wd, c, _ = _nhwc32(a, dense=True)
    k = w.shape[0]
    logits = torch.empty((n, k, h, wd), device=a.device, dtype=F32)
    _C.call("ub2_f32_outc", ptr(a), ptr(w.reshape(k, -1).contiguous()), ptr(bias), ptr(logits), n, h, wd, c, k,
            stream(), work=(0.0, _nbytes(a, logits)) if claim_work else None)
    return logits


def f32_outc_bwd(dlogits, a, w, need_da=True):
    """(da or None, dw (K,C,1,1), db (K,)) from dense fp32 NCHW dlogits."""
    n, h, wd, c, _ = _nhwc32(a, dense=True)
    assert dlogits.dtype == F32 and dlogits.is_contiguous()
    k = w.shape[0]
    rows = _rows("ub2_f32_outc_rows", n, h, wd)
    part = torch.empty((rows, k * c + k), device=a.device, dtype=F64)
    da = torch.empty_like(a) if need_da else None
    dw = torch.zeros(w.shape, device=a.device, dtype=F32)
    db = torch.zeros((k,), device=a.device, dtype=F32)
    _C.call("ub2_f32_outc_bwd", ptr(dlogits), ptr(a), ptr(w.reshape(k, -1).contiguous()), ptr(da), ptr(part), rows,
            ptr(dw), ptr(db), n, h, wd, c, k, stream(), work=(0.0, _nbytes(dlogits, a, da)))
    return da, dw, db


def f32_pack_convt_weight(weight, bias):
    """(Cin, Cout, 2, 2) fp32 parameter -> (the exact 1x1 weight (4*Cout, Cin, 1, 1) OIHW, row (i*2+j)*Cout + co;
    scale4 = ones, shift4 = bias tiled four times)."""
    cin, cout = weight.shape[0], weight.shape[1]
    w1 = torch.empty((4 * cout, cin, 1, 1), device=weight.device, dtype=F32)
    ss = torch.empty((2, 4 * cout), device=weight.device, dtype=F32)
    _C.call("ub2_f32_pack_convt_weight", ptr(weight.contiguous()), ptr(bias), ptr(w1), ptr(ss[0]), ptr(ss[1]), cin,
            cout, stream())
    return w1, ss[0], ss[1]


def f32_shuffle2x2(t, cout, out_h, out_w):
    """t (N,h,w,4*Cout) fp32 -> (N,out_h,out_w,Cout): pixel shuffle of the transposed convolution + F.pad (zeros)."""
    n, h, w, c4, ld = _nhwc32(t)
    assert c4 == 4 * cout
    out = torch.empty((n, out_h, out_w, cout), device=t.device, dtype=F32)
    _C.call("ub2_f32_shuffle2x2_fwd", ptr(t), ld, ptr(out), cout, n, h, w, cout, out_h, out_w, stream(),
            work=(0.0, _nbytes(t, out)))
    return out


def f32_shuffle2x2_bwd(dout, h, w, want_bias=True):
    """Transpose of f32_shuffle2x2: dout (N,Ho,Wo,Cout), channel stride may exceed Cout -> (dt (N,h,w,4*Cout),
    bias gradient (Cout,) or None)."""
    n, ho, wo, cout, ld = _nhwc32(dout)
    dt = torch.empty((n, h, w, 4 * cout), device=dout.device, dtype=F32)
    partials = db = None
    rows = 0
    if want_bias:
        rows = _rows("ub2_f32_shuffle2x2_rows", n, h, w, cout, ho, wo)
        partials = torch.empty((rows, cout), device=dout.device, dtype=F64)
        db = torch.zeros((cout,), device=dout.device, dtype=F32)
    _C.call("ub2_f32_shuffle2x2_bwd", ptr(dout), ld, ptr(dt), 4 * cout, ptr(partials), rows, ptr(db), n, h, w, cout,
            ho, wo, stream(), work=(0.0, _nbytes(dout, dt)))
    return dt, db
