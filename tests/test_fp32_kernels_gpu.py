"""fp32 / TF32 mode one entry point at a time: every C entry point of csrc/fp32_train.cu and csrc/fp32_eval.cu, and
the four finalize kernels it shares with the bf16 path, called through ``_C.call`` on caller-built tensors and
compared with a float64 reference of the same formula on the same fp32 operands.

Gates are derived from the arithmetic of each kernel, with u = 2^-24 (half an fp32 ulp, the bound of one
round-to-nearest step relative to its result):

* copies, packs, splits and max-pool values / indices: bit-exact;
* element-wise kernels: ``|got - ref| <= 2 u * steps * sum|terms|``, one fp32 ulp per rounding step of the kernel,
  with ``sum|terms|`` the magnitudes that step adds, computed in float64 from the same operands;
* reductions: the same bound with ``steps`` = the sequential fp32 additions one thread performs (the rows it folds
  in fp64 add nothing visible), read off the launch geometry — never relative to the sum's own value, which
  nearly cancels for gradients such as dbeta or dwpsi;
* the eval kernels that round their output to TF32 (f32_conv_in, f32_upsample, f32_gate): one TF32 ulp (2^-10
  relative) on top;
* the 3xTF32 convolution: rel-L2 <= 1e-5 (its error is ~2^-21; a single pass or a lost lo term sits at >= 3e-4),
  the bf16 hi/lo weight gradient: rel-L2 <= 1e-4 (~2^-16; a dropped cross term costs ~2^-9).

Every launch writes into the middle of a NaN-filled buffer whose bands are checked afterwards, every reduction runs
twice and must repeat bit for bit, and workspace rows come from the matching ``*_rows`` query.

Not covered on purpose: NaN inputs.  The ReLU and max-pool kernels use ``fmaxf`` and comparisons that drop a NaN
(``fmaxf(NaN, 0) = 0``; a NaN never wins a window), where ATen's ``relu`` and ``max_pool2d`` propagate it.

The host-side argument checks (no ``gpu`` mark) run every entry point in a child process without a device: bad
arguments must come back as their negative UB2_ERR code, valid ones — including every NULL the modules pass — as a
CUDA error, which proves they got past the checks."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from parity_log import record

GPU = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24
F32, F64 = torch.float32, torch.float64
BAND = 256            # guard band, in elements (a multiple of 4: 16-byte alignment is kept)
KFT = 256             # threads per block of the fp32 kernels


# =============================================================================================== helpers
def _C():
    from unet import _C
    return _C


_LIVE = []      # the tensors of the call being assembled: a temporary passed as _p(t.cuda()) must outlive the launch


def _p(t):
    _LIVE.append(t)
    return _C().ptr(t)


def _s():
    return _C().stream()


def _call(name, *args):
    _C().call(name, *args)
    _LIVE.clear()      # the caching allocator reuses memory in stream order, after the launch


def _rows(name, *args):
    from unet import kernels as K
    return K._rows(name, *args)


class Guarded:
    """A tensor in the middle of a buffer filled with NaN (floats) or 0xA5 (bytes); ``ok()`` checks both bands."""

    def __init__(self, shape, dtype=F32, fill=None):
        n = int(np.prod(shape))
        self.n = n
        if dtype == torch.uint8:
            self.buf = torch.full((2 * BAND + n,), 0xA5, device="cuda", dtype=dtype)
        else:
            self.buf = torch.full((2 * BAND + n,), float("nan"), device="cuda", dtype=dtype)
        self.t = self.buf[BAND:BAND + n].view(shape)
        if fill is not None:
            self.t.copy_(fill)
        self.ref = self.buf.clone()

    def ok(self):
        torch.cuda.synchronize()
        ints = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[self.buf.element_size()]
        a, b = self.buf.view(ints), self.ref.view(ints)
        return torch.equal(a[:BAND], b[:BAND]) and torch.equal(a[BAND + self.n:], b[BAND + self.n:])


def _within(got, ref, terms, steps, what, tf32=False):
    """|got - ref| <= 2u * steps * terms (+ steps subnormal spacings), + one TF32 ulp (2^-10 |ref|) for outputs rounded
    to TF32; returns the worst error in units of 2u * terms."""
    got = got.detach().double().cpu()
    ref = torch.as_tensor(ref).detach().double().cpu()
    terms = torch.as_tensor(terms).detach().double().cpu()
    err = (got - ref).abs()
    tol = 2 * U * steps * terms + steps * 2.0 ** -149 + (2.0 ** -10 * ref.abs() if tf32 else 0)
    bad = ~(err <= tol)
    assert not bool(bad.any()), (what, int(bad.sum()), float(err[bad].max()), float(tol[bad][err[bad].argmax()]),
                                 float(ref[bad][err[bad].argmax()]))
    scale = 2 * U * terms
    ratio = torch.where(scale > 0, err / scale.clamp_min(1e-300), torch.zeros_like(err))
    return float(ratio.max()) if ratio.numel() else 0.0


def _rel_l2(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return float((got - ref).norm() / ref.norm().clamp_min(1e-300))


def _tf32(x):
    """round to nearest TF32 (10-bit mantissa), ties away from zero like cvt.rna"""
    i = x.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(F32)


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == F32 else t.contiguous().view(torch.int16)


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _randn(shape, g, scale=1.0, shift=0.0):
    return (torch.randn(shape, generator=g, dtype=F64) * scale + shift).float()


def _lanes(C):
    return max(KFT // (C // 4), 1)


def _per_thread(items, workers):
    return -(-items // workers)


def _folded(part):
    """Rows (rows, S, C) fp64 -> (S, C) in float64 (the order does not matter at fp64 precision)."""
    return part.double().cpu().sum(0)


# =============================================================================================== host checks
CHILD = r'''
import ctypes, sys
sys.path.insert(0, sys.argv[1] + "/unet-segment-pytorch_b200")
from unet import _C
lib = _C.lib()
P = 1 << 20                      # a 16-byte-aligned fake device address: the calls below must never use it
Q = P + 4                        # 4-byte aligned only
# the fp32 entry points under test, with their parameters as include/unetb200.h declares them
SIG = {name: _C.SIGNATURES[name] for name in """
ub2_f32_channel_stats ub2_f32_scalar_stats ub2_f32_affine_act ub2_f32_maxpool_idx ub2_f32_act_bwd_reduce
ub2_f32_act_bwd_apply ub2_f32_upsample_bwd ub2_f32_gate_psi ub2_f32_gate_apply ub2_f32_gate_bwd_a
ub2_f32_gate_bwd_s ub2_f32_gate_bwd_xg ub2_f32_outc_bwd ub2_f32_conv_in_raw ub2_f32_conv_in_wgrad
ub2_f32_split_bf16 ub2_f32_split_tf32 ub2_f32_pack_weight3 ub2_f32_upsample_fwd ub2_f32_pack_weight
ub2_f32_conv_in ub2_f32_maxpool ub2_f32_upsample ub2_f32_gate ub2_f32_outc""".split()}
N, H, W, C = 2, 8, 8, 16
pix = N * H * W
chan = lib.ub2_f32_channel_rows(pix, C)
gater = lib.ub2_f32_gate_rows(pix)
outcr = lib.ub2_f32_outc_rows(N, H, W)
scal = lib.ub2_f32_scalar_rows(pix)
wg4 = lib.ub2_f32_channel_rows(pix, 4)
assert min(chan, gater, outcr, scal, wg4) > 0
# every pointer argument defaults to P, the stream to NULL
BASE = {
 "ub2_f32_channel_stats": dict(ld=C, pixels=pix, C=C, rows=chan),
 "ub2_f32_scalar_stats": dict(n=pix, rows=scal),
 "ub2_f32_affine_act": dict(pixels=pix, C=C, relu=1),
 "ub2_f32_maxpool_idx": dict(N=N, H=H, W=W, C=C),
 "ub2_f32_act_bwd_reduce": dict(ld_da=C, rows=chan, N=N, H=H, W=W, C=C, relu=1),
 "ub2_f32_act_bwd_apply": dict(ld_da=C, N=N, H=H, W=W, C=C, relu=1),
 "ub2_f32_upsample_bwd": dict(ld_dout=C, N=N, hin=4, win=4, hu=8, wu=8, Ho=H, Wo=W, C=C),
 "ub2_f32_gate_psi": dict(pixels=pix, Ci=C),
 "ub2_f32_gate_apply": dict(pixels=pix, Cx=C),
 "ub2_f32_gate_bwd_a": dict(ld_do=C, rows=gater, pixels=pix, Cx=C),
 "ub2_f32_gate_bwd_s": dict(rows=gater, pixels=pix, Ci=C),
 "ub2_f32_gate_bwd_xg": dict(pixels=pix, Ci=C),
 "ub2_f32_outc_bwd": dict(rows=outcr, N=N, H=H, W=W, C=C, K=2),
 "ub2_f32_conv_in_raw": dict(N=N, Cin=1, H=H, W=W, Cout=C),
 "ub2_f32_conv_in_wgrad": dict(rows=chan, N=N, Cin=1, H=H, W=W, Cout=C),
 "ub2_f32_split_bf16": dict(n=pix * C),
 "ub2_f32_split_tf32": dict(ld0=C, C0=C, ld1=C, C1=C, pixels=pix),
 "ub2_f32_pack_weight3": dict(Cout=C, Cin=C, taps=9, dgrad=0),
 "ub2_f32_upsample_fwd": dict(N=N, hin=4, win=4, hu=8, wu=8, Ho=H, Wo=W, C=C),
 "ub2_f32_pack_weight": dict(Cout=C, Cin=C, taps=9),
 "ub2_f32_conv_in": dict(N=N, Cin=1, H=H, W=W, Cout=C),
 "ub2_f32_maxpool": dict(N=N, H=H, W=W, C=C),
 "ub2_f32_upsample": dict(N=N, hin=4, win=4, hu=8, wu=8, Ho=H, Wo=W, C=C),
 "ub2_f32_gate": dict(N=N, hin=4, win=4, H=H, W=W, Ci=C, Cx=2 * C),
 "ub2_f32_outc": dict(N=N, H=H, W=W, C=C, K=2),
}
def call(name, **kw):
    vals = []
    assert set(kw) <= {a for a, _ in SIG[name]}, (name, kw)
    for a, t in SIG[name]:
        if a == "stream":
            vals.append(None)
        elif a in kw:
            vals.append(kw[a])
        elif t is ctypes.c_void_p:
            vals.append(P)
        else:
            vals.append(BASE[name][a])
    return getattr(lib, name)(*vals)
S, A, WS = -1, -2, -3
BAD = [
 # the cases that reached the device before these checks
 ("ub2_f32_upsample", dict(hin=0), S), ("ub2_f32_upsample", dict(hu=-2, Ho=-2), S), ("ub2_f32_upsample", dict(src=None), S),
 ("ub2_f32_gate", dict(hin=0), S), ("ub2_f32_gate", dict(H=0), S), ("ub2_f32_gate", dict(Ci=0), S), ("ub2_f32_gate", dict(q=None), S),
 ("ub2_f32_conv_in", dict(H=-1), S), ("ub2_f32_conv_in", dict(Cout=0), S), ("ub2_f32_conv_in", dict(Cout=-4), S),
 ("ub2_f32_maxpool", dict(C=0), S), ("ub2_f32_maxpool", dict(C=-4), S),
 ("ub2_f32_outc", dict(H=0), S), ("ub2_f32_outc", dict(C=0), S), ("ub2_f32_outc", dict(C=-4), S),
 ("ub2_f32_upsample_bwd", dict(hu=0), S), ("ub2_f32_maxpool_idx", dict(idx=None), S),
 ("ub2_f32_act_bwd_apply", dict(dA=None, idx=None), S),
 ("ub2_f32_channel_stats", dict(ld=8), S), ("ub2_f32_split_tf32", dict(ld0=8), S), ("ub2_f32_split_tf32", dict(ld1=8), S),
 ("ub2_f32_act_bwd_reduce", dict(ld_da=8), S), ("ub2_f32_act_bwd_apply", dict(ld_da=8), S),
 ("ub2_f32_gate_bwd_a", dict(ld_do=8), S), ("ub2_f32_upsample_bwd", dict(ld_dout=8), S),
 # counts
 ("ub2_f32_channel_stats", dict(pixels=0), S), ("ub2_f32_channel_stats", dict(C=6, ld=8), S),
 ("ub2_f32_channel_stats", dict(C=1028, ld=1028), S), ("ub2_f32_scalar_stats", dict(n=0), S),
 ("ub2_f32_affine_act", dict(pixels=0), S), ("ub2_f32_affine_act", dict(C=0), S), ("ub2_f32_affine_act", dict(C=6), S),
 ("ub2_f32_maxpool_idx", dict(N=0), S), ("ub2_f32_maxpool_idx", dict(H=1), S), ("ub2_f32_maxpool_idx", dict(W=1), S),
 ("ub2_f32_maxpool_idx", dict(C=0), S),
 ("ub2_f32_act_bwd_reduce", dict(N=0), S), ("ub2_f32_act_bwd_reduce", dict(H=0), S), ("ub2_f32_act_bwd_reduce", dict(C=0), S),
 ("ub2_f32_act_bwd_apply", dict(W=0), S), ("ub2_f32_act_bwd_apply", dict(C=-4), S),
 ("ub2_f32_upsample_bwd", dict(N=0), S), ("ub2_f32_upsample_bwd", dict(hin=0), S), ("ub2_f32_upsample_bwd", dict(win=-1), S),
 ("ub2_f32_upsample_bwd", dict(wu=0), S), ("ub2_f32_upsample_bwd", dict(Ho=7), S), ("ub2_f32_upsample_bwd", dict(Wo=7), S),
 ("ub2_f32_upsample_bwd", dict(hu=-2, Ho=-2), S), ("ub2_f32_upsample_bwd", dict(C=0), S),
 ("ub2_f32_upsample_fwd", dict(hin=0), S), ("ub2_f32_upsample_fwd", dict(win=0), S), ("ub2_f32_upsample_fwd", dict(hu=0), S),
 ("ub2_f32_upsample_fwd", dict(wu=-8, Wo=-8), S), ("ub2_f32_upsample_fwd", dict(Ho=4), S), ("ub2_f32_upsample_fwd", dict(N=0), S),
 ("ub2_f32_upsample", dict(win=0), S), ("ub2_f32_upsample", dict(wu=0), S), ("ub2_f32_upsample", dict(Wo=4), S),
 ("ub2_f32_upsample", dict(C=0), S),
 ("ub2_f32_gate_psi", dict(pixels=0), S), ("ub2_f32_gate_psi", dict(Ci=0), S), ("ub2_f32_gate_psi", dict(Ci=6), S),
 ("ub2_f32_gate_apply", dict(pixels=0), S), ("ub2_f32_gate_apply", dict(Cx=0), S),
 ("ub2_f32_gate_bwd_a", dict(Cx=0, ld_do=0), S), ("ub2_f32_gate_bwd_a", dict(pixels=0), S),
 ("ub2_f32_gate_bwd_s", dict(Ci=0), S), ("ub2_f32_gate_bwd_s", dict(Ci=516), S), ("ub2_f32_gate_bwd_s", dict(pixels=0), S),
 ("ub2_f32_gate_bwd_xg", dict(Ci=0), S), ("ub2_f32_gate_bwd_xg", dict(pixels=0), S),
 ("ub2_f32_outc_bwd", dict(K=0), S), ("ub2_f32_outc_bwd", dict(K=9), S), ("ub2_f32_outc_bwd", dict(C=0), S),
 ("ub2_f32_outc_bwd", dict(N=0), S), ("ub2_f32_outc_bwd", dict(H=0, rows=outcr), S),
 ("ub2_f32_outc_bwd", dict(C=192, K=8), S),
 ("ub2_f32_conv_in_raw", dict(N=0), S), ("ub2_f32_conv_in_raw", dict(Cin=0), S), ("ub2_f32_conv_in_raw", dict(W=0), S),
 ("ub2_f32_conv_in_raw", dict(Cout=6), S),
 ("ub2_f32_conv_in_wgrad", dict(Cin=0), S), ("ub2_f32_conv_in_wgrad", dict(Cout=1028), S), ("ub2_f32_conv_in_wgrad", dict(H=0), S),
 ("ub2_f32_split_bf16", dict(n=0), S), ("ub2_f32_split_bf16", dict(n=6), S),
 ("ub2_f32_split_tf32", dict(C0=0), S), ("ub2_f32_split_tf32", dict(C1=-4), S), ("ub2_f32_split_tf32", dict(C1=6, ld1=8), S),
 ("ub2_f32_split_tf32", dict(pixels=0), S),
 ("ub2_f32_pack_weight3", dict(Cout=0), S), ("ub2_f32_pack_weight3", dict(Cin=0), S), ("ub2_f32_pack_weight3", dict(taps=0), S),
 ("ub2_f32_pack_weight", dict(taps=4), S), ("ub2_f32_pack_weight", dict(Cin=0), S),
 ("ub2_f32_conv_in", dict(N=0), S), ("ub2_f32_conv_in", dict(Cin=0), S), ("ub2_f32_conv_in", dict(W=0), S),
 ("ub2_f32_maxpool", dict(N=0), S), ("ub2_f32_maxpool", dict(H=1), S),
 ("ub2_f32_gate", dict(N=0), S), ("ub2_f32_gate", dict(win=0), S), ("ub2_f32_gate", dict(W=0), S), ("ub2_f32_gate", dict(Cx=0), S),
 ("ub2_f32_gate", dict(Ci=6), S),
 ("ub2_f32_outc", dict(N=0), S), ("ub2_f32_outc", dict(W=0), S), ("ub2_f32_outc", dict(K=0), S), ("ub2_f32_outc", dict(K=9), S),
 # gradient sources
 ("ub2_f32_act_bwd_reduce", dict(dA=None, dP=None), S), ("ub2_f32_act_bwd_apply", dict(dA=None, dP=None), S),
 ("ub2_f32_act_bwd_reduce", dict(idx=None), S), ("ub2_f32_act_bwd_apply", dict(idx=None), S),
 ("ub2_f32_act_bwd_reduce", dict(dA=None, idx=None), S),
 ("ub2_f32_split_tf32", dict(x1=None), S),
 # strides and alignment
 ("ub2_f32_channel_stats", dict(ld=18), A), ("ub2_f32_act_bwd_reduce", dict(ld_da=18), A), ("ub2_f32_act_bwd_apply", dict(ld_da=18), A),
 ("ub2_f32_upsample_bwd", dict(ld_dout=18), A), ("ub2_f32_gate_bwd_a", dict(ld_do=18), A), ("ub2_f32_split_tf32", dict(ld0=18), A),
 ("ub2_f32_split_tf32", dict(ld1=18), A),
 ("ub2_f32_channel_stats", dict(x=Q), A), ("ub2_f32_affine_act", dict(y=Q), A), ("ub2_f32_affine_act", dict(scale=Q), A),
 ("ub2_f32_affine_act", dict(out=Q), A), ("ub2_f32_maxpool_idx", dict(a=Q), A), ("ub2_f32_maxpool_idx", dict(idx=P + 2), A),
 ("ub2_f32_act_bwd_reduce", dict(dP=Q), A), ("ub2_f32_act_bwd_reduce", dict(partials=Q), A), ("ub2_f32_act_bwd_apply", dict(dy=Q), A),
 ("ub2_f32_act_bwd_apply", dict(coef=Q), A), ("ub2_f32_upsample_bwd", dict(din=Q), A), ("ub2_f32_gate_psi", dict(u=Q), A),
 ("ub2_f32_gate_psi", dict(wpsi=Q), A), ("ub2_f32_gate_apply", dict(x=Q), A), ("ub2_f32_gate_bwd_a", dict(dout=Q), A),
 ("ub2_f32_gate_bwd_s", dict(ds=Q), A), ("ub2_f32_gate_bwd_xg", dict(coef=Q), A), ("ub2_f32_outc_bwd", dict(a=Q), A),
 ("ub2_f32_outc_bwd", dict(da=Q), A), ("ub2_f32_conv_in_raw", dict(out=Q), A), ("ub2_f32_conv_in_wgrad", dict(dy=Q), A),
 ("ub2_f32_split_bf16", dict(x=Q), A), ("ub2_f32_split_tf32", dict(x1=Q), A), ("ub2_f32_split_tf32", dict(out=Q), A),
 ("ub2_f32_upsample_fwd", dict(src=Q), A), ("ub2_f32_conv_in", dict(out=Q), A), ("ub2_f32_maxpool", dict(out=Q), A),
 ("ub2_f32_upsample", dict(out=Q), A), ("ub2_f32_gate", dict(q=Q), A), ("ub2_f32_gate", dict(x=Q), A), ("ub2_f32_outc", dict(a=Q), A),
 # workspace rows
 ("ub2_f32_channel_stats", dict(rows=chan + 1), WS), ("ub2_f32_scalar_stats", dict(rows=scal - 1), WS),
 ("ub2_f32_act_bwd_reduce", dict(rows=chan + 1), WS), ("ub2_f32_gate_bwd_a", dict(rows=gater + 1), WS),
 ("ub2_f32_gate_bwd_s", dict(rows=gater - 1), WS), ("ub2_f32_outc_bwd", dict(rows=outcr + 1), WS),
 ("ub2_f32_conv_in_wgrad", dict(rows=chan + 1), WS),
]
# a NULL for every pointer the kernel dereferences unconditionally
OPTIONAL = {"ub2_f32_act_bwd_reduce": {"dA", "dP"}, "ub2_f32_act_bwd_apply": {"dA", "dP", "scale", "shift"},
            "ub2_f32_split_tf32": {"x1"}, "ub2_f32_gate_apply": {"a_out"}, "ub2_f32_outc_bwd": {"da", "dw", "db"},
            "ub2_f32_outc": {"bias"}}
for name, args in SIG.items():
    for a, t in args:
        if t is ctypes.c_void_p and a != "stream" and a not in OPTIONAL.get(name, ()):
            BAD.append((name, {a: None}, S))
BAD.append(("ub2_f32_act_bwd_apply", dict(scale=None), S))       # relu = 1 reads scale and shift
BAD.append(("ub2_f32_act_bwd_apply", dict(shift=None), S))
GOOD = [(name, {}) for name in SIG] + [
 # every NULL the modules pass
 ("ub2_f32_act_bwd_reduce", dict(dA=None, ld_da=0)), ("ub2_f32_act_bwd_reduce", dict(dP=None, idx=None)),
 ("ub2_f32_act_bwd_reduce", dict(dP=None)), ("ub2_f32_act_bwd_apply", dict(dA=None, ld_da=0)),
 ("ub2_f32_act_bwd_apply", dict(dP=None, idx=None)),
 ("ub2_f32_act_bwd_apply", dict(dA=None, ld_da=0, relu=0, scale=None, shift=None)),
 ("ub2_f32_split_tf32", dict(x1=None, ld1=0, C1=0)), ("ub2_f32_gate_apply", dict(a_out=None)),
 ("ub2_f32_outc_bwd", dict(da=None)), ("ub2_f32_outc_bwd", dict(dw=None, db=None)), ("ub2_f32_outc_bwd", dict(da=None, dw=None, db=None)),
 ("ub2_f32_outc", dict(bias=None)),
 # edges that are valid
 ("ub2_f32_channel_stats", dict(ld=24)), ("ub2_f32_channel_stats", dict(C=1024, ld=1024, rows=lib.ub2_f32_channel_rows(pix, 1024))),
 ("ub2_f32_act_bwd_reduce", dict(ld_da=24)), ("ub2_f32_upsample_bwd", dict(ld_dout=20)), ("ub2_f32_upsample_bwd", dict(hin=1, hu=1, Ho=1)),
 ("ub2_f32_upsample_bwd", dict(Ho=11, Wo=13)), ("ub2_f32_upsample_fwd", dict(hin=7, win=7, hu=16, wu=16, Ho=16, Wo=16)),
 ("ub2_f32_gate_bwd_a", dict(ld_do=20)), ("ub2_f32_gate_bwd_s", dict(Ci=388)), ("ub2_f32_gate_bwd_s", dict(Ci=512)),
 ("ub2_f32_outc_bwd", dict(C=188, K=8)), ("ub2_f32_outc_bwd", dict(K=1)),
 ("ub2_f32_conv_in_raw", dict(Cin=7, Cout=1024)), ("ub2_f32_conv_in_wgrad", dict(Cin=7, Cout=4, rows=wg4)),
 ("ub2_f32_split_tf32", dict(ld0=24, ld1=20)), ("ub2_f32_pack_weight3", dict(taps=1, dgrad=1)),
 ("ub2_f32_maxpool_idx", dict(H=3, W=5)), ("ub2_f32_gate", dict(Cx=12)), ("ub2_f32_outc", dict(K=8)),
]
for name, kw, want in BAD:
    rc = call(name, **kw)
    print(name, sorted(kw.items()), rc, want, "OK" if rc == want else "WRONG", flush=True)
for name, kw in GOOD:
    rc = call(name, **kw)
    print(name, "valid", sorted(kw.items()), rc, "positive", "OK" if rc > 0 else "WRONG", flush=True)
print("DONE", len(BAD), len(GOOD), flush=True)
'''


def test_fp32_entry_points_check_arguments_on_the_host():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")      # argument checks only, also on a GPU box
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, env=env)
    lines = r.stdout.strip().splitlines()
    assert r.returncode == 0 and lines and lines[-1].startswith("DONE"), (r.returncode, lines[-3:], r.stderr[-2000:])
    wrong = [l for l in lines if l.endswith("WRONG")]
    assert not wrong, wrong
    _, nbad, ngood = lines[-1].split()
    assert sum(l.endswith("OK") for l in lines) == int(nbad) + int(ngood) >= 300


# =============================================================================================== BatchNorm statistics
def _stats_case(pixels, C, ld, seed, far_mean=False):
    g = _gen(seed)
    full = _randn((pixels, ld), g)
    if far_mean:
        full[:, 1] = _randn((pixels,), g, 1.0, 100.0)      # mean = 100 std: the one-pass variance's hard case
    x = Guarded((pixels, ld), fill=full.cuda()).t
    rows = _rows("ub2_f32_channel_rows", pixels, C)
    parts = []
    for _ in range(2):
        pg = Guarded((rows, 2, C), F64)
        _call("ub2_f32_channel_stats", _p(x), ld, pixels, C, _p(pg.t), rows, _s())
        assert pg.ok(), ("partials bands", pixels, C, ld)
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]), ("not repeatable", pixels, C)
    xs = full[:, :C].double()
    got = _folded(parts[0])
    k = _per_thread(pixels, _lanes(C) * rows)              # sequential fp32 adds per thread
    e0 = _within(got[0], xs.sum(0), xs.abs().sum(0), k, ("sum", pixels, C))
    e1 = _within(got[1], (xs * xs).sum(0), (xs * xs).sum(0), 2 * k, ("sumsq", pixels, C))
    return x, parts[0], xs, k, max(e0, e1)


@GPU
@pytest.mark.parametrize("C", [4, 12, 20, 64, 100, 1024])
def test_channel_stats_and_bn_finalize(C):
    """f32_channel_stats over pixels fewer than the lanes of one block, a count that is not a multiple of the grid and
    a channel stride above C; then bn_finalize (scale, shift, mean, invstd, running statistics with momentum and the
    unbiased variance, num_batches_tracked) and bn_eval_coeffs on the result."""
    log = {}
    for pixels, ld in ((3, C), (12345, C + 8), (2 * 17 * 33, C)):
        x, part, xs, k, e = _stats_case(pixels, C, ld, seed=C * 7 + pixels, far_mean=(C >= 4 and pixels > 100))
        log[f"stats p{pixels} ld{ld} worst/2u"] = e
        # bn_finalize on the kernel's rows: float64 math cast once to fp32
        g = _gen(C + 1)
        gamma, beta = _randn((C,), g, 0.5, 1.0), _randn((C,), g)
        rm0, rv0 = _randn((C,), g), _randn((C,), g).abs() + 0.5
        rm, rv = rm0.clone().cuda(), rv0.clone().cuda()
        nbt = torch.tensor([5], dtype=torch.int64, device="cuda")
        mom, eps = 0.1, 1e-5
        out = Guarded((4, C))
        _call("ub2_bn_finalize", _p(part), part.shape[0], C, pixels, _p(gamma.cuda()),
              _p(beta.cuda()), _p(rm), _p(rv), _p(nbt), mom, eps, _p(out.t[0]),
              _p(out.t[1]), _p(out.t[2]), _p(out.t[3]), _s())
        assert out.ok()
        s = _folded(part)
        m = s[0] / pixels
        var = (s[1] / pixels - m * m).clamp_min(0)
        inv = 1 / (var + float(np.float32(eps))).sqrt()
        g64, b64 = gamma.double(), beta.double()
        o = out.t.cpu().double()
        ef = max(_within(o[0], g64 * inv, (g64 * inv).abs(), 1, "scale"),
                 _within(o[1], b64 - m * g64 * inv, b64.abs() + (m * g64 * inv).abs(), 1, "shift"),
                 _within(o[2], m, m.abs(), 1, "mean"), _within(o[3], inv, inv, 1, "invstd"))
        unb = var * pixels / (pixels - 1) if pixels > 1 else var
        m32, u32 = m.float().double(), unb.float().double()
        # (1 - mom) * r + mom * v in fp32: three roundings (1 - mom is exact in float64 of the fp32 momentum)
        m1 = 1 - torch.tensor(mom, dtype=F32).double()
        mo = torch.tensor(mom, dtype=F32).double()
        ef = max(ef, _within(rm.cpu(), m1 * rm0.double() + mo * m32, (m1 * rm0.double()).abs() + (mo * m32).abs(), 3, "rm"),
                 _within(rv.cpu(), m1 * rv0.double() + mo * u32, (m1 * rv0.double()).abs() + (mo * u32).abs(), 3, "rv"))
        assert int(nbt.item()) == 6
        log[f"bn_finalize p{pixels} worst/2u"] = ef
        # end to end: the batch variance from fp32 per-thread sums against the two-pass float64 variance
        ref_var = xs.var(0, unbiased=False)
        bound = 2 * U * 2 * k * (xs * xs).sum(0) / pixels + 2 * U * 2 * k * xs.abs().sum(0) / pixels * m.abs() * 2
        err = (var - ref_var).abs()
        assert bool((err <= bound + 1e-300).all()), ("variance", pixels, C, float((err - bound).max()))
        log[f"variance p{pixels} worst rel"] = float((err / ref_var.clamp_min(1e-30)).max())
        if C >= 4 and pixels > 100:
            log[f"variance mean=100std p{pixels} rel"] = float(err[1] / ref_var[1])
        # eval coefficients: 1/sqrtf(rv + eps) (3 roundings), * gamma, beta - rm*g*inv (3 more)
        ec = Guarded((2, C))
        _call("ub2_bn_eval_coeffs", _p(gamma.cuda()), _p(beta.cuda()), _p(rm), _p(rv), eps, C,
              _p(ec.t[0]), _p(ec.t[1]), _s())
        assert ec.ok()
        rmd, rvd = rm.cpu().double(), rv.cpu().double()
        iv = 1 / (rvd + torch.tensor(eps, dtype=F32).double()).sqrt()
        e2 = max(_within(ec.t[0].cpu(), g64 * iv, (g64 * iv).abs(), 4, "eval scale"),
                 _within(ec.t[1].cpu(), b64 - rmd * g64 * iv, b64.abs() + (rmd * g64 * iv).abs() * 4, 7, "eval shift"))
        log[f"bn_eval_coeffs p{pixels} worst/2u"] = e2
    record(f"fp32 kernels channel_stats/bn_finalize C{C}", **log)


@GPU
def test_scalar_stats():
    log = {}
    for n in (1, 7, 2 * 33 * 17, 300001):
        g = _gen(n)
        x = Guarded((n,), fill=_randn((n,), g, 2.0, 0.5).cuda()).t
        rows = _rows("ub2_f32_scalar_rows", n)
        parts = []
        for _ in range(2):
            pg = Guarded((rows, 2, 1), F64)
            _call("ub2_f32_scalar_stats", _p(x), n, _p(pg.t), rows, _s())
            assert pg.ok()
            parts.append(pg.t.clone())
        assert torch.equal(parts[0], parts[1])
        xs = x.cpu().double()
        k = _per_thread(n, rows * KFT) + 5 + 1                 # per-thread adds, the warp tree, the 8-warp fold
        got = _folded(parts[0])
        log[f"n{n} worst/2u"] = max(_within(got[0, 0], xs.sum(), xs.abs().sum(), k, "sum"),
                                    _within(got[1, 0], (xs * xs).sum(), (xs * xs).sum(), k + 1, "sumsq"))
    record("fp32 kernels scalar_stats", **log)


# =============================================================================================== BN apply, max-pool
@GPU
@pytest.mark.parametrize("C", [4, 12, 20, 64])
@pytest.mark.parametrize("relu", [1, 0])
def test_affine_act(C, relu):
    g = _gen(C + relu)
    pixels = 2 * 13 * 7
    y = _randn((pixels, C), g)
    sc, sh = _randn((C,), g), _randn((C,), g)
    out = Guarded((pixels, C))
    _call("ub2_f32_affine_act", _p(y.cuda()), _p(sc.cuda()), _p(sh.cuda()), _p(out.t), pixels, C, relu, _s())
    assert out.ok()
    z = y.double() * sc.double() + sh.double()
    ref = z.clamp_min(0) if relu else z
    e = _within(out.t.cpu(), ref, z.abs(), 1, ("affine", C, relu))     # one fmaf
    record(f"fp32 kernels affine_act C{C} relu{relu}", worst_over_2u=e)


def _window_pos(flat, H, W):
    """F.max_pool2d's flat index (h*W + w) -> position (row*2 + col) inside the 2x2 window."""
    Hp, Wp = H // 2, W // 2
    hp = torch.arange(Hp).view(1, 1, Hp, 1)
    wp = torch.arange(Wp).view(1, 1, 1, Wp)
    return ((flat // W - 2 * hp) * 2 + (flat % W - 2 * wp)).to(torch.uint8)


@GPU
@pytest.mark.parametrize("N,H,W,C", [(2, 7, 9, 12), (1, 8, 6, 4), (3, 5, 4, 100), (1, 2, 2, 1024)])
def test_maxpool_idx_and_eval_maxpool(N, H, W, C):
    """Values from {-1, -0.0, +0.0, 1}, so nearly every window ties; four planted windows tie at every position.
    The first maximum in window order must win (ATen's rule), values compare by value (-0.0 == +0.0)."""
    g = _gen(N * H * W * C)
    vals = torch.tensor([-1.0, -0.0, 0.0, 1.0])
    a = vals[torch.randint(0, 4, (N, H, W, C), generator=g)]
    a[0, 0:2, 0:2, 0] = 2.0                                   # all four positions equal
    a[0, 0:2, 0:2, 1] = torch.tensor([[-0.0, 0.0], [0.0, -0.0]])
    a[-1, H - 2:H, W - 2:W, C - 1] = 3.0
    a[0, 0, 0, 2] = float("-inf")
    ad = a.cuda()
    p, idx = Guarded((N, H // 2, W // 2, C)), Guarded((N, H // 2, W // 2, C), torch.uint8)
    _call("ub2_f32_maxpool_idx", _p(ad), _p(p.t), _p(idx.t), N, H, W, C, _s())
    pe = Guarded((N, H // 2, W // 2, C))
    _call("ub2_f32_maxpool", _p(ad), _p(pe.t), N, H, W, C, _s())
    assert p.ok() and idx.ok() and pe.ok()
    rv, ri = F.max_pool2d(a.double().permute(0, 3, 1, 2), 2, return_indices=True)
    rpos = _window_pos(ri, H, W).permute(0, 2, 3, 1)
    rv = rv.permute(0, 2, 3, 1).float()
    assert bool((p.t.cpu() == rv).all()) and bool((pe.t.cpu() == rv).all())
    assert torch.equal(idx.t.cpu(), rpos), int((idx.t.cpu() != rpos).sum())
    # the sign of the returned zero is that of the first maximum (the value that won), as ATen returns it
    assert torch.equal(_bits(p.t.cpu()), _bits(rv))


# =============================================================================================== BN(+ReLU)(+pool) backward
def _routed(dA, dP, idx, N, H, W, C):
    """dA + the pooled gradient routed to the saved window position, float64 (NHWC)."""
    g = torch.zeros((N, H, W, C), dtype=F64)
    if dA is not None:
        g += dA.double()
    if dP is not None:
        Hp, Wp = H // 2, W // 2
        for r in range(2):
            for c in range(2):
                sel = (idx.long() == r * 2 + c).double() * dP.double()
                g[:, r:2 * Hp:2, c:2 * Wp:2, :] += sel
    return g


def _act_bwd(dA_full, ld_da, dP, idx, y, sc, sh, N, H, W, C, relu, mean, invstd, gamma, frozen, dgamma0, dbeta0):
    pixels = N * H * W
    dA = dA_full[..., :C] if dA_full is not None else None
    rows = _rows("ub2_f32_channel_rows", pixels, C)
    dev = {k: (v.cuda() if v is not None else None) for k, v in dict(dA=dA_full, dP=dP, idx=idx, y=y, sc=sc, sh=sh).items()}
    dA_ptr = _p(dev["dA"]) if dA is not None else _p(None)
    parts = []
    for _ in range(2):
        pg = Guarded((rows, 2, C), F64)
        _call("ub2_f32_act_bwd_reduce", dA_ptr, ld_da if dA is not None else 0, _p(dev["dP"]), _p(dev["idx"]), _p(dev["y"]),
              _p(dev["sc"]), _p(dev["sh"]), _p(pg.t), rows, N, H, W, C, relu, _s())
        assert pg.ok()
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1])
    dgamma, dbeta = dgamma0.clone().cuda(), dbeta0.clone().cuda()
    coef = Guarded((3, C))
    _call("ub2_bn_bwd_finalize", _p(parts[0]), rows, C, pixels, _p(gamma.cuda()), _p(mean.cuda()),
          _p(invstd.cuda()), int(frozen), _p(dgamma), _p(dbeta), _p(coef.t), _s())
    dy = Guarded((N, H, W, C))
    _call("ub2_f32_act_bwd_apply", dA_ptr, ld_da if dA is not None else 0, _p(dev["dP"]), _p(dev["idx"]), _p(dev["y"]),
          _p(dev["sc"]), _p(dev["sh"]), _p(coef.t), _p(dy.t), N, H, W, C, relu, _s())
    assert coef.ok() and dy.ok()
    return parts[0], rows, dgamma.cpu(), dbeta.cpu(), coef.t.cpu(), dy.t.cpu()


@GPU
@pytest.mark.parametrize("N,H,W,C,src,ld_extra,frozen", [
    (2, 7, 9, 12, "dA", 8, False), (2, 7, 9, 12, "dP", 0, False), (2, 7, 9, 12, "both", 4, False),
    (2, 7, 9, 12, "both", 0, True), (1, 6, 5, 100, "both", 0, False), (1, 3, 5, 1024, "both", 8, False),
    (2, 8, 8, 20, "dP", 0, True)])
def test_act_backward(N, H, W, C, src, ld_extra, frozen):
    """act_bwd_reduce -> bn_bwd_finalize -> act_bwd_apply against float64 autograd of
    relu(gamma * (y - mean) * invstd + beta) (batch statistics from y, or frozen running statistics), with the
    pooled gradient routed through idx; odd H / W leave the last row / column without a pooled gradient."""
    g = _gen(N * H * W * C + ld_extra)
    eps = 1e-5
    y = _randn((N, H, W, C), g, 1.5, 0.3)
    gamma, beta = _randn((C,), g, 0.5, 1.0), _randn((C,), g, 0.5)
    if frozen:
        mean64, var64 = _randn((C,), g).double(), (_randn((C,), g).abs() + 0.5).double()
    else:
        mean64, var64 = y.double().mean((0, 1, 2)), y.double().var((0, 1, 2), unbiased=False)
    mean, invstd = mean64.float(), (1 / (var64 + eps).sqrt()).float()
    sc = gamma * invstd
    sh = (beta.double() - mean.double() * gamma.double() * invstd.double()).float()
    dA_full = _randn((N, H, W, C + ld_extra), g) if src in ("dA", "both") else None
    dP = _randn((N, H // 2, W // 2, C), g) if src in ("dP", "both") else None
    idx = torch.randint(0, 4, (N, H // 2, W // 2, C), generator=g, dtype=torch.uint8) if dP is not None else None
    dg0, db0 = _randn((C,), g), _randn((C,), g)
    part, rows, dgamma, dbeta, coef, dy = _act_bwd(dA_full, C + ld_extra, dP, idx, y, sc, sh, N, H, W, C, 1, mean, invstd,
                                                   gamma, frozen, dg0, db0)
    dA = dA_full[..., :C] if dA_full is not None else None
    gin = _routed(dA, dP, idx, N, H, W, C)
    # the ReLU decision of the kernel: fmaf(y, scale, shift) > 0, whose sign is that of the exact value
    live = (y.double() * sc.double() + sh.double()) > 0
    gz = gin * live
    y64 = y.double()
    k = _per_thread(N * H * W, _lanes(C) * rows) + 1         # + the dA + dP add
    got = _folded(part)
    e_red = max(_within(got[0], gz.sum((0, 1, 2)), gz.abs().sum((0, 1, 2)), k, "sum g"),
                _within(got[1], (gz * y64).sum((0, 1, 2)), (gz * y64).abs().sum((0, 1, 2)), k + 1, "sum g*y"))
    # float64 autograd of the forward with the same (fp32) gamma / beta; batch mode recomputes the statistics
    yv = y64.clone().requires_grad_(True)
    gm, bt = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    if frozen:
        m_, is_ = mean.double(), invstd.double()
    else:
        m_ = yv.mean((0, 1, 2))
        is_ = 1 / (((yv - m_) ** 2).mean((0, 1, 2)) + eps).sqrt()
    z = gm * (yv - m_) * is_ + bt
    (z * live * gin).sum().backward()        # the ReLU as the kernel decides it (a decision at |z| ~ u is either way)
    # terms: |A g|, |B y|, |C| with dgamma and dbeta replaced by the magnitudes of their own sums
    A = (gamma.double() * invstd.double()).abs()
    M = N * H * W
    mu, iv = mean.double(), invstd.double()
    terms_dg = iv * ((gz * y64).abs().sum((0, 1, 2)) + mu.abs() * gz.abs().sum((0, 1, 2)))
    terms_dy = A * gz.abs() + (0 if frozen else A * iv * terms_dg / M * (y64.abs() + mu.abs()) + A * gz.abs().sum((0, 1, 2)) / M)
    e_dy = _within(dy, yv.grad, terms_dy, 8 + k, "dy")
    e_dg = _within(dgamma, dg0.double() + gm.grad, dg0.double().abs() + terms_dg * (k + 4), 2, "dgamma")
    e_db = _within(dbeta, db0.double() + bt.grad, db0.double().abs() + gz.abs().sum((0, 1, 2)) * (k + 2), 2, "dbeta")
    record(f"fp32 kernels act_backward {N}x{H}x{W}x{C} {src} ld+{ld_extra} frozen={frozen}",
           reduce_worst_over_2u=e_red, dy_worst_over_2u=e_dy, dgamma_worst_over_2u=e_dg, dbeta_worst_over_2u=e_db,
           dy_rel_l2=_rel_l2(dy, yv.grad))


@GPU
@pytest.mark.parametrize("N,H,W,C", [(2, 7, 9, 12), (1, 4, 4, 4), (1, 5, 3, 1024)])
def test_maxpool_backward_routing(N, H, W, C):
    """relu = 0 with identity coefficients and y = 0 (MaxPoolF32.backward): dy is the routed gradient, bit for bit."""
    g = _gen(N + H + W + C)
    dP = _randn((N, H // 2, W // 2, C), g)
    a = torch.randint(-1, 2, (N, H, W, C), generator=g).float()          # ties: the saved idx decides
    p, idx = torch.empty((N, H // 2, W // 2, C), device="cuda"), torch.empty((N, H // 2, W // 2, C), device="cuda", dtype=torch.uint8)
    _call("ub2_f32_maxpool_idx", _p(a.cuda()), _p(p), _p(idx), N, H, W, C, _s())
    ones, zeros = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
    coef = torch.stack([ones, zeros, zeros])
    dy = Guarded((N, H, W, C))
    _call("ub2_f32_act_bwd_apply", _p(None), 0, _p(dP.cuda()), _p(idx), _p(torch.zeros((N, H, W, C), device="cuda")), _p(ones),
          _p(zeros), _p(coef), _p(dy.t), N, H, W, C, 0, _s())
    assert dy.ok()
    ref = _routed(None, dP, idx.cpu(), N, H, W, C).float()
    assert torch.equal(_bits(dy.t.cpu()), _bits(ref))
    # and the same through autograd of F.max_pool2d (odd H / W: the last row / column get nothing)
    av = a.double().permute(0, 3, 1, 2).requires_grad_(True)
    (F.max_pool2d(av, 2) * dP.double().permute(0, 3, 1, 2)).sum().backward()
    assert torch.equal(dy.t.cpu().double(), av.grad.permute(0, 2, 3, 1))


# =============================================================================================== resampling
def _lerp_rows(n_out, n_in):
    """The kernels' align_corners=True taps in fp32 (resample.cuh src_index), as an (n_out, n_in) float64 matrix."""
    r = np.float32(np.float32(n_in - 1) / np.float32(n_out - 1)) if n_out > 1 else np.float32(0)
    M = np.zeros((n_out, n_in))
    for d in range(n_out):
        s = np.float32(r * np.float32(d))
        i0 = min(int(s), n_in - 1)
        i1 = i0 + (1 if i0 < n_in - 1 else 0)
        l1 = np.float32(s - np.float32(i0))
        l0 = np.float32(np.float32(1) - l1)
        M[d, i0] += float(l0)
        M[d, i1] += float(l1)
    return torch.from_numpy(M)


def _resample_ref(x, hu, wu, Ho, Wo):
    """x (N,hin,win,C) fp32 -> (N,Ho,Wo,C) float64 and the |terms| bound, with the padding of layers.py:98-102."""
    N, hin, win, C = x.shape
    Mh, Mw = _lerp_rows(hu, hin), _lerp_rows(wu, win)
    x64 = x.double()
    core = torch.einsum("ai,bj,nijc->nabc", Mh, Mw, x64)
    terms = torch.einsum("ai,bj,nijc->nabc", Mh.abs(), Mw.abs(), x64.abs())
    dh, dw = Ho - hu, Wo - wu
    pad = (0, 0, dw // 2, dw - dw // 2, dh // 2, dh - dh // 2)
    return F.pad(core, pad), F.pad(terms, pad), Mh, Mw


RESAMPLE = [(4, 5, 8, 10, 8, 10), (4, 5, 8, 10, 11, 13), (4, 5, 8, 10, 9, 10), (1, 5, 2, 10, 3, 10), (4, 1, 8, 2, 8, 3),
            (3, 4, 1, 8, 2, 8), (7, 7, 16, 16, 16, 16), (7, 9, 16, 17, 16, 17), (1, 1, 2, 2, 2, 2)]


@GPU
@pytest.mark.parametrize("hin,win,hu,wu,Ho,Wo", RESAMPLE)
def test_upsample_forward_backward_eval(hin, win, hu, wu, Ho, Wo):
    """f32_upsample_fwd (unrounded), f32_upsample (eval, TF32-rounded) and f32_upsample_bwd (gather transpose, dout
    with a channel stride above C) against the fp32 taps in float64; the taps themselves against F.interpolate +
    F.pad in float64 (to the taps' own fp32 rounding)."""
    N, C, ld = 2, 12, 20
    g = _gen(hin * 100 + win * 10 + hu + Ho)
    x = _randn((N, hin, win, C), g)
    ref, terms, Mh, Mw = _resample_ref(x, hu, wu, Ho, Wo)
    # the reference's taps are those of ATen to fp32 rounding of the source coordinate
    xt = x.double().permute(0, 3, 1, 2)
    ti = F.interpolate(xt, size=(hu, wu), mode="bilinear", align_corners=True)
    dh, dw = Ho - hu, Wo - wu
    ti = F.pad(ti, (dw // 2, dw - dw // 2, dh // 2, dh - dh // 2)).permute(0, 2, 3, 1)
    assert float((ti - ref).abs().max()) <= 16 * max(hin, win) * U * float(x.abs().max())
    xd = x.cuda()
    out = Guarded((N, Ho, Wo, C))
    _call("ub2_f32_upsample_fwd", _p(xd), _p(out.t), N, hin, win, hu, wu, Ho, Wo, C, _s())
    ev = Guarded((N, Ho, Wo, C))
    _call("ub2_f32_upsample", _p(xd), _p(ev.t), N, hin, win, hu, wu, Ho, Wo, C, _s())
    assert out.ok() and ev.ok()
    e_f = _within(out.t.cpu(), ref, terms, 4, "upsample_fwd")      # a0*(b0*v00 + b1*v01) + a1*(...)
    e_e = _within(ev.t.cpu(), ref, terms, 4, "upsample eval", tf32=True)
    # transpose: din = Mh^T dout Mw over the un-padded window
    dfull = _randn((N, Ho, Wo, ld), g)
    dout = dfull[..., :C]
    d64 = dout.double()[:, dh // 2:dh // 2 + hu, dw // 2:dw // 2 + wu, :]
    rb = torch.einsum("ai,bj,nabc->nijc", Mh, Mw, d64)
    tb = torch.einsum("ai,bj,nabc->nijc", Mh.abs(), Mw.abs(), d64.abs())
    k = int((Mh != 0).sum(0).max()) * int((Mw != 0).sum(0).max()) + 3   # fmaf per tap + the tap weight products
    din = Guarded((N, hin, win, C))
    _call("ub2_f32_upsample_bwd", _p(dfull.cuda()), ld, _p(din.t), N, hin, win, hu, wu, Ho, Wo, C, _s())
    assert din.ok()
    e_b = _within(din.t.cpu(), rb, tb, k, "upsample_bwd")
    # and against autograd of F.interpolate + F.pad (ATen's own taps)
    xv = xt.clone().requires_grad_(True)
    yv = F.pad(F.interpolate(xv, size=(hu, wu), mode="bilinear", align_corners=True), (dw // 2, dw - dw // 2, dh // 2, dh - dh // 2))
    (yv * dout.double().permute(0, 3, 1, 2)).sum().backward()
    e_ag = _rel_l2(din.t.cpu().permute(0, 3, 1, 2), xv.grad)
    assert e_ag <= 2e-5, e_ag                # ATen's float64 taps differ from the fp32 ones by ~u * hin
    record(f"fp32 kernels upsample {hin}x{win}->{hu}x{wu} in {Ho}x{Wo}", fwd_worst_over_2u=e_f, eval_worst_over_2u=e_e,
           bwd_worst_over_2u=e_b, bwd_rel_l2_vs_aten_autograd=e_ag)


# =============================================================================================== attention gate
def _fma32(a, b, c):
    """fp32 fmaf emulated in float64 (the product of two fp32 is exact in float64, so the sign is exact)."""
    return (a.double() * b.double() + c.double()).float()


def _gate_t(u, xp, sg, hg, sx, hx):
    """The training kernels' t = fmaf(u, sg, fmaf(xp, sx, hg + hx)) in fp32 (for the ReLU decision) and its terms."""
    t32 = _fma32(u, sg, _fma32(xp, sx, hg + hx))
    terms = (u.double() * sg.double()).abs() + (xp.double() * sx.double()).abs() + hg.double().abs() + hx.double().abs()
    return t32, terms


GATE_CI = [4, 36, 128, 132, 384, 388, 512]


@GPU
@pytest.mark.parametrize("Ci", GATE_CI)
def test_gate_training_passes(Ci):
    """gate_psi -> gate_apply -> gate_bwd_a -> bn_bwd_finalize(psi) -> gate_bwd_s -> gate_bwd_finalize -> gate_bwd_xg,
    each against float64 of its own formula on the operands it was given (layers.py:183-192 and its autograd)."""
    N, H, W = 2, 5, 7
    pixels = N * H * W
    Cx = Ci + 8 if Ci != 4 else 12
    ld_do = Cx + 4
    g = _gen(Ci)
    u, xp, x = _randn((pixels, Ci), g), _randn((pixels, Ci), g), _randn((pixels, Cx), g)
    sg, hg, sx, hx = _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5), _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5)
    wpsi = _randn((Ci,), g, 1 / math.sqrt(Ci))
    dev = lambda t: t.cuda()
    ud, xpd, xd, sgd, hgd, sxd, hxd, wd = map(dev, (u, xp, x, sg, hg, sx, hx, wpsi))
    log = {}
    # psi
    psi = Guarded((pixels,))
    _call("ub2_f32_gate_psi", _p(ud), _p(xpd), _p(sgd), _p(hgd), _p(sxd), _p(hxd), _p(wd), _p(psi.t), pixels, Ci, _s())
    assert psi.ok()
    t32, tt = _gate_t(u, xp, sg, hg, sx, hx)
    psi_ref = (wpsi.double() * t32.double().clamp_min(0)).sum(1)
    k_dot = 4 * _per_thread(Ci, 128) + 5 + 3
    log["psi"] = _within(psi.t.cpu(), psi_ref, (wpsi.double().abs() * tt).sum(1), k_dot, "psi")
    # apply, with and without a_out
    spsi, hpsi = torch.tensor([0.7]), torch.tensor([-0.2])
    out, a_out, out2 = Guarded((pixels, Cx)), Guarded((pixels,)), Guarded((pixels, Cx))
    _call("ub2_f32_gate_apply", _p(psi.t), _p(spsi.cuda()), _p(hpsi.cuda()), _p(xd), _p(out.t), _p(a_out.t), pixels, Cx, _s())
    _call("ub2_f32_gate_apply", _p(psi.t), _p(spsi.cuda()), _p(hpsi.cuda()), _p(xd), _p(out2.t), _p(None), pixels, Cx, _s())
    assert out.ok() and a_out.ok() and out2.ok()
    assert torch.equal(_bits(out.t), _bits(out2.t))
    psi32 = psi.t.cpu()
    z = psi32.double() * spsi.double() + hpsi.double()
    a_ref = torch.sigmoid(z)
    steps_a = z.abs() + 6              # fmaf, expf (2 ulp), 1 + e, the division; d a / d z = a (1 - a) <= a |z|-scaled
    log["a"] = _within(a_out.t.cpu(), a_ref, a_ref * steps_a, 1, "a")
    log["out"] = _within(out.t.cpu(), x.double() * a_ref.view(-1, 1), (x.double() * a_ref.view(-1, 1)).abs() * (steps_a.view(-1, 1) + 1), 1, "out")
    # backward a: dot over Cx, dn = dot * a * (1 - a), dx = dout * a, rows of (sum dn, sum dn * psi)
    a32 = a_out.t.cpu()
    dfull = _randn((pixels, ld_do), g)
    dout = dfull[:, :Cx]
    rows = _rows("ub2_f32_gate_rows", pixels)
    dx, dpsin = Guarded((pixels, Cx)), Guarded((pixels,))
    parts = []
    for _ in range(2):
        pg = Guarded((rows, 2, 1), F64)
        _call("ub2_f32_gate_bwd_a", _p(dfull.cuda()), ld_do, _p(xd), _p(a_out.t), _p(psi.t), _p(dx.t), _p(dpsin.t), _p(pg.t), rows,
              pixels, Cx, _s())
        assert pg.ok()
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and dx.ok() and dpsin.ok()
    a64 = a32.double()
    dot = (dout.double() * x.double()).sum(1)
    dot_t = (dout.double() * x.double()).abs().sum(1)
    w_a = a64 * (1 - a64)
    dn_ref = dot * w_a
    k_a = 4 * _per_thread(Cx, 128) + 5 + 3
    log["dx"] = _within(dx.t.cpu(), dout.double() * a64.view(-1, 1), (dout.double() * a64.view(-1, 1)).abs(), 1, "dx")
    log["dpsin"] = _within(dpsin.t.cpu(), dn_ref, dot_t * w_a, k_a, "dpsin")
    kp = _per_thread(pixels, rows * 8) + 1
    s = _folded(parts[0])
    psi64 = psi32.double()
    log["rows_a"] = max(_within(s[0, 0], dn_ref.sum(), (dot_t * w_a).sum() * (k_a + kp), 1, "sum dn"),
                        _within(s[1, 0], (dn_ref * psi64).sum(), (dot_t * w_a * psi64.abs()).sum() * (k_a + kp + 1), 1, "sum dn psi"))
    # BN_psi backward (batch statistics of psi, C = 1)
    mp, ip, gp = torch.tensor([0.1]), torch.tensor([1.3]), torch.tensor([0.7])
    dgp, dbp = torch.tensor([0.25]).cuda(), torch.tensor([-0.5]).cuda()
    coef_p = Guarded((3, 1))
    _call("ub2_bn_bwd_finalize", _p(parts[0]), rows, 1, pixels, _p(gp.cuda()), _p(mp.cuda()), _p(ip.cuda()), 0,
          _p(dgp), _p(dbp), _p(coef_p.t), _s())
    assert coef_p.ok()
    dbr, dgr = s[0, 0], ip.double()[0] * (s[1, 0] - mp.double()[0] * s[0, 0])
    A = gp.double()[0] * ip.double()[0]
    B = -A * ip.double()[0] * dgr / pixels
    Cc = -A * dbr / pixels - B * mp.double()[0]
    cp = coef_p.t.cpu().double().view(-1)
    log["bn_bwd_finalize"] = max(
        _within(dbp.cpu().double(), -0.5 + dbr, 0.5 + abs(dbr), 2, "dbeta_psi"),
        _within(dgp.cpu().double(), 0.25 + dgr, 0.25 + abs(dgr) + ip.double()[0] * abs(mp.double()[0] * s[0, 0]), 2, "dgamma_psi"),
        _within(cp[0], A, abs(A), 1, "A"), _within(cp[1], B, abs(B), 1, "B"), _within(cp[2], Cc, abs(A * dbr / pixels) + abs(B * mp.double()[0]), 1, "C"))
    # backward s
    ds = Guarded((pixels, Ci))
    rows_s = rows
    parts2 = []
    for _ in range(2):
        pg = Guarded((rows_s, 4, Ci), F64)
        _call("ub2_f32_gate_bwd_s", _p(dpsin.t), _p(psi.t), _p(coef_p.t), _p(ud), _p(xpd), _p(sgd), _p(hgd), _p(sxd), _p(hxd), _p(wd),
              _p(ds.t), _p(pg.t), rows_s, pixels, Ci, _s())
        assert pg.ok()
        parts2.append(pg.t.clone())
    assert torch.equal(parts2[0], parts2[1]) and ds.ok()
    c32 = coef_p.t.cpu().view(-1)
    dpsin64 = dpsin.t.cpu().double()
    dpr = c32[0].double() * dpsin64 + c32[1].double() * psi64 + c32[2].double()
    dpr_t = (c32[0].double() * dpsin64).abs() + (c32[1].double() * psi64).abs() + c32[2].double().abs()
    live = (t32 > 0).double()
    d_ref = dpr.view(-1, 1) * wpsi.double() * live
    d_t = dpr_t.view(-1, 1) * wpsi.double().abs() * live
    log["ds"] = _within(ds.t.cpu(), d_ref, d_t, 3, "ds")
    k_s = _per_thread(pixels, rows_s * 8) + 4
    s2 = _folded(parts2[0])
    relu_t = t32.double().clamp_min(0)
    u64, xp64 = u.double(), xp.double()
    log["rows_s"] = max(
        _within(s2[0], d_ref.sum(0), d_t.sum(0), k_s, "sum ds"),
        _within(s2[1], (d_ref * xp64).sum(0), (d_t * xp64.abs()).sum(0), k_s + 1, "sum ds xp"),
        _within(s2[2], (d_ref * u64).sum(0), (d_t * u64.abs()).sum(0), k_s + 1, "sum ds u"),
        _within(s2[3], (dpr.view(-1, 1) * relu_t).sum(0), (dpr_t.view(-1, 1) * relu_t).sum(0), k_s + 3, "sum dpsi relu(t)"))
    # gate_bwd_finalize into non-zero targets
    mx, ix, gx = _randn((Ci,), g), _randn((Ci,), g).abs() + 0.5, _randn((Ci,), g)
    mg, ig, gg = _randn((Ci,), g), _randn((Ci,), g).abs() + 0.5, _randn((Ci,), g)
    t0 = _randn((5, Ci), g)
    targets = t0.clone().cuda()
    coef = Guarded((6, Ci))
    _call("ub2_gate_bwd_finalize", _p(parts2[0]), rows_s, Ci, pixels, _p(gx.cuda()), _p(mx.cuda()),
          _p(ix.cuda()), _p(gg.cuda()), _p(mg.cuda()), _p(ig.cuda()), 0, _p(targets[0]), _p(targets[1]), _p(targets[2]),
          _p(targets[3]), _p(targets[4]), _p(coef.t), _s())
    assert coef.ok()
    mx6, ix6, gx6, mg6, ig6, gg6 = (v.double() for v in (mx, ix, gx, mg, ig, gg))
    db = s2[0]
    dgx = ix6 * (s2[1] - mx6 * s2[0])
    dgg = ig6 * (s2[2] - mg6 * s2[0])
    vals = [dgx, db, dgg, db, s2[3]]
    got_t = targets.cpu().double()
    e_fin = max(_within(got_t[r], t0[r].double() + vals[r], t0[r].double().abs() + vals[r].abs(), 2, f"target {r}") for r in range(5))
    Ax, Ag = gx6 * ix6, gg6 * ig6
    Bx, Bg = -Ax * ix6 * dgx / pixels, -Ag * ig6 * dgg / pixels
    cref = [Ax, Bx, -Ax * db / pixels - Bx * mx6, Ag, Bg, -Ag * db / pixels - Bg * mg6]
    cterm = [Ax.abs(), Bx.abs(), (Ax * db / pixels).abs() + (Bx * mx6).abs(), Ag.abs(), Bg.abs(), (Ag * db / pixels).abs() + (Bg * mg6).abs()]
    cg = coef.t.cpu().double()
    e_fin = max([e_fin] + [_within(cg[r], cref[r], cterm[r], 1, f"coef {r}") for r in range(6)])
    log["gate_bwd_finalize"] = e_fin
    # backward xg
    dxp, du = Guarded((pixels, Ci)), Guarded((pixels, Ci))
    _call("ub2_f32_gate_bwd_xg", _p(ds.t), _p(xpd), _p(ud), _p(coef.t), _p(dxp.t), _p(du.t), pixels, Ci, _s())
    assert dxp.ok() and du.ok()
    c6 = coef.t.cpu().double()
    ds64 = ds.t.cpu().double()
    log["dxp"] = _within(dxp.t.cpu(), c6[0] * ds64 + c6[1] * xp64 + c6[2],
                         (c6[0] * ds64).abs() + (c6[1] * xp64).abs() + c6[2].abs(), 2, "dxp")
    log["du"] = _within(du.t.cpu(), c6[3] * ds64 + c6[4] * u64 + c6[5],
                        (c6[3] * ds64).abs() + (c6[4] * u64).abs() + c6[5].abs(), 2, "du")
    record(f"fp32 kernels gate training Ci{Ci} Cx{Cx} (worst error / 2u*terms)", **log)


@GPU
@pytest.mark.parametrize("Ci", GATE_CI)
def test_gate_eval(Ci):
    """f32_gate: q at low resolution resampled to (H, W) (the gate's arbitrary size, 7x5 -> 16x9), Cx != 2 Ci."""
    N, hin, win, H, W = 2, 7, 5, 16, 9
    Cx = Ci + 8 if Ci != 4 else 12
    g = _gen(Ci + 1)
    q, xp, x = _randn((N, hin, win, Ci), g), _randn((N, H, W, Ci), g), _randn((N, H, W, Cx), g)
    sg, hg, sx, hx = _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5), _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5)
    wpsi = _randn((Ci,), g, 1 / math.sqrt(Ci))
    spsi, hpsi = torch.tensor([0.9]), torch.tensor([0.1])
    out = Guarded((N, H, W, Cx))
    _call("ub2_f32_gate", _p(q.cuda()), _p(xp.cuda()), _p(x.cuda()), _p(sg.cuda()), _p(hg.cuda()), _p(sx.cuda()), _p(hx.cuda()),
          _p(wpsi.cuda()), _p(spsi.cuda()), _p(hpsi.cuda()), _p(out.t), N, hin, win, H, W, Ci, Cx, _s())
    assert out.ok()
    up, up_t, _, _ = _resample_ref(q, H, W, H, W)
    t = up * sg.double() + hg.double() + xp.double() * sx.double() + hx.double()
    t_terms = up_t * sg.double().abs() + hg.double().abs() + (xp.double() * sx.double()).abs() + hx.double().abs()
    dot = (torch.relu(t) * wpsi.double()).sum(-1)
    k = 4 * _per_thread(Ci, 128) + 5 + 8                     # fma chain + warp tree + the interpolation and t roundings
    dot_err = 2 * U * k * (t_terms * wpsi.double().abs()).sum(-1)
    z = dot * spsi.double() + hpsi.double()
    a = torch.sigmoid(z)
    ref = x.double() * a.unsqueeze(-1)
    # |d out / d z| = |x| a (1 - a); the sigmoid itself and x * a: (|z| + 7) roundings; then one TF32 ulp
    zerr = spsi.double().abs() * dot_err + 2 * U * z.abs()
    bound = x.double().abs() * (a * (1 - a) * zerr + 2 * U * a * (z.abs() + 7)).unsqueeze(-1)
    bound = bound + 2.0 ** -10 * ref.abs()
    err = (out.t.cpu().double() - ref).abs()
    assert bool((err <= bound + 2.0 ** -140).all()), float((err - bound).max())
    record(f"fp32 kernels gate eval Ci{Ci} Cx{Cx}", worst_err_over_bound=float((err / bound.clamp_min(1e-300)).max()),
           rel_l2=_rel_l2(out.t.cpu(), ref))


# =============================================================================================== output head
@GPU
@pytest.mark.parametrize("K,C", [(1, 4), (2, 64), (3, 12), (8, 188), (8, 20)])
def test_outc_backward_and_eval(K, C):
    """f32_outc_bwd (da optional; dw and db accumulate into non-zero tensors) and f32_outc (bias optional); K = 8 with
    C = 188 is the largest head that fits the 48 KB of shared memory (C = 192 is refused on the host)."""
    N, H, W = 2, 9, 11
    pixels = N * H * W
    g = _gen(K * 1000 + C)
    a, w, b = _randn((N, H, W, C), g), _randn((K, C), g, 1 / math.sqrt(C)), _randn((K,), g)
    dl = _randn((N, K, H, W), g)
    dw0, db0 = _randn((K, C), g), _randn((K,), g)
    ad, wd, dld = a.cuda(), w.cuda(), dl.cuda()
    rows = _rows("ub2_f32_outc_rows", N, H, W)
    a64, w64, dl64 = a.double(), w.double(), dl.double().permute(0, 2, 3, 1)
    res = {}
    for with_da in (True, False):
        da = Guarded((N, H, W, C))
        dw, db = dw0.clone().cuda(), db0.clone().cuda()
        pg = Guarded((rows, K * C + K), F64)
        _call("ub2_f32_outc_bwd", _p(dld), _p(ad), _p(wd), _p(da.t) if with_da else _p(None), _p(pg.t), rows, _p(dw), _p(db), N, H, W, C,
              K, _s())
        assert pg.ok() and da.ok()
        res[with_da] = (da, dw.cpu(), db.cpu(), pg.t.clone())
    assert torch.equal(res[True][3], res[False][3]) and torch.equal(res[True][1], res[False][1])
    assert bool(torch.isnan(res[False][0].t).all())                 # da = NULL writes nothing
    da, dw, db, _ = res[True]
    log = {"da": _within(da.t.cpu(), dl64 @ w64, dl64.abs() @ w64.abs(), K, "da")}
    k = _per_thread(pixels, rows * 8) + 2
    dwr = torch.einsum("nhwk,nhwc->kc", dl64, a64)
    dwt = torch.einsum("nhwk,nhwc->kc", dl64.abs(), a64.abs())
    log["dw"] = _within(dw, dw0.double() + dwr, dw0.double().abs() + dwt * k, 1, "dw")
    log["db"] = _within(db, db0.double() + dl64.sum((0, 1, 2)), db0.double().abs() + dl64.abs().sum((0, 1, 2)) * k, 1, "db")
    for bias in (b, None):
        lg = Guarded((N, K, H, W))
        _call("ub2_f32_outc", _p(ad), _p(wd), _p(bias.cuda() if bias is not None else None), _p(lg.t), N, H, W, C, K, _s())
        assert lg.ok()
        ref = torch.einsum("nhwc,kc->nkhw", a64, w64) + (b.double().view(1, K, 1, 1) if bias is not None else 0)
        terms = torch.einsum("nhwc,kc->nkhw", a64.abs(), w64.abs()) + (b.double().abs().view(1, K, 1, 1) if bias is not None else 0)
        log[f"logits bias={bias is not None}"] = _within(lg.t.cpu(), ref, terms, C + 1, "logits")
    record(f"fp32 kernels outc K{K} C{C}", **log)


# =============================================================================================== first convolution
CONV_IN = [(1, 4, 2, 5, 7), (3, 20, 1, 1, 9), (4, 64, 2, 8, 1), (7, 1024, 1, 3, 4), (1, 64, 2, 16, 16), (3, 4, 1, 1, 1),
           (7, 20, 2, 6, 5)]


@GPU
@pytest.mark.parametrize("Cin,Cout,N,H,W", CONV_IN)
def test_conv_in(Cin, Cout, N, H, W):
    """f32_conv_in_raw (exact fp32), f32_conv_in (eval: + folded BN + ReLU, TF32-rounded) and f32_conv_in_wgrad
    (accumulating into a non-zero gradient) against float64 conv2d / conv2d_weight."""
    g = _gen(Cin * 10000 + Cout + H)
    x, w = _randn((N, Cin, H, W), g), _randn((Cout, Cin, 3, 3), g, 1 / math.sqrt(9 * Cin))
    xd, wd = x.cuda(), w.cuda()
    x64, w64 = x.double(), w.double()
    ref = F.conv2d(x64, w64, padding=1).permute(0, 2, 3, 1)
    terms = F.conv2d(x64.abs(), w64.abs(), padding=1).permute(0, 2, 3, 1)
    out = Guarded((N, H, W, Cout))
    _call("ub2_f32_conv_in_raw", _p(xd), _p(wd), _p(out.t), N, Cin, H, W, Cout, _s())
    assert out.ok()
    log = {"raw": _within(out.t.cpu(), ref, terms, 9 * Cin, "conv_in_raw")}
    sc, sh = _randn((Cout,), g, 0.5, 1.0), _randn((Cout,), g, 0.3)
    ev = Guarded((N, H, W, Cout))
    _call("ub2_f32_conv_in", _p(xd), _p(wd), _p(sc.cuda()), _p(sh.cuda()), _p(ev.t), N, Cin, H, W, Cout, _s())
    assert ev.ok()
    pre = ref * sc.double() + sh.double()
    pre_t = terms * sc.double().abs() + sh.double().abs()
    evr = pre.clamp_min(0)
    log["eval"] = _within(ev.t.cpu(), evr, pre_t, 9 * Cin + 1, "conv_in eval", tf32=True)
    dy = _randn((N, H, W, Cout), g)
    g0 = _randn((Cout, Cin, 3, 3), g)
    rows = _rows("ub2_f32_channel_rows", N * H * W, Cout)
    grads, parts = [], []
    for _ in range(2):
        grad = Guarded((Cout, Cin, 3, 3), fill=g0.cuda())
        pg = Guarded((rows, Cin, 9, Cout), F64)
        _call("ub2_f32_conv_in_wgrad", _p(xd), _p(dy.cuda()), _p(pg.t), rows, _p(grad.t), N, Cin, H, W, Cout, _s())
        assert grad.ok() and pg.ok()
        grads.append(grad.t.cpu())
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(grads[0], grads[1])
    dy64 = dy.double().permute(0, 3, 1, 2)
    gr = torch.nn.grad.conv2d_weight(x64, w64.shape, dy64, padding=1)
    gt = torch.nn.grad.conv2d_weight(x64.abs(), w64.shape, dy64.abs(), padding=1)
    k = _per_thread(N * H * W, _lanes(Cout) * rows) + 1
    log["wgrad"] = _within(grads[0], g0.double() + gr, g0.double().abs() + gt * k, 1, "conv_in_wgrad")
    record(f"fp32 kernels conv_in Cin{Cin} Cout{Cout} {N}x{H}x{W}", **log)


# =============================================================================================== splits and packs
def _with_denormals(shape, g):
    x = _randn(shape, g, 3.0)
    flat = x.view(-1)
    n = flat.numel()
    sel = torch.randperm(n, generator=g)[: max(n // 16, 4)]
    flat[sel[0::4]] = torch.tensor(1.1e-39)                 # subnormal
    flat[sel[1::4]] = torch.tensor(-7.3e-41)
    flat[sel[2::4]] = torch.tensor(2.0 ** -126 * 1.4999)     # smallest normals, whose lo is subnormal
    flat[sel[3::4]] = 0.0
    # mantissas with the TF32 rounding bit pattern exactly at the tie (ties away from zero)
    ties = torch.randperm(n, generator=g)[: max(n // 16, 4)]
    tb = flat[ties].view(torch.int32)
    flat[ties] = ((tb & ~0x1FFF) | 0x1000).view(F32)
    return x


@GPU
@pytest.mark.parametrize("C0,ld0,C1,ld1", [(16, 16, 0, 0), (12, 20, 8, 16), (4, 4, 4, 12), (64, 64, 64, 128)])
def test_split_tf32(C0, ld0, C1, ld1):
    """[hi(x0) | hi(x1) | lo(x0) | lo(x1)], hi = tf32(x), lo = tf32(x - hi), bit for bit; channel strides above C,
    C1 = 0 (x1 NULL), subnormals and exact TF32 ties."""
    pixels = 3 * 7
    g = _gen(C0 * 100 + C1 + ld0)
    x0f = _with_denormals((pixels, ld0), g)
    x1f = _with_denormals((pixels, ld1), g) if C1 else None
    C = C0 + C1
    out = Guarded((pixels, 2 * C))
    _call("ub2_f32_split_tf32", _p(x0f.cuda()), ld0, C0, _p(x1f.cuda() if C1 else None), ld1, C1, _p(out.t), pixels, _s())
    assert out.ok()
    v = torch.cat([x0f[:, :C0]] + ([x1f[:, :C1]] if C1 else []), 1)
    hi = _tf32(v)
    lo = _tf32(v - hi)
    assert torch.equal(_bits(out.t.cpu()), _bits(torch.cat([hi, lo], 1)))


@GPU
@pytest.mark.parametrize("Cout,Cin,taps", [(16, 16, 9), (20, 12, 1), (4, 36, 9), (64, 48, 1)])
def test_weight_packs(Cout, Cin, taps):
    """f32_pack_weight3 (forward and data-gradient packs, taps flipped) and f32_pack_weight (eval: TF32-rounded),
    bit for bit."""
    g = _gen(Cout * Cin * taps)
    k = int(round(math.sqrt(taps)))
    w = _with_denormals((Cout, Cin, k, k), g)
    wd = w.cuda()
    hi, lo = _tf32(w), _tf32(w - _tf32(w))
    for dgrad in (0, 1):
        R, Kc = (Cin, Cout) if dgrad else (Cout, Cin)
        out = Guarded((R, taps, 3 * Kc))
        _call("ub2_f32_pack_weight3", _p(wd), _p(out.t), Cout, Cin, taps, dgrad, _s())
        assert out.ok()
        if dgrad:
            h = hi.flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, taps, Cout)
            l = lo.flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, taps, Cout)
        else:
            h = hi.permute(0, 2, 3, 1).reshape(Cout, taps, Cin)
            l = lo.permute(0, 2, 3, 1).reshape(Cout, taps, Cin)
        assert torch.equal(_bits(out.t.cpu()), _bits(torch.cat([h, h, l], 2))), dgrad
    pk = Guarded((Cout, taps, Cin))
    _call("ub2_f32_pack_weight", _p(wd), _p(pk.t), Cout, Cin, taps, _s())
    assert pk.ok()
    assert torch.equal(_bits(pk.t.cpu()), _bits(hi.permute(0, 2, 3, 1).reshape(Cout, taps, Cin)))


@GPU
def test_split_bf16():
    """x -> (hi, lo) bf16 with hi = bf16(x) and lo = bf16(x - hi), round to nearest even, bit for bit."""
    g = _gen(77)
    x = _with_denormals((4 * 9 * 5 * 12,), g)
    hi, lo = Guarded((x.numel(),), torch.bfloat16), Guarded((x.numel(),), torch.bfloat16)
    _call("ub2_f32_split_bf16", _p(x.cuda()), _p(hi.t), _p(lo.t), x.numel(), _s())
    assert hi.ok() and lo.ok()
    rh = x.to(torch.bfloat16)
    rl = (x - rh.float()).to(torch.bfloat16)
    assert torch.equal(_bits(hi.t.cpu()), _bits(rh)) and torch.equal(_bits(lo.t.cpu()), _bits(rl))


# =============================================================================================== compositions
CONV3 = [  # N, H, W, C0, ld0, C1, ld1, Cout, k
    (2, 9, 7, 16, 16, 0, 0, 16, 3), (1, 8, 8, 16, 32, 16, 48, 32, 3), (2, 1, 12, 32, 32, 0, 0, 16, 3),
    (1, 11, 1, 16, 16, 16, 16, 48, 3), (2, 6, 10, 48, 64, 0, 0, 64, 1), (1, 13, 17, 16, 16, 32, 32, 16, 1)]


@GPU
@pytest.mark.parametrize("N,H,W,C0,ld0,C1,ld1,Cout,k", CONV3)
def test_conv3_and_weight_grad(N, H, W, C0, ld0, C1, ld1, Cout, k):
    """fp32.conv3 (forward and dgrad) and fp32.weight_grad on full-precision fp32 operands (not TF32-representable)
    against float64 conv2d / conv2d_input / conv2d_weight: two-source virtual concat, sources with channel strides
    above C, taps 1 and 9, H or W = 1, odd sizes."""
    from unet import fp32
    g = _gen(N * H * W + C0 + C1 + Cout + k)
    f0 = _randn((N, H, W, ld0), g)
    f1 = _randn((N, H, W, ld1), g) if C1 else None
    Cin = C0 + C1
    w = _randn((Cout, Cin, k, k), g, 1 / math.sqrt(k * k * Cin))
    x0 = f0.cuda()[..., :C0]
    x1 = f1.cuda()[..., :C1] if C1 else None
    wd = w.cuda()
    x = torch.cat([f0[..., :C0]] + ([f1[..., :C1]] if C1 else []), 3).double().permute(0, 3, 1, 2)
    ref = F.conv2d(x, w.double(), padding=k // 2).permute(0, 2, 3, 1)
    y = fp32.conv3(x0, x1, wd)
    e_f = _rel_l2(y.cpu(), ref)
    dy = _randn((N, H, W, Cout), g)
    dx = fp32.conv3(dy.cuda(), None, wd, dgrad=True)
    dxr = torch.nn.grad.conv2d_input(x.shape, w.double(), dy.double().permute(0, 3, 1, 2), padding=k // 2).permute(0, 2, 3, 1)
    e_d = _rel_l2(dx.cpu(), dxr)
    gw = fp32.weight_grad(x0, x1, dy.cuda(), w.shape)
    gw2 = fp32.weight_grad(x0, x1, dy.cuda(), w.shape)
    assert torch.equal(gw, gw2)
    gwr = torch.nn.grad.conv2d_weight(x, w.shape, dy.double().permute(0, 3, 1, 2), padding=k // 2)
    e_w = _rel_l2(gw.cpu(), gwr)
    record(f"fp32 kernels conv3/weight_grad {N}x{H}x{W} C{C0}+{C1} ld{ld0}/{ld1} Cout{Cout} k{k}", conv3_fwd_rel_l2=e_f,
           conv3_dgrad_rel_l2=e_d, weight_grad_rel_l2=e_w)
    assert e_f <= 1e-5 and e_d <= 1e-5, (e_f, e_d)       # 3xTF32: ~2^-21; one pass or no lo terms: >= 3e-4
    assert e_w <= 1e-4, e_w                              # bf16 hi/lo: ~2^-16; a dropped cross term: ~2^-9


# =============================================================================================== 64-bit offsets
@GPU
def test_offsets_past_2_pow_31():
    """(33, 256, 256, 1024) fp32 = 2.2e9 elements: f32_affine_act, f32_maxpool_idx and f32_act_bwd_apply with dP
    routing; the last rows of the last image and a seeded sample of pixels against float64 computed on the device
    for just those pixels."""
    N, H, W, C = 33, 256, 256, 1024
    assert N * H * W * C > 2 ** 31
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory, {free / 1e9:.1f} GB free")
    gen = torch.Generator(device="cuda").manual_seed(11)
    y = torch.empty((N, H, W, C), device="cuda")
    for i in range(0, N, 4):
        y[i:i + 4].normal_(generator=gen)
    sc = torch.rand(C, device="cuda", generator=gen) + 0.5
    sh = torch.randn(C, device="cuda", generator=gen)
    out = torch.empty_like(y)
    pixels = N * H * W
    _call("ub2_f32_affine_act", _p(y), _p(sc), _p(sh), _p(out), pixels, C, 1, _s())
    p = torch.empty((N, H // 2, W // 2, C), device="cuda")
    idx = torch.empty((N, H // 2, W // 2, C), device="cuda", dtype=torch.uint8)
    _call("ub2_f32_maxpool_idx", _p(out), _p(p), _p(idx), N, H, W, C, _s())
    # sample: the last two rows of the last image and 512 seeded pixels
    gs = torch.Generator().manual_seed(12)
    flat = torch.cat([torch.arange(pixels - 2 * W, pixels), torch.randint(0, pixels, (512,), generator=gs)]).cuda()
    yf, of = y.view(pixels, C), out.view(pixels, C)
    z = yf[flat].double() * sc.double() + sh.double()
    e_a = _within(of[flat], z.clamp_min(0), z.abs(), 1, "affine_act 64-bit")
    # pooled pixels: last rows of the last image and a sample
    Hp, Wp = H // 2, W // 2
    pp = torch.cat([torch.arange(N * Hp * Wp - Wp, N * Hp * Wp), torch.randint(0, N * Hp * Wp, (512,), generator=gs)]).cuda()
    n, hp, wp = pp // (Hp * Wp), (pp // Wp) % Hp, pp % Wp
    win = torch.stack([out[n, 2 * hp + r, 2 * wp + c] for r in (0, 1) for c in (0, 1)], 1).double()   # (P, 4, C)
    rv, ri = win.max(1)
    # first maximum in window order
    first = (win == rv.unsqueeze(1)).double().argmax(1)
    assert torch.equal(p.view(-1, C)[pp].double(), rv)
    assert torch.equal(idx.view(-1, C)[pp].long(), first)
    del win
    # backward routing: dy = dP routed (identity coefficients, relu off), y reused as the output buffer
    dP = torch.empty_like(p).normal_(generator=gen)
    ones, zeros = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
    coef = torch.stack([ones, zeros, zeros])
    _call("ub2_f32_act_bwd_apply", _p(None), 0, _p(dP), _p(idx), _p(out), _p(ones), _p(zeros), _p(coef), _p(y), N, H, W, C, 0, _s())
    n, h, w_ = flat // (H * W), (flat // W) % H, flat % W
    inside = ((h // 2) < Hp) & ((w_ // 2) < Wp)
    ppi = (n * Hp + h // 2) * Wp + w_ // 2
    pos = ((h % 2) * 2 + (w_ % 2)).unsqueeze(1)
    routed = torch.where(idx.view(-1, C)[ppi].long() == pos, dP.view(-1, C)[ppi], torch.zeros((), device="cuda"))
    routed = routed * inside.unsqueeze(1)
    assert torch.equal(yf[flat], routed)
    record("fp32 kernels 64-bit offsets 33x256x256x1024", affine_worst_over_2u=e_a)
    del y, out, p, idx, dP
    torch.cuda.empty_cache()
