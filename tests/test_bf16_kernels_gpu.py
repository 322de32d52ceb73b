"""bf16 mode one entry point at a time: the bandwidth-bound kernels between the convolutions (csrc/bn.cu, gate.cu,
head.cu, shuffle.cu) called through ``_C.call`` on caller-built tensors and compared with a float64 reference of the
same formula on the same operands, at the channel geometries each kernel's thread mapping produces.

Gates are derived from the arithmetic of each kernel, as in test_fp32_kernels_gpu.py (u = 2^-24):

* fp32 steps: ``|got - ref| <= 2 u * steps * sum|terms|``, ``steps`` read off the launch geometry (the fp32
  additions one thread performs; the rows a block folds in fp64 add nothing visible); reductions are bounded by the
  magnitudes of their terms, never relative to the sum, which nearly cancels for dbeta, dwpsi or a bias gradient;
* a bf16 output adds one bf16 rounding, ``2^-8 |ref|``; each test also counts the elements that are not
  bit-identical to RN_bf16(ref) and writes the count to the parity log;
* exact: the ReLU masks of bn.cu (y (bf16) * scale (fp32) is exact in float64, and neither float64 rounding nor the
  kernel's fmaf changes the sign of y*scale + shift), max-pool values and window positions (taken on the kernel's
  own ``a``: strict ``>``, the first maximum wins, -0 == +0, the pooled value is the selected element bit for bit),
  copies and packs;
* attention gate: the up-sampling weights are built as resample.cuh:src_index builds them (fp32 ratio and source
  coordinate, reproduced by NumPy float32) and interpolated in float64; a channel whose |t| lies within t's own fp32
  error bound is undecided for the ReLU, which the bounds of psi and of gate_bwd_s's sums absorb and where ``ds``
  may take either branch's value; the sigmoid uses ``__expf`` (CUDA: 2 + floor(1.16 |z|) ulp) and an IEEE
  division.

Every launch writes into the middle of a NaN / 0xA5 guard band whose bands are checked afterwards; outputs with a
channel stride above C have their pad channels filled with a bf16 sentinel that must survive; inputs are channel
slices of wider tensors; every reduction runs twice and must repeat bit for bit; workspace rows come from the
matching ``*_rows`` query.  Each test records its worst error in units of its bound in the parity log.

Not covered on purpose, as in the fp32 file: NaN inputs.

The host-side argument checks (no ``gpu`` mark) run every entry point in a child process without a device: bad
arguments must come back as their negative UB2_ERR code, valid ones, including every NULL the modules pass, as a
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
from test_fp32_kernels_gpu import (F32, F64, ROOT, U, Guarded, _bits, _call, _folded, _gen, _lerp_rows, _p, _per_thread,
                                   _randn, _routed, _rows, _s)

GPU = pytest.mark.gpu
BF16 = torch.bfloat16
SENT = 0x7FA5                 # a bf16 NaN payload in the pad channels of strided outputs
KBN = 256                     # threads per block of bn.cu (bn_block = cgs * floor(256 / cgs))
KGATE = 256                   # threads per block of gate.cu and head.cu
STRIP = 16                    # kGateStrip: rows per strip block


# =============================================================================================== helpers
def _bf(x):
    return torch.as_tensor(x).to(BF16)


def _rand_bf(shape, g, scale=1.0, shift=0.0):
    return _bf(_randn(shape, g, scale, shift))


class Out:
    """An NHWC output of C channels with channel stride ld inside a Guarded buffer: pad channels hold SENT."""

    def __init__(self, lead, C, ld, dtype=BF16):
        self.g = Guarded(tuple(lead) + (ld,), dtype)
        self.C, self.ld = C, ld
        if ld > C:
            self.g.t[..., C:].view(torch.int16).fill_(SENT)
        self.t = self.g.t[..., :C]

    def ok(self):
        return self.g.ok() and bool((self.g.t[..., self.C:].view(torch.int16) == SENT).all())


def _slice(full_cpu, C):
    """A channel slice of a wider tensor on the device (the kernels' channel stride = full width)."""
    return full_cpu.cuda()[..., :C]


def _check(got, ref, tol, what):
    """|got - ref| <= tol elementwise; returns the worst error in units of the bound."""
    got = torch.as_tensor(got).detach().double().cpu()
    ref = torch.as_tensor(ref).detach().double().cpu()
    tol = torch.as_tensor(tol).detach().double().cpu()
    err = (got - ref).abs()
    bad = ~(err <= tol)
    if bool(bad.any()):
        i = int(torch.nonzero(bad.reshape(-1))[0])
        raise AssertionError((what, int(bad.sum()), "first at", i, float(got.reshape(-1)[i]), float(ref.reshape(-1)[i]),
                              float(tol.reshape(-1)[i])))
    r = err / tol.clamp_min(1e-300)
    return float(r.max()) if r.numel() else 0.0


def _tol32(terms, steps):
    return 2 * U * steps * torch.as_tensor(terms).double() + steps * 2.0 ** -149


def _tol_bf(ref, e32):
    """fp32 error e32 before the bf16 rounding of a result whose exact value is ref."""
    ref = torch.as_tensor(ref).double()
    return e32 * (1 + 2.0 ** -8) + 2.0 ** -8 * ref.abs() + 2.0 ** -133


def _not_rn(got_bf, ref):
    """Elements of a bf16 result that differ from RN_bf16(ref) (reported, not gated: the kernels round twice,
    fp32 then bf16, and the reference float64 -> fp32 -> bf16 can itself double-round)."""
    got = got_bf.detach().cpu().float().double()
    ref = torch.as_tensor(ref).double().cpu()
    rn = ref.float().to(BF16).double()
    return int(((got != rn) & ~((got == 0) & (rn == 0))).sum())


def _lanes(cgs, threads=KBN):
    return threads // cgs


# =============================================================================================== host checks
CHILD = r'''
import ctypes, sys
sys.path.insert(0, sys.argv[1] + "/unet-segment-pytorch_b200")
from unet import _C
lib = _C.lib()
P = 1 << 20                      # a 16-byte-aligned fake device address: the calls below must never use it
Q = P + 4                        # 4-byte aligned only
SIG = {name: _C.SIGNATURES[name] for name in """
ub2_bn_eval_coeffs ub2_bn_act ub2_bn_bwd_reduce ub2_bn_bwd_apply ub2_gate_upstats ub2_gate_psi ub2_gate_fused_eval
ub2_gate_apply ub2_gate_bwd_a ub2_gate_bwd_s ub2_gate_bwd_xg ub2_conv_in_fwd ub2_conv_in_wgrad ub2_outc_fwd
ub2_outc_bwd ub2_shuffle2x2_fwd ub2_shuffle2x2_bwd ub2_pack_convt_weight ub2_convt_wgrad_reduce""".split()}
N, H, W, C = 2, 8, 8, 16
bnr = lib.ub2_bn_bwd_rows(N, H, W, C, 1)
bnr0 = lib.ub2_bn_bwd_rows(N, H, W, C, 0)
strip = lib.ub2_gate_strip_rows(N, H, W, C)
gater = lib.ub2_gate_rows(N, H, W, 2 * C)
cinr = lib.ub2_conv_in_rows(N, H, W, C)
outr = lib.ub2_outc_rows(N, H, W, C)
shr = lib.ub2_shuffle2x2_rows(N, 4, 4, C, H, W)
assert min(bnr, bnr0, strip, gater, cinr, outr, shr) > 0
GEO = dict(N=N, hin=4, win=4, H=H, W=W, Ci=C)
BASE = {
 "ub2_bn_eval_coeffs": dict(eps=1e-5, C=C),
 "ub2_bn_act": dict(ld_y=C, ld_a=C, ld_p=C, N=N, H=H, W=W, C=C, relu=1),
 "ub2_bn_bwd_reduce": dict(ld_da=C, ld_dp=C, ld_y=C, rows=bnr, N=N, H=H, W=W, C=C, relu=1),
 "ub2_bn_bwd_apply": dict(ld_da=C, ld_dp=C, ld_y=C, ld_dy=C, N=N, H=H, W=W, C=C, relu=1),
 "ub2_gate_upstats": dict(ld_q=C, rows=strip, **GEO),
 "ub2_gate_psi": dict(ld_q=C, ld_xp=C, rows=strip, **GEO),
 "ub2_gate_fused_eval": dict(ld_q=C, ld_xp=C, ld_x=2 * C, ld_out=2 * C, Cx=2 * C, **GEO),
 "ub2_gate_apply": dict(ld_x=2 * C, ld_out=2 * C, N=N, H=H, W=W, Cx=2 * C),
 "ub2_gate_bwd_a": dict(ld_do=2 * C, ld_x=2 * C, ld_dx=2 * C, rows=gater, N=N, H=H, W=W, Cx=2 * C),
 "ub2_gate_bwd_s": dict(ld_q=C, ld_xp=C, ld_ds=C, rows=strip, **GEO),
 "ub2_gate_bwd_xg": dict(ld_ds=C, ld_xp=C, ld_q=C, ld_dxp=C, ld_dg=C, **GEO),
 "ub2_conv_in_fwd": dict(ld_y=C, rows=cinr, N=N, Cin=1, H=H, W=W, Cout=C),
 "ub2_conv_in_wgrad": dict(ld_dy=C, rows=cinr, N=N, Cin=1, H=H, W=W, Cout=C),
 "ub2_outc_fwd": dict(ld_a=C, N=N, H=H, W=W, C=C, K=2),
 "ub2_outc_bwd": dict(ld_a=C, ld_da=C, rows=outr, N=N, H=H, W=W, C=C, K=2),
 "ub2_shuffle2x2_fwd": dict(ld_t=4 * C, ld_out=C, N=N, h=4, w=4, C=C, Ho=H, Wo=W),
 "ub2_shuffle2x2_bwd": dict(ld_dout=C, ld_dt=4 * C, rows=shr, N=N, h=4, w=4, C=C, Ho=H, Wo=W),
 "ub2_pack_convt_weight": dict(Cin=C, Cout=C),
 "ub2_convt_wgrad_reduce": dict(splits=3, Cin=C, Cout=C, accumulate=1),
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
 # host crashes and silent launches before these checks
 ("ub2_conv_in_fwd", dict(Cout=0), S), ("ub2_conv_in_wgrad", dict(Cout=0), S), ("ub2_conv_in_fwd", dict(Cout=-8), S),
 ("ub2_gate_psi", dict(hin=0), S), ("ub2_gate_psi", dict(win=-1), S), ("ub2_gate_bwd_s", dict(hin=0), S),
 ("ub2_gate_bwd_xg", dict(win=0), S), ("ub2_gate_upstats", dict(hin=-2), S), ("ub2_gate_fused_eval", dict(hin=0), S),
 ("ub2_gate_apply", dict(H=0), S), ("ub2_gate_apply", dict(W=-1), S), ("ub2_gate_apply", dict(Cx=0, ld_x=0, ld_out=0), S),
 ("ub2_bn_bwd_apply", dict(ld_dy=12), S), ("ub2_bn_bwd_apply", dict(ld_dy=20), A),
 ("ub2_bn_bwd_reduce", dict(scale=None), S), ("ub2_bn_bwd_reduce", dict(shift=None), S),
 ("ub2_bn_bwd_apply", dict(scale=None), S), ("ub2_bn_bwd_apply", dict(shift=None), S),
 ("ub2_conv_in_fwd", dict(Cin=4, Cout=256, ld_y=256, W=9), S),            # weights + lanes over 48 KB
 ("ub2_conv_in_fwd", dict(Cout=1024, ld_y=1024, W=9), S),
 # counts
 ("ub2_bn_eval_coeffs", dict(C=0), S), ("ub2_bn_act", dict(N=0), S), ("ub2_bn_act", dict(H=0), S), ("ub2_bn_act", dict(W=-1), S),
 ("ub2_bn_act", dict(C=12, ld_y=16, ld_a=16, ld_p=16), S), ("ub2_bn_act", dict(C=2056, ld_y=2056, ld_a=2056, ld_p=2056), S),
 ("ub2_bn_bwd_reduce", dict(N=0), S), ("ub2_bn_bwd_reduce", dict(C=0), S), ("ub2_bn_bwd_apply", dict(H=-2), S),
 ("ub2_bn_bwd_apply", dict(C=2056, ld_da=2056, ld_dp=2056, ld_y=2056, ld_dy=2056), S),
 ("ub2_gate_psi", dict(N=0), S), ("ub2_gate_psi", dict(H=0), S), ("ub2_gate_psi", dict(Ci=0), S), ("ub2_gate_psi", dict(Ci=12), S),
 ("ub2_gate_psi", dict(Ci=520, ld_q=520, ld_xp=520), S), ("ub2_gate_bwd_s", dict(Ci=520, ld_q=520, ld_xp=520, ld_ds=520), S),
 ("ub2_gate_bwd_xg", dict(Ci=520, ld_ds=520, ld_xp=520, ld_q=520, ld_dxp=520, ld_dg=520), S),
 ("ub2_gate_fused_eval", dict(Ci=520, Cx=1040, ld_q=520, ld_xp=520, ld_x=1040, ld_out=1040), S),
 ("ub2_gate_fused_eval", dict(Cx=24), S), ("ub2_gate_bwd_a", dict(Cx=520, ld_do=520, ld_x=520, ld_dx=520), S),
 ("ub2_gate_bwd_a", dict(W=0), S), ("ub2_gate_bwd_xg", dict(N=-1), S), ("ub2_gate_apply", dict(Cx=12, ld_x=16, ld_out=16), S),
 ("ub2_gate_psi", dict(hin=20, H=8), S),                                 # down-sampling: no ring size
 ("ub2_gate_fused_eval", dict(Ci=384, Cx=768, ld_q=384, ld_xp=384, ld_x=768, ld_out=768, hin=8, win=8), S),  # ring > 200 KB
 ("ub2_gate_fused_eval", dict(Ci=264, Cx=528, ld_q=264, ld_xp=264, ld_x=528, ld_out=528, hin=8, win=8), S),
 ("ub2_gate_bwd_xg", dict(Ci=344, ld_ds=344, ld_xp=344, ld_q=344, ld_dxp=344, ld_dg=344, hin=8, win=8), S),
 ("ub2_conv_in_fwd", dict(N=0), S), ("ub2_conv_in_fwd", dict(H=-1), S), ("ub2_conv_in_fwd", dict(Cin=0), S),
 ("ub2_conv_in_fwd", dict(Cin=5), S), ("ub2_conv_in_fwd", dict(Cout=12, ld_y=16), S),
 ("ub2_conv_in_wgrad", dict(W=0), S), ("ub2_conv_in_wgrad", dict(Cin=5), S), ("ub2_conv_in_wgrad", dict(Cout=2056, ld_dy=2056), S),
 ("ub2_outc_fwd", dict(K=0), S), ("ub2_outc_fwd", dict(K=9), S), ("ub2_outc_fwd", dict(C=0), S), ("ub2_outc_fwd", dict(H=0), S),
 ("ub2_outc_bwd", dict(K=9), S), ("ub2_outc_bwd", dict(C=520, ld_a=520, ld_da=520), S), ("ub2_outc_bwd", dict(N=0), S),
 ("ub2_shuffle2x2_fwd", dict(h=0), S), ("ub2_shuffle2x2_fwd", dict(Ho=7), S), ("ub2_shuffle2x2_fwd", dict(C=12, ld_out=16, ld_t=48), S),
 ("ub2_shuffle2x2_bwd", dict(Wo=7), S), ("ub2_shuffle2x2_bwd", dict(N=0), S),
 ("ub2_shuffle2x2_bwd", dict(C=2056, ld_dout=2056, ld_dt=8224), S),
 ("ub2_pack_convt_weight", dict(Cin=0), S), ("ub2_pack_convt_weight", dict(Cout=-1), S),
 ("ub2_convt_wgrad_reduce", dict(splits=0), S), ("ub2_convt_wgrad_reduce", dict(Cin=0), S),
 # gradient sources
 ("ub2_bn_bwd_reduce", dict(dA=None, dP=None), S), ("ub2_bn_bwd_apply", dict(dA=None, dP=None), S),
 ("ub2_bn_bwd_reduce", dict(pidx=None), S), ("ub2_bn_bwd_apply", dict(pidx=None), S),
 ("ub2_shuffle2x2_bwd", dict(dbias=None), S), ("ub2_pack_convt_weight", dict(shift4=None), S),
 # channel strides below C
 ("ub2_bn_act", dict(ld_y=8), S), ("ub2_bn_act", dict(ld_a=8), S), ("ub2_bn_act", dict(ld_p=8), S),
 ("ub2_bn_bwd_reduce", dict(ld_da=8), S), ("ub2_bn_bwd_reduce", dict(ld_dp=8), S), ("ub2_bn_bwd_reduce", dict(ld_y=8), S),
 ("ub2_bn_bwd_apply", dict(ld_da=8), S), ("ub2_bn_bwd_apply", dict(ld_dp=8), S), ("ub2_bn_bwd_apply", dict(ld_y=8), S),
 ("ub2_gate_upstats", dict(ld_q=8), S), ("ub2_gate_psi", dict(ld_q=8), S), ("ub2_gate_psi", dict(ld_xp=8), S),
 ("ub2_gate_fused_eval", dict(ld_x=16), S), ("ub2_gate_fused_eval", dict(ld_out=24), S), ("ub2_gate_fused_eval", dict(ld_q=8), S),
 ("ub2_gate_apply", dict(ld_x=16), S), ("ub2_gate_apply", dict(ld_out=24), S), ("ub2_gate_bwd_a", dict(ld_do=16), S),
 ("ub2_gate_bwd_a", dict(ld_x=24), S), ("ub2_gate_bwd_a", dict(ld_dx=8), S), ("ub2_gate_bwd_s", dict(ld_ds=8), S),
 ("ub2_gate_bwd_s", dict(ld_xp=8), S), ("ub2_gate_bwd_xg", dict(ld_dg=8), S), ("ub2_gate_bwd_xg", dict(ld_dxp=8), S),
 ("ub2_gate_bwd_xg", dict(ld_ds=8), S), ("ub2_conv_in_fwd", dict(ld_y=8), S), ("ub2_conv_in_wgrad", dict(ld_dy=8), S),
 ("ub2_outc_fwd", dict(ld_a=8), S), ("ub2_outc_bwd", dict(ld_a=8), S), ("ub2_outc_bwd", dict(ld_da=8), S),
 ("ub2_shuffle2x2_fwd", dict(ld_t=56), S), ("ub2_shuffle2x2_fwd", dict(ld_out=8), S), ("ub2_shuffle2x2_bwd", dict(ld_dout=8), S),
 ("ub2_shuffle2x2_bwd", dict(ld_dt=56), S),
 # channel strides that are not multiples of 8
 ("ub2_bn_act", dict(ld_y=20), A), ("ub2_bn_act", dict(ld_a=20), A), ("ub2_bn_act", dict(ld_p=20), A),
 ("ub2_bn_bwd_reduce", dict(ld_da=20), A), ("ub2_bn_bwd_reduce", dict(ld_dp=20), A), ("ub2_bn_bwd_reduce", dict(ld_y=20), A),
 ("ub2_bn_bwd_apply", dict(ld_dp=20), A), ("ub2_gate_upstats", dict(ld_q=20), A), ("ub2_gate_psi", dict(ld_q=20), A),
 ("ub2_gate_psi", dict(ld_xp=20), A), ("ub2_gate_fused_eval", dict(ld_x=36), A), ("ub2_gate_apply", dict(ld_out=36), A),
 ("ub2_gate_bwd_a", dict(ld_do=36), A), ("ub2_gate_bwd_s", dict(ld_ds=20), A), ("ub2_gate_bwd_xg", dict(ld_dxp=20), A),
 ("ub2_conv_in_fwd", dict(ld_y=20), A), ("ub2_conv_in_wgrad", dict(ld_dy=20), A), ("ub2_outc_fwd", dict(ld_a=20), A),
 ("ub2_outc_bwd", dict(ld_da=20), A), ("ub2_shuffle2x2_fwd", dict(ld_t=68), A), ("ub2_shuffle2x2_bwd", dict(ld_dout=20), A),
 # pointers off the alignment of their accesses
 ("ub2_bn_act", dict(y=Q), A), ("ub2_bn_act", dict(a=Q), A), ("ub2_bn_act", dict(pooled=Q), A), ("ub2_bn_act", dict(pidx=Q), A),
 ("ub2_bn_bwd_reduce", dict(dA=Q), A), ("ub2_bn_bwd_reduce", dict(dP=Q), A), ("ub2_bn_bwd_reduce", dict(y=Q), A),
 ("ub2_bn_bwd_reduce", dict(pidx=Q), A), ("ub2_bn_bwd_reduce", dict(partials=Q), A), ("ub2_bn_bwd_apply", dict(dY=Q), A),
 ("ub2_bn_bwd_apply", dict(dA=Q), A), ("ub2_gate_upstats", dict(q=Q), A), ("ub2_gate_upstats", dict(partials=Q), A),
 ("ub2_gate_psi", dict(q=Q), A), ("ub2_gate_psi", dict(xp=Q), A), ("ub2_gate_psi", dict(psi_raw=P + 2), A),
 ("ub2_gate_psi", dict(partials=Q), A), ("ub2_gate_fused_eval", dict(x=Q), A), ("ub2_gate_fused_eval", dict(out=Q), A),
 ("ub2_gate_fused_eval", dict(q=Q), A), ("ub2_gate_apply", dict(x=Q), A), ("ub2_gate_apply", dict(out=Q), A),
 ("ub2_gate_apply", dict(a_out=P + 2), A), ("ub2_gate_bwd_a", dict(dout=Q), A), ("ub2_gate_bwd_a", dict(dx=Q), A),
 ("ub2_gate_bwd_a", dict(partials=Q), A), ("ub2_gate_bwd_s", dict(ds=Q), A), ("ub2_gate_bwd_s", dict(dpsin=P + 2), A),
 ("ub2_gate_bwd_xg", dict(dgup=Q), A), ("ub2_gate_bwd_xg", dict(xp=Q), A), ("ub2_conv_in_fwd", dict(y=Q), A),
 ("ub2_conv_in_fwd", dict(partials=Q), A), ("ub2_conv_in_fwd", dict(x=P + 2), A), ("ub2_conv_in_wgrad", dict(dy=Q), A),
 ("ub2_conv_in_wgrad", dict(partials=Q), A), ("ub2_outc_fwd", dict(a=Q), A), ("ub2_outc_fwd", dict(w=Q), A),
 ("ub2_outc_bwd", dict(a=Q), A), ("ub2_outc_bwd", dict(da=Q), A), ("ub2_outc_bwd", dict(partials=Q), A),
 ("ub2_shuffle2x2_fwd", dict(t=Q), A), ("ub2_shuffle2x2_fwd", dict(out=Q), A), ("ub2_shuffle2x2_bwd", dict(dt=Q), A),
 ("ub2_shuffle2x2_bwd", dict(partials=Q), A), ("ub2_convt_wgrad_reduce", dict(grad=P + 2), A),
 # workspace rows
 ("ub2_bn_bwd_reduce", dict(rows=bnr + 1), WS), ("ub2_bn_bwd_reduce", dict(dP=None, rows=bnr0 + 1), WS),
 ("ub2_gate_upstats", dict(rows=strip + 1), WS), ("ub2_gate_psi", dict(rows=strip + 1), WS),
 ("ub2_gate_bwd_a", dict(rows=gater - 1), WS), ("ub2_gate_bwd_s", dict(rows=strip - 1), WS),
 ("ub2_conv_in_fwd", dict(rows=cinr + 1), WS), ("ub2_conv_in_wgrad", dict(rows=cinr + 1), WS),
 ("ub2_outc_bwd", dict(rows=outr + 1), WS), ("ub2_shuffle2x2_bwd", dict(rows=shr + 1), WS),
]
# a NULL for every pointer the kernels dereference unconditionally
OPTIONAL = {"ub2_bn_eval_coeffs": {"gamma", "beta"}, "ub2_bn_act": {"scale", "shift", "a", "pooled", "pidx"},
            "ub2_bn_bwd_reduce": {"dA", "dP"}, "ub2_bn_bwd_apply": {"dA", "dP"}, "ub2_gate_psi": {"partials"},
            "ub2_gate_apply": {"a_out"}, "ub2_conv_in_fwd": {"partials"}, "ub2_outc_fwd": {"bias"},
            "ub2_outc_bwd": {"da", "dw", "db"}, "ub2_shuffle2x2_bwd": {"partials", "dbias"},
            "ub2_pack_convt_weight": {"bias", "fwd", "dg", "scale4", "shift4"}}
for name, args in SIG.items():
    for a, t in args:
        if t is ctypes.c_void_p and a != "stream" and a not in OPTIONAL.get(name, ()):
            BAD.append((name, {a: None}, S))
GOOD = [(name, {}) for name in SIG] + [
 # every NULL unet/kernels.py passes
 ("ub2_bn_act", dict(a=None)), ("ub2_bn_act", dict(pooled=None, pidx=None)), ("ub2_bn_act", dict(pidx=None)),
 ("ub2_bn_act", dict(scale=None, shift=None, relu=0, a=None)), ("ub2_bn_act", dict(scale=None, shift=None)),
 ("ub2_bn_bwd_reduce", dict(dP=None, pidx=None, rows=bnr0)), ("ub2_bn_bwd_reduce", dict(dA=None, ld_da=0)),
 ("ub2_bn_bwd_apply", dict(dP=None, pidx=None, ld_dp=0)), ("ub2_bn_bwd_apply", dict(dA=None, ld_da=0, relu=0)),
 ("ub2_bn_eval_coeffs", dict(gamma=None, beta=None)),
 ("ub2_gate_psi", dict(partials=None, rows=0)), ("ub2_gate_apply", dict(a_out=None)),
 ("ub2_conv_in_fwd", dict(partials=None, rows=0)), ("ub2_outc_fwd", dict(bias=None)), ("ub2_outc_bwd", dict(da=None, ld_da=0)),
 ("ub2_outc_bwd", dict(dw=None, db=None)), ("ub2_shuffle2x2_bwd", dict(partials=None, dbias=None, rows=0)),
 ("ub2_pack_convt_weight", dict(bias=None)), ("ub2_pack_convt_weight", dict(fwd=None, scale4=None, shift4=None)),
 # edges that are valid
 ("ub2_bn_act", dict(ld_y=24, ld_a=32, ld_p=40)), ("ub2_bn_act", dict(H=3, W=5)), ("ub2_bn_act", dict(H=1, W=1)),
 ("ub2_bn_act", dict(C=2048, ld_y=2048, ld_a=2048, ld_p=2048)), ("ub2_bn_act", dict(a=P + 16, pidx=P + 8)),
 ("ub2_bn_bwd_apply", dict(ld_dy=24, ld_y=32, ld_dp=24, ld_da=40)),
 ("ub2_gate_psi", dict(Ci=512, ld_q=512, ld_xp=512, rows=lib.ub2_gate_strip_rows(N, H, W, 512))),
 ("ub2_gate_psi", dict(hin=8, win=8)), ("ub2_gate_psi", dict(hin=1, win=1)), ("ub2_gate_psi", dict(ld_q=24, ld_xp=32)),
 ("ub2_gate_apply", dict(Cx=1024, ld_x=1024, ld_out=1032)), ("ub2_gate_bwd_a", dict(ld_do=40, ld_x=48)),
 ("ub2_gate_bwd_s", dict(ld_ds=24)), ("ub2_gate_bwd_xg", dict(ld_dg=24, ld_dxp=32)),
 ("ub2_gate_fused_eval", dict(Ci=384, Cx=768, ld_q=384, ld_xp=384, ld_x=768, ld_out=768)),
 ("ub2_gate_bwd_xg", dict(Ci=336, ld_ds=336, ld_xp=336, ld_q=336, ld_dxp=336, ld_dg=336, hin=8, win=8)),
 ("ub2_conv_in_fwd", dict(Cout=1024, ld_y=1024, rows=lib.ub2_conv_in_rows(N, H, W, 1024))),
 ("ub2_conv_in_fwd", dict(Cin=4, Cout=192, ld_y=200, W=9, rows=lib.ub2_conv_in_rows(N, H, 9, 192))),
 ("ub2_conv_in_fwd", dict(x=P + 4)), ("ub2_conv_in_wgrad", dict(Cin=4, W=7, rows=lib.ub2_conv_in_rows(N, H, 7, C))),
 ("ub2_outc_fwd", dict(C=512, ld_a=512, K=8)),
 ("ub2_outc_bwd", dict(C=512, ld_a=512, ld_da=520, K=8, rows=lib.ub2_outc_rows(N, H, W, 512))),
 ("ub2_shuffle2x2_fwd", dict(Ho=11, Wo=9, ld_t=72, ld_out=24)), ("ub2_convt_wgrad_reduce", dict(accumulate=0)),
]
for name, kw, want in BAD:
    rc = call(name, **kw)
    print(name, sorted(kw.items()), rc, want, "OK" if rc == want else "WRONG", flush=True)
for name, kw in GOOD:
    rc = call(name, **kw)
    print(name, "valid", sorted(kw.items()), rc, "positive", "OK" if rc > 0 else "WRONG", flush=True)
print("DONE", len(BAD), len(GOOD), flush=True)
'''


def test_bf16_entry_points_check_arguments_on_the_host():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")      # argument checks only, also on a GPU box
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, env=env)
    lines = r.stdout.strip().splitlines()
    assert r.returncode == 0 and lines and lines[-1].startswith("DONE"), (r.returncode, lines[-3:], r.stderr[-2000:])
    wrong = [l for l in lines if l.endswith("WRONG")]
    assert not wrong, wrong
    _, nbad, ngood = lines[-1].split()
    assert sum(l.endswith("OK") for l in lines) == int(nbad) + int(ngood) >= 300


# =============================================================================================== BatchNorm
BN_C = [8, 24, 40, 48, 64, 72, 128, 384, 1024]
BN_SHAPES = [(2, 7, 9), (1, 8, 6), (3, 1, 1), (2, 2, 2)]


@GPU
@pytest.mark.parametrize("C", BN_C)
def test_bn_eval_coeffs(C):
    """1/sqrtf(rv + eps) (3 roundings), scale = g * inv (4), shift = beta - rm * g * inv (7, with its terms)."""
    g = _gen(C)
    gamma, beta, rm, rv = _randn((C,), g, 0.5, 1.0), _randn((C,), g), _randn((C,), g), _randn((C,), g).abs() + 0.1
    eps = 1e-5
    ec = Guarded((2, C))
    _call("ub2_bn_eval_coeffs", _p(gamma.cuda()), _p(beta.cuda()), _p(rm.cuda()), _p(rv.cuda()), eps, C,
          _p(ec.t[0]), _p(ec.t[1]), _s())
    assert ec.ok()
    g64, b64, rm64 = gamma.double(), beta.double(), rm.double()
    iv = 1 / (rv.double() + torch.tensor(eps, dtype=F32).double()).sqrt()
    got = ec.t.cpu()
    e = max(_check(got[0], g64 * iv, _tol32((g64 * iv).abs(), 4), "eval scale"),
            _check(got[1], b64 - rm64 * g64 * iv, _tol32(b64.abs() + (rm64 * g64 * iv).abs() * 4, 7), "eval shift"))
    record(f"bf16 kernels bn_eval_coeffs C{C}", worst_over_bound=e)


def _bn_inputs(N, H, W, C, ld, g):
    """y (bf16, channel slice of width ld) with ties and signed zeros planted, scale / shift fp32."""
    y = _rand_bf((N, H, W, ld), g, 1.5, 0.2).float()
    tie = torch.tensor([-1.0, -0.0, 0.0, 1.0, 0.5])
    sel = torch.rand((N, H, W, ld), generator=g) < 0.4
    y[sel] = tie[torch.randint(0, 5, (int(sel.sum()),), generator=g)]
    y = y.to(BF16)
    sc = _randn((C,), g, 0.7, 0.0)
    sc[::3] = -sc[::3].abs()                                 # negative scales flip the mask
    sh = _randn((C,), g, 0.5)
    return y, sc, sh


def _pool_ref(a_bf):
    """First-maximum 2x2 pool of the kernel's own a (strict >, -0 == +0): values (bits of the selected element)
    and window positions, over complete windows only."""
    N, H, W, C = a_bf.shape
    Hp, Wp = H // 2, W // 2
    v = a_bf[:, :2 * Hp, :2 * Wp].float()
    bits = a_bf[:, :2 * Hp, :2 * Wp].contiguous().view(torch.int16)
    win = [v[:, r::2, c::2] for r in (0, 1) for c in (0, 1)]
    wbits = [bits[:, r::2, c::2] for r in (0, 1) for c in (0, 1)]
    mx = torch.full_like(win[0], -float("inf"))
    arg = torch.zeros_like(win[0], dtype=torch.uint8)
    sel = wbits[0].clone()
    for d in range(4):
        take = win[d] > mx
        mx = torch.where(take, win[d], mx)
        arg = torch.where(take, torch.full_like(arg, d), arg)
        sel = torch.where(take, wbits[d], sel)
    return sel, arg


@GPU
@pytest.mark.parametrize("C", BN_C)
@pytest.mark.parametrize("N,H,W", BN_SHAPES)
def test_bn_act(C, N, H, W):
    """Every combination of relu, pool, a == NULL and scale/shift == NULL (among them ops.py's pool-only call:
    relu off, no coefficients); odd H / W leave edge windows unpooled; y, a and pooled with channel strides above C."""
    g = _gen(C * 100 + H * 10 + W)
    ld_y, ld_a, ld_p = C + 8, C + 16, C + 8
    y, sc, sh = _bn_inputs(N, H, W, C, ld_y, g)
    yd, scd, shd = _slice(y, C), sc.cuda(), sh.cuda()
    ys = y[..., :C].double()
    Hp, Wp = H // 2, W // 2
    log, not_rn = {}, 0
    a_of = {}
    for relu in (1, 0):
        for coef in (True, False):
            s_, h_ = (sc.double(), sh.double()) if coef else (torch.ones(C, dtype=F64), torch.zeros(C, dtype=F64))
            z = ys * s_ + h_                                 # exact sign; float64 of an exact product
            ref = z.clamp_min(0) if relu else z
            for pool in (0, 1):
                for write_a in (True, False):
                    a = Out((N, H, W), C, ld_a) if write_a else None
                    p = Out((N, Hp, Wp), C, ld_p) if pool else None
                    idx = Guarded((N, Hp, Wp, C), torch.uint8) if pool else None
                    _call("ub2_bn_act", _p(yd), ld_y, _p(scd) if coef else _p(None), _p(shd) if coef else _p(None),
                          _p(a.t) if a else _p(None), ld_a, _p(p.t) if p else _p(None), ld_p,
                          _p(idx.t) if idx else _p(None), N, H, W, C, relu, _s())
                    what = f"relu{relu} coef{int(coef)} pool{pool} a{int(write_a)}"
                    assert (a is None or a.ok()) and (p is None or p.ok()) and (idx is None or idx.ok()), what
                    if a is not None:
                        got = a.t.cpu()
                        key = (relu, coef)
                        if key in a_of:
                            assert torch.equal(_bits(got), _bits(a_of[key])), ("a differs between launches", what)
                        a_of[key] = got
                        if relu:       # the mask is exact: zero exactly where y*scale + shift <= 0
                            assert torch.equal(got.double() != 0, z > 0), ("relu mask", what)
                        e32 = _tol32(z.abs(), 1)
                        log[f"a {what}"] = _check(got, ref, _tol_bf(ref, e32), ("a", what))
                        not_rn += _not_rn(got, ref)
                        if not coef and not relu:        # the identity, up to the sign of zero (fmaf(-0, 1, 0) = +0)
                            assert torch.equal(got.float(), y[..., :C].float())
                    if p is not None:
                        sel, arg = _pool_ref(a_of[(relu, coef)])   # a from this launch or its twin that wrote a
                        assert torch.equal(p.t.cpu().contiguous().view(torch.int16), sel), ("pooled bits", what)
                        assert torch.equal(idx.t.cpu(), arg), ("pidx", what, int((idx.t.cpu() != arg).sum()))
    record(f"bf16 kernels bn_act {N}x{H}x{W}x{C}", not_rn_bf16=not_rn, **log)


BWD_SRC = ["dA", "dP", "both"]


@GPU
@pytest.mark.parametrize("C", BN_C)
@pytest.mark.parametrize("src", BWD_SRC)
def test_bn_backward(C, src):
    """bn_bwd_reduce (rows of sum g, sum g*y) and bn_bwd_apply (dy = A g + B y + C) with g = (dA + dP routed
    through pidx) * [y*scale + shift > 0]; frozen (B = C = 0) and batch coefficients built in float64 here; dA / dP
    / y / dy with channel strides above C.  With dP alone: also the identity-coefficient call of
    kernels.maxpool_bwd, bit for bit."""
    N, H, W = 2, 7, 9
    g = _gen(C * 7 + len(src))
    ld_y, ld_da, ld_dp, ld_dy = C + 8, C + 16, C + 8, C + 24
    y, sc, sh = _bn_inputs(N, H, W, C, ld_y, g)
    dA = _rand_bf((N, H, W, ld_da), g) if src in ("dA", "both") else None
    dP = _rand_bf((N, H // 2, W // 2, ld_dp), g) if src in ("dP", "both") else None
    pidx = torch.randint(0, 4, (N, H // 2, W // 2, C), generator=g, dtype=torch.uint8) if dP is not None else None
    yd, scd, shd = _slice(y, C), sc.cuda(), sh.cuda()
    dAd = _slice(dA, C) if dA is not None else None
    dPd = _slice(dP, C) if dP is not None else None
    pd = pidx.cuda() if pidx is not None else None
    pool = int(dP is not None)
    rows = _rows("ub2_bn_bwd_rows", N, H, W, C, pool)
    ys = y[..., :C].double()
    live = (ys * sc.double() + sh.double()) > 0
    gin = _routed(dA[..., :C] if dA is not None else None, dP[..., :C] if dP is not None else None, pidx, N, H, W, C)
    gz = gin * live
    # the reduce
    parts = []
    for _ in range(2):
        pg = Guarded((rows, 2, C), F64)
        _call("ub2_bn_bwd_reduce", _p(dAd), ld_da, _p(dPd), ld_dp, _p(pd), _p(yd), ld_y, _p(scd), _p(shd), _p(pg.t), rows,
              N, H, W, C, 1, _s())
        assert pg.ok()
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]), "not repeatable"
    lanes = _lanes(C // 8)
    items = N * ((H + 1) // 2) * ((W + 1) // 2) if pool else N * H * W
    k = _per_thread(items, rows * lanes) * (4 if pool else 1) + 1     # sequential fp32 adds per thread + the dA+dP add
    s = _folded(parts[0])
    log = {"sum g": _check(s[0], gz.sum((0, 1, 2)), _tol32(gz.abs().sum((0, 1, 2)), k), "sum g"),
           "sum g y": _check(s[1], (gz * ys).sum((0, 1, 2)), _tol32((gz * ys).abs().sum((0, 1, 2)), k + 1), "sum g*y")}
    not_rn = 0
    for frozen in (True, False):
        A = (_randn((C,), g, 0.5, 1.0)).double()
        B = torch.zeros(C, dtype=F64) if frozen else _randn((C,), g, 0.3).double()
        Cc = torch.zeros(C, dtype=F64) if frozen else _randn((C,), g, 0.3).double()
        coef = torch.stack([A, B, Cc]).float()
        A, B, Cc = coef.double()
        dy = Out((N, H, W), C, ld_dy)
        _call("ub2_bn_bwd_apply", _p(dAd), ld_da, _p(dPd), ld_dp, _p(pd), _p(yd), ld_y, _p(scd), _p(shd), _p(coef.cuda()),
              _p(dy.t), ld_dy, N, H, W, C, 1, _s())
        assert dy.ok()
        ref = A * gz + B * ys + Cc
        terms = (A * gz).abs() + (B * ys).abs() + Cc.abs()
        log[f"dy frozen={frozen}"] = _check(dy.t.cpu(), ref, _tol_bf(ref, _tol32(terms, 3)), ("dy", frozen))
        not_rn += _not_rn(dy.t.cpu(), ref)
    if src == "dP":
        # kernels.maxpool_bwd: relu off, scale 1, shift 0, coefficients (1, 0, 0): dy is the routed dP, exactly
        ident = torch.zeros((5, C), device="cuda")
        ident[0] = 1.0
        ident[2] = 1.0
        dy = Out((N, H, W), C, C)
        _call("ub2_bn_bwd_apply", _p(None), 0, _p(dPd), ld_dp, _p(pd), _p(yd), ld_y, _p(ident[0]), _p(ident[1]),
              _p(ident[2]), _p(dy.t), C, N, H, W, C, 0, _s())
        assert dy.ok()
        assert torch.equal(_bits(dy.t.cpu()), _bits(gin.to(BF16)))
    record(f"bf16 kernels bn_backward C{C} {src}", not_rn_bf16=not_rn, **log)


# =============================================================================================== attention gate
def _gate_geom(Ci):
    cgs = Ci // 8
    tpp = 1
    while tpp < cgs and tpp < 32:
        tpp *= 2
    G = -(-cgs // tpp)
    return tpp, G, KGATE // tpp


GATE_CI = [8, 24, 40, 64, 192, 256, 384, 512]
# (N, hin, win, H, W) as a function of the strip kernels' column tile `slots`
GATE_GEOMS = {
    "8x8->16x16 N2": lambda s: (2, 8, 8, 16, 16),             # 2x: QR = 4, H a multiple of the strip
    "6x5->13x9": lambda s: (1, 6, 5, 13, 9),                  # QR = 4, H not a multiple of 16
    "16->17 W>slots": lambda s: (2, 16, s // 2 + 3, 17, s + 5),   # QR = 8, two column tiles, N > 1
    "12x12->12x12": lambda s: (1, 12, 12, 12, 12),            # QR = 8
    "1x1": lambda s: (3, 1, 1, 1, 1),
    "1x1->2x2": lambda s: (2, 1, 1, 2, 2),
}


def _up_ref(q, H, W):
    """q (N,hin,win,C) bf16 -> up (N,H,W,C) float64 with the kernels' fp32 taps, and sum |taps * q|."""
    Mh, Mw = _lerp_rows(H, q.shape[1]), _lerp_rows(W, q.shape[2])
    q64 = q.double()
    up = torch.einsum("ai,bj,nijc->nabc", Mh, Mw, q64)
    up_t = torch.einsum("ai,bj,nijc->nabc", Mh.abs(), Mw.abs(), q64.abs())
    return up, up_t


def _sig_err(z, ez):
    """|a - sigmoid(z)| bound for a = 1 / (1 + __expf(-z_k)), |z_k - z| <= ez."""
    a = torch.sigmoid(z)
    rel_e = (2 + torch.floor(1.16 * z.abs())) * 2.0 ** -23
    return a, a * (1 - a) * (ez + rel_e) * 1.01 + 3 * 2 * U * a


@GPU
@pytest.mark.parametrize("Ci", GATE_CI)
@pytest.mark.parametrize("geom", list(GATE_GEOMS))
def test_gate_passes(Ci, geom):
    """gate_psi (with and without statistics) -> gate_apply (with and without a_out) and gate_fused_eval against
    float64; gate_bwd_a, gate_bwd_s and gate_bwd_xg on the forward's outputs against float64 of their own formulas
    (coefficients built here, so the already-tested finalizes are not in the loop)."""
    tpp, G, slots = _gate_geom(Ci)
    N, hin, win, H, W = GATE_GEOMS[geom](slots)
    Cx = 2 * Ci
    px = N * H * W
    g = _gen(Ci * 1000 + H * 7 + W)
    ld_q, ld_xp, ld_x = Ci + 8, Ci + 16, Cx + 8
    q, xp = _rand_bf((N, hin, win, ld_q), g), _rand_bf((N, H, W, ld_xp), g)
    x = _rand_bf((N, H, W, ld_x), g)
    sg, hg = _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5)
    sx, hx = _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.5)
    wpsi = _randn((Ci,), g, 1 / math.sqrt(Ci))
    spsi, hpsi = torch.tensor([0.9]), torch.tensor([-0.1])
    qd, xpd, xd = _slice(q, Ci), _slice(xp, Ci), _slice(x, Cx)
    sgd, hgd, sxd, hxd, wd, spd, hpd = (t.cuda() for t in (sg, hg, sx, hx, wpsi, spsi, hpsi))
    log, not_rn = {}, 0
    # float64 forward
    up, up_t = _up_ref(q[..., :Ci], H, W)
    e_u = 2 * U * 4 * up_t                                       # two lerps of two fp32 roundings each
    x64, xp64 = x[..., :Cx].double(), xp[..., :Ci].double()
    sg6, hg6, sx6, hx6, w6 = (t.double() for t in (sg, hg, sx, hx, wpsi))
    t = up * sg6 + xp64 * sx6 + hg6 + hx6
    e_t = 2 * U * 3 * ((up * sg6).abs() + (xp64 * sx6).abs() + hg6.abs() + hx6.abs()) + sg6.abs() * e_u
    e_t = e_t * 1.01
    und = t.abs() <= e_t                                         # undecided ReLU
    log["undecided relu"] = int(und.sum())
    psi_ref = (w6 * t.clamp_min(0)).sum(-1)
    steps_dot = 8 * G + int(math.log2(tpp))
    e_psi = (2 * U * steps_dot * (w6.abs() * (t.clamp_min(0) + e_t)).sum(-1) + (w6.abs() * e_t).sum(-1)
             + (w6.abs() * t.abs() * und).sum(-1))
    # gate_psi
    rows = _rows("ub2_gate_strip_rows", N, H, W, Ci)
    psis, parts = [], []
    for stats in (True, True, False):
        psi = Guarded((N, H, W))
        pg = Guarded((rows, 2, 1), F64) if stats else None
        _call("ub2_gate_psi", _p(qd), ld_q, _p(xpd), ld_xp, _p(sgd), _p(hgd), _p(sxd), _p(hxd), _p(wd), _p(psi.t),
              _p(pg.t) if pg else _p(None), rows, N, hin, win, H, W, Ci, _s())
        assert psi.ok() and (pg is None or pg.ok())
        psis.append(psi.t.cpu())
        if pg:
            parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(psis[0], psis[1]) and torch.equal(psis[0], psis[2])
    psi32 = psis[0]
    log["psi"] = _check(psi32, psi_ref, e_psi, "psi")
    p64 = psi32.double()
    sp = _folded(parts[0]).view(-1)
    k_st = min(STRIP, H) + 5 + 1                                 # rows of the strip, the warp tree, the fma
    log["psi stats"] = max(_check(sp[0], p64.sum(), _tol32(p64.abs().sum(), k_st), "sum psi"),
                           _check(sp[1], (p64 * p64).sum(), _tol32((p64 * p64).sum(), k_st), "sum psi^2"))
    # gate_apply on the kernel's psi: z = fmaf(psi, s, h) exact in float64 up to one rounding
    z = p64 * spsi.double() + hpsi.double()
    a_ref, e_a = _sig_err(z, 2 * U * ((p64 * spsi.double()).abs() + hpsi.double().abs()))
    psid = psi32.cuda()
    outs = []
    for with_a in (True, False):
        out = Out((N, H, W), Cx, Cx + 16)
        a_out = Guarded((N, H, W)) if with_a else None
        _call("ub2_gate_apply", _p(psid), _p(spd), _p(hpd), _p(xd), ld_x, _p(out.t), Cx + 16,
              _p(a_out.t) if a_out else _p(None), N, H, W, Cx, _s())
        assert out.ok() and (a_out is None or a_out.ok())
        outs.append(out.t.cpu())
        if a_out:
            a32 = a_out.t.cpu()
    assert torch.equal(_bits(outs[0]), _bits(outs[1]))
    log["a"] = _check(a32, a_ref, e_a, "a")
    ref = x64 * a_ref.unsqueeze(-1)
    e_out = x64.abs() * e_a.unsqueeze(-1) + 2 * U * ref.abs()
    log["apply out"] = _check(outs[0], ref, _tol_bf(ref, e_out), "apply out")
    not_rn += _not_rn(outs[0], ref)
    # gate_fused_eval against float64 (psi's own error enters z); at two channel groups per thread its 8-row ring
    # does not fit the shared memory of a block, and the entry point refuses the shape before the launch
    rh = np.float32(hin - 1) / np.float32(H - 1) if H > 1 else np.float32(0)
    qr8 = int(3 * float(rh) + 1e-4) + 3 > 4                      # gate.cu:strip_qr
    fo = Out((N, H, W), Cx, Cx + 8)
    args = (_p(qd), ld_q, _p(xpd), ld_xp, _p(xd), ld_x, _p(sgd), _p(hgd), _p(sxd), _p(hxd), _p(wd), _p(spd), _p(hpd), _p(fo.t),
            Cx + 8, N, hin, win, H, W, Ci, Cx, _s())
    if G == 2 and qr8:
        with pytest.raises(RuntimeError, match=r"code -1"):
            _call("ub2_gate_fused_eval", *args)
        assert fo.ok() and bool(torch.isnan(fo.t.float()).all())
    else:
        _call("ub2_gate_fused_eval", *args)
        assert fo.ok()
        zr = psi_ref * spsi.double() + hpsi.double()
        af, e_af = _sig_err(zr, spsi.double().abs() * e_psi + 2 * U * ((psi_ref * spsi.double()).abs() + hpsi.double().abs()))
        reff = x64 * af.unsqueeze(-1)
        log["fused out"] = _check(fo.t.cpu(), reff, _tol_bf(reff, x64.abs() * e_af.unsqueeze(-1) + 2 * U * reff.abs()), "fused")
        log["fused vs two-pass differing elements"] = int((_bits(fo.t.cpu()) != _bits(outs[0])).sum())
    # gate_bwd_a (Cx up to the kernel's 512 channels)
    Cb = Cx if Cx <= 512 else Ci
    ld_do = Cb + 8
    dout = _rand_bf((N, H, W, ld_do), g)
    rows_a = _rows("ub2_gate_rows", N, H, W, Cb)
    tpp_b, G_b, slots_b = _gate_geom(Cb)
    a32d = a32.cuda()
    dpsins, parts = [], []
    for _ in range(2):
        dx, dpsin, pg = Out((N, H, W), Cb, Cb + 8), Guarded((N, H, W)), Guarded((rows_a, 2, 1), F64)
        _call("ub2_gate_bwd_a", _p(_slice(dout, Cb)), ld_do, _p(xd), ld_x, _p(a32d), _p(psid), _p(dx.t), Cb + 8, _p(dpsin.t),
              _p(pg.t), rows_a, N, H, W, Cb, _s())
        assert dx.ok() and dpsin.ok() and pg.ok()
        dpsins.append(dpsin.t.cpu())
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(dpsins[0], dpsins[1])
    a64 = a32.double()
    d64, xb = dout[..., :Cb].double(), x[..., :Cb].double()
    dot, dot_t = (d64 * xb).sum(-1), (d64 * xb).abs().sum(-1)
    w_a = a64 * (1 - a64)
    steps_a = 8 * G_b + int(math.log2(tpp_b))
    log["dpsin"] = _check(dpsins[0], dot * w_a, (_tol32(dot_t, steps_a) + _tol32(dot.abs(), 3)) * w_a, "dpsin")
    refdx = d64 * a64.unsqueeze(-1)
    log["dx"] = _check(dx.t.cpu(), refdx, _tol_bf(refdx, _tol32(refdx.abs(), 1)), "dx")
    not_rn += _not_rn(dx.t.cpu(), refdx)
    dn = dpsins[0].double()
    s = _folded(parts[0]).view(-1)
    k_a = _per_thread(px, rows_a * slots_b) + 5 + 1
    log["bwd_a rows"] = max(_check(s[0], dn.sum(), _tol32(dn.abs().sum(), k_a), "sum dn"),
                            _check(s[1], (dn * p64).sum(), _tol32((dn * p64).abs().sum(), k_a), "sum dn psi"))
    # gate_bwd_s: BN_psi backward coefficients chosen here
    cpsi = torch.tensor([1.3, -0.4, 0.05])
    dpsind = dpsins[0].cuda()
    c6 = cpsi.double()
    dpr = c6[0] * dn + c6[1] * p64 + c6[2]
    e_dpr = _tol32((c6[0] * dn).abs() + (c6[1] * p64).abs() + c6[2].abs(), 2)
    d_live = dpr.unsqueeze(-1) * w6
    e_d = e_dpr.unsqueeze(-1) * w6.abs() + 2 * U * d_live.abs()
    live = (t > 0).double()
    d_ref = d_live * live
    ld_ds = Ci + 8
    dss, parts = [], []
    for _ in range(2):
        ds, pg = Out((N, H, W), Ci, ld_ds), Guarded((rows, 4, Ci), F64)
        _call("ub2_gate_bwd_s", _p(dpsind), _p(psid), _p(cpsi.cuda()), _p(qd), ld_q, _p(xpd), ld_xp, _p(sgd), _p(hgd), _p(sxd),
              _p(hxd), _p(wd), _p(ds.t), ld_ds, _p(pg.t), rows, N, hin, win, H, W, Ci, _s())
        assert ds.ok() and pg.ok()
        dss.append(ds.t)
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(_bits(dss[0].cpu()), _bits(dss[1].cpu()))
    ds_cpu = dss[0].cpu().double()
    tol_ds = _tol_bf(d_ref, e_d)
    either = und & ((ds_cpu == 0) | ((ds_cpu - d_live).abs() <= _tol_bf(d_live, e_d)))
    log["ds"] = _check(torch.where(either, d_ref, ds_cpu), d_ref, tol_ds, "ds")
    not_rn += _not_rn(dss[0].cpu()[~und], d_ref[~und])
    k_s = min(STRIP, H) + 1
    s4 = _folded(parts[0])
    ud = und.double()
    dl_abs = d_live.abs()
    log["bwd_s rows"] = max(
        _check(s4[0], d_ref.sum((0, 1, 2)), (_tol32(d_ref.abs(), k_s) + e_d + dl_abs * ud).sum((0, 1, 2)), "sum ds"),
        _check(s4[1], (d_ref * xp64).sum((0, 1, 2)),
               ((_tol32(d_ref.abs(), k_s + 1) + e_d + dl_abs * ud) * xp64.abs()).sum((0, 1, 2)), "sum ds xp"),
        _check(s4[2], (d_ref * up).sum((0, 1, 2)),
               ((_tol32(d_ref.abs(), k_s + 1) + e_d + dl_abs * ud) * (up.abs() + e_u) + dl_abs * e_u).sum((0, 1, 2)), "sum ds up"),
        _check(s4[3], (dpr.unsqueeze(-1) * t.clamp_min(0)).sum((0, 1, 2)),
               (_tol32((dpr.unsqueeze(-1) * t.clamp_min(0)).abs(), k_s + 1)
                + (dpr.abs().unsqueeze(-1) + e_dpr.unsqueeze(-1)) * e_t
                + e_dpr.unsqueeze(-1) * t.clamp_min(0)).sum((0, 1, 2)), "sum dpsi relu(t)"))
    # gate_bwd_xg on the kernel's ds (a channel slice: stride ld_ds)
    coef = torch.stack([_randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.1), _randn((Ci,), g, 0.1),
                        _randn((Ci,), g, 0.5, 1.0), _randn((Ci,), g, 0.1), _randn((Ci,), g, 0.1)])
    cf = coef.double()
    dxp, dgup = Out((N, H, W), Ci, Ci + 8), Out((N, H, W), Ci, Ci + 16)
    args = (_p(dss[0]), ld_ds, _p(xpd), ld_xp, _p(qd), ld_q, _p(coef.cuda()), _p(dxp.t), Ci + 8, _p(dgup.t), Ci + 16, N, hin, win,
            H, W, Ci, _s())
    if qr8 and Ci > 336:          # 8-row ring of two channel groups + 6 Ci coefficients over 200 KB: refused
        with pytest.raises(RuntimeError, match=r"code -1"):
            _call("ub2_gate_bwd_xg", *args)
        assert dxp.ok() and dgup.ok()
        record(f"bf16 kernels gate Ci{Ci} {geom}", not_rn_bf16=not_rn, **log)
        return
    _call("ub2_gate_bwd_xg", *args)
    assert dxp.ok() and dgup.ok()
    r1 = cf[0] * ds_cpu + cf[1] * xp64 + cf[2]
    t1 = (cf[0] * ds_cpu).abs() + (cf[1] * xp64).abs() + cf[2].abs()
    r2 = cf[3] * ds_cpu + cf[4] * up + cf[5]
    t2 = (cf[3] * ds_cpu).abs() + (cf[4] * up).abs() + cf[5].abs()
    log["dxp"] = _check(dxp.t.cpu(), r1, _tol_bf(r1, _tol32(t1, 2)), "dxp")
    log["dgup"] = _check(dgup.t.cpu(), r2, _tol_bf(r2, _tol32(t2, 2) + cf[4].abs() * e_u), "dgup")
    not_rn += _not_rn(dxp.t.cpu(), r1)
    record(f"bf16 kernels gate Ci{Ci} {geom}", not_rn_bf16=not_rn, **log)


# =============================================================================================== stem convolution
CONV_IN = [  # Cin, Cout, N, H, W, x offset (elements): which forward / weight-gradient variant runs
    (1, 64, 2, 8, 16, 0), (1, 1024, 1, 3, 8, 0), (1, 24, 2, 5, 12, 0),            # Cin 1, W % 4 == 0, x aligned: *4 kernels
    (1, 40, 2, 7, 9, 0), (1, 72, 1, 6, 8, 1), (1, 384, 1, 2, 3, 0), (1, 8, 3, 1, 1, 0),   # Cin 1, general
    (2, 8, 2, 9, 7, 0), (3, 48, 1, 8, 8, 0), (4, 128, 2, 5, 6, 0), (4, 192, 1, 4, 5, 1)]  # Cin 2-4


@GPU
@pytest.mark.parametrize("Cin,Cout,N,H,W,off", CONV_IN)
def test_conv_in(Cin, Cout, N, H, W, off):
    """conv_in_fwd (y bf16 with a channel stride above Cout; with and without statistics rows, which sum the
    bf16-rounded y) and conv_in_wgrad (+= into an existing gradient) against float64 conv2d / conv2d_weight."""
    g = _gen(Cin * 10000 + Cout + H * 10 + W + off)
    xf = _randn((N * Cin * H * W + off,), g)
    w = _randn((Cout, Cin, 3, 3), g, 1 / math.sqrt(9 * Cin))
    xbuf = xf.cuda()
    xd = xbuf[off:].view(N, Cin, H, W)
    x64, w64 = xf[off:].view(N, Cin, H, W).double(), w.double()
    ref = F.conv2d(x64, w64, padding=1).permute(0, 2, 3, 1)
    terms = F.conv2d(x64.abs(), w64.abs(), padding=1).permute(0, 2, 3, 1)
    rows = _rows("ub2_conv_in_rows", N, H, W, Cout)
    ld_y = Cout + 8
    ys, parts = [], []
    for stats in (True, True, False):
        y = Out((N, H, W), Cout, ld_y)
        pg = Guarded((rows, 2, Cout), F64) if stats else None
        _call("ub2_conv_in_fwd", _p(xd), _p(w.cuda()), _p(y.t), ld_y, _p(pg.t) if pg else _p(None), rows, N, Cin, H, W, Cout, _s())
        assert y.ok() and (pg is None or pg.ok())
        ys.append(y.t.cpu())
        if pg:
            parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and all(torch.equal(_bits(ys[0]), _bits(v)) for v in ys[1:])
    log = {"y": _check(ys[0], ref, _tol_bf(ref, _tol32(terms, 9 * Cin)), "y"), "y not_rn_bf16": _not_rn(ys[0], ref)}
    cgs = Cout // 8
    lanes = KGATE // cgs
    four = Cin == 1 and W % 4 == 0 and off % 4 == 0
    per_row = 4 * _per_thread(W, 4 * lanes) if four else _per_thread(W, lanes)
    k = _per_thread(N * H, rows) * per_row                # pixels one thread folds in fp32
    yk = ys[0].double()
    s = _folded(parts[0])
    log["stats"] = max(_check(s[0], yk.sum((0, 1, 2)), _tol32(yk.abs().sum((0, 1, 2)), k), "sum y"),
                       _check(s[1], (yk * yk).sum((0, 1, 2)), _tol32((yk * yk).sum((0, 1, 2)), k + 1), "sum y^2"))
    # weight gradient, accumulating into g0
    dyf = _rand_bf((N, H, W, Cout + 16), g)
    dyd = _slice(dyf, Cout)
    g0 = _randn((Cout, Cin, 3, 3), g)
    grads, parts = [], []
    for _ in range(2):
        grad = Guarded((Cout, Cin, 3, 3), fill=g0.cuda())
        pg = Guarded((rows, Cin, 9, Cout), F64)
        _call("ub2_conv_in_wgrad", _p(xd), _p(dyd), Cout + 16, _p(pg.t), rows, _p(grad.t), N, Cin, H, W, Cout, _s())
        assert grad.ok() and pg.ok()
        grads.append(grad.t.cpu())
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(grads[0], grads[1])
    dy64 = dyf[..., :Cout].double().permute(0, 3, 1, 2)
    gr = torch.nn.grad.conv2d_weight(x64, w64.shape, dy64, padding=1)
    gt = torch.nn.grad.conv2d_weight(x64.abs(), w64.shape, dy64.abs(), padding=1)
    kw = (4 * _per_thread(N * H * (W // 4), rows * lanes) if four else _per_thread(N * H * W, rows * lanes)) + 1
    log["wgrad"] = _check(grads[0], g0.double() + gr, _tol32(g0.double().abs() + gt * kw, 1), "wgrad")
    record(f"bf16 kernels conv_in Cin{Cin} Cout{Cout} {N}x{H}x{W} off{off}", **log)


# =============================================================================================== output head
@GPU
@pytest.mark.parametrize("K", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("C", [8, 24, 64, 384, 512])
def test_outc(K, C):
    """outc_fwd (bias optional) and outc_bwd (da optional; dw and db accumulate into non-zero tensors) against
    float64; all three KMAX instances, one and two channel groups per thread, a channel stride above C."""
    N, H, W = 2, 9, 11
    px = N * H * W
    g = _gen(K * 1000 + C)
    ld_a = C + 8
    af = _rand_bf((N, H, W, ld_a), g)
    w, b = _randn((K, C), g, 1 / math.sqrt(C)), _randn((K,), g)
    dl = _randn((N, K, H, W), g)
    dw0, db0 = _randn((K, C), g), _randn((K,), g)
    ad, wd, dld = _slice(af, C), w.cuda(), dl.cuda()
    a64, w64, dl64 = af[..., :C].double(), w.double(), dl.double().permute(0, 2, 3, 1)
    cgs = C // 8
    tpp = 1
    while tpp < cgs and tpp < 32:
        tpp *= 2
    G = -(-cgs // tpp)
    log = {}
    steps = 8 * G + int(math.log2(tpp)) + 1
    for bias in (b, None):
        lg = Guarded((N, K, H, W))
        _call("ub2_outc_fwd", _p(ad), ld_a, _p(wd), _p(bias.cuda() if bias is not None else None), _p(lg.t), N, H, W, C, K, _s())
        assert lg.ok()
        ref = torch.einsum("nhwc,kc->nkhw", a64, w64) + (b.double().view(1, K, 1, 1) if bias is not None else 0)
        terms = torch.einsum("nhwc,kc->nkhw", a64.abs(), w64.abs()) + (b.double().abs().view(1, K, 1, 1) if bias is not None else 0)
        log[f"logits bias={bias is not None}"] = _check(lg.t.cpu(), ref, _tol32(terms, steps), "logits")
    rows = _rows("ub2_outc_rows", N, H, W, C)
    res = {}
    for with_da in (True, False, True):
        da = Out((N, H, W), C, C + 16)
        dw, db = dw0.clone().cuda(), db0.clone().cuda()
        pg = Guarded((rows, K * C + K), F64)
        _call("ub2_outc_bwd", _p(dld), _p(ad), ld_a, _p(wd), _p(da.t) if with_da else _p(None), C + 16, _p(pg.t), rows,
              _p(dw), _p(db), N, H, W, C, K, _s())
        assert pg.ok() and da.ok()
        if with_da in res:
            assert torch.equal(res[with_da][3], pg.t) and torch.equal(_bits(res[with_da][0].t.cpu()), _bits(da.t.cpu()))
        res[with_da] = (da, dw.cpu(), db.cpu(), pg.t.clone())
    assert torch.equal(res[True][3], res[False][3]) and torch.equal(res[True][1], res[False][1])
    assert bool(torch.isnan(res[False][0].t.float()).all())            # da = NULL writes nothing
    da, dw, db, _ = res[True]
    rda = dl64 @ w64
    log["da"] = _check(da.t.cpu(), rda, _tol_bf(rda, _tol32(dl64.abs() @ w64.abs(), K)), "da")
    log["da not_rn_bf16"] = _not_rn(da.t.cpu(), rda)
    slots = KGATE // tpp
    k = _per_thread(px, rows * slots) + 5 + 1
    dwr = torch.einsum("nhwk,nhwc->kc", dl64, a64)
    dwt = torch.einsum("nhwk,nhwc->kc", dl64.abs(), a64.abs())
    log["dw"] = _check(dw, dw0.double() + dwr, _tol32(dw0.double().abs() + dwt * k, 1), "dw")
    log["db"] = _check(db, db0.double() + dl64.sum((0, 1, 2)), _tol32(db0.double().abs() + dl64.abs().sum((0, 1, 2)) * k, 1), "db")
    record(f"bf16 kernels outc K{K} C{C}", **log)


# =============================================================================================== ConvTranspose2d pieces
SHUF = [(2, 3, 5, 7, 11), (1, 4, 4, 8, 8), (3, 2, 1, 5, 2)]   # N, h, w, Ho, Wo (padding: F.pad's split)


@GPU
@pytest.mark.parametrize("C", [24, 40])
@pytest.mark.parametrize("N,h,w,Ho,Wo", SHUF)
def test_shuffle_and_convt_packs(C, N, h, w, Ho, Wo):
    """shuffle2x2_fwd / _bwd (copies: bit-exact, padded outputs zero) with the bias gradient (a reduction, into a
    non-zero dbias), pack_convt_weight (bf16 packs: bit-exact) and convt_wgrad_reduce (fixed-order fp32 sum)."""
    g = _gen(C * 100 + h * 10 + Ho)
    py, pxo = (Ho - 2 * h) // 2, (Wo - 2 * w) // 2
    ld_t, ld_out = 4 * C + 8, C + 8
    t = _rand_bf((N, h, w, ld_t), g)
    out = Out((N, Ho, Wo), C, ld_out)
    _call("ub2_shuffle2x2_fwd", _p(_slice(t, 4 * C)), ld_t, _p(out.t), ld_out, N, h, w, C, Ho, Wo, _s())
    assert out.ok()
    ref = torch.zeros((N, Ho, Wo, C), dtype=BF16)
    tv = t[..., :4 * C].reshape(N, h, w, 2, 2, C)
    core = tv.permute(0, 1, 3, 2, 4, 5).reshape(N, 2 * h, 2 * w, C)
    ref[:, py:py + 2 * h, pxo:pxo + 2 * w] = core
    assert torch.equal(_bits(out.t.cpu()), _bits(ref))
    # transpose + bias gradient
    ld_do, ld_dt = C + 16, 4 * C + 8
    dout = _rand_bf((N, Ho, Wo, ld_do), g)
    rows = _rows("ub2_shuffle2x2_rows", N, h, w, C, Ho, Wo)
    db0 = _randn((C,), g)
    dts, dbs, parts = [], [], []
    for _ in range(2):
        dt, pg = Out((N, h, w), 4 * C, ld_dt), Guarded((rows, C), F64)
        dbias = db0.clone().cuda()
        _call("ub2_shuffle2x2_bwd", _p(_slice(dout, C)), ld_do, _p(dt.t), ld_dt, _p(pg.t), rows, _p(dbias), N, h, w, C, Ho, Wo, _s())
        assert dt.ok() and pg.ok()
        dts.append(dt.t.cpu())
        dbs.append(dbias.cpu())
        parts.append(pg.t.clone())
    assert torch.equal(parts[0], parts[1]) and torch.equal(dbs[0], dbs[1]) and torch.equal(_bits(dts[0]), _bits(dts[1]))
    dcore = dout[:, py:py + 2 * h, pxo:pxo + 2 * w, :C]
    rdt = dcore.reshape(N, h, 2, w, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(N, h, w, 4 * C)
    assert torch.equal(_bits(dts[0]), _bits(rdt))
    d64 = dcore.double()
    lanes = 256 // (C // 8)
    k = _per_thread(N * h * w * 4, rows * lanes)
    log = {"partials": _check(_folded(parts[0]), d64.sum((0, 1, 2)), _tol32(d64.abs().sum((0, 1, 2)), k), "bias partials"),
           "dbias": _check(dbs[0], db0.double() + d64.sum((0, 1, 2)),
                           _tol32(db0.double().abs() + d64.abs().sum((0, 1, 2)) * (k + 1), 1), "dbias")}
    # weight packs: (Cin, Cout, 2, 2) -> fwd (4*Cout, Cin) row (i*2+j)*Cout + co, dg (Cin, 4*Cout), scale4, shift4
    Cin, Cout = C, C // 2 + 4
    wt, bias = _randn((Cin, Cout, 2, 2), g), _randn((Cout,), g)
    wb = wt.to(BF16)
    rf = wb.permute(2, 3, 1, 0).reshape(4 * Cout, Cin)
    rg = wb.permute(0, 2, 3, 1).reshape(Cin, 4 * Cout)
    for b in (bias, None):
        fwd, dg = Guarded((4 * Cout, Cin), BF16), Guarded((Cin, 4 * Cout), BF16)
        ss = Guarded((2, 4 * Cout))
        _call("ub2_pack_convt_weight", _p(wt.cuda()), _p(b.cuda() if b is not None else None), _p(fwd.t), _p(dg.t), _p(ss.t[0]),
              _p(ss.t[1]), Cin, Cout, _s())
        assert fwd.ok() and dg.ok() and ss.ok()
        assert torch.equal(_bits(fwd.t.cpu()), _bits(rf)) and torch.equal(_bits(dg.t.cpu()), _bits(rg))
        assert bool((ss.t[0] == 1).all())
        assert torch.equal(ss.t[1].cpu(), (b if b is not None else torch.zeros(Cout)).repeat(4))
    # split-K fold: grad[ci][co][i][j] (+)= sum_s partial[s][ci][(i*2+j)*Cout + co], in split order
    splits = 5
    part = _randn((splits, Cin, 4 * Cout), g)
    g0 = _randn((Cin, Cout, 2, 2), g)
    p64 = part.double().sum(0).view(Cin, 2, 2, Cout).permute(0, 3, 1, 2)
    pt = part.double().abs().sum(0).view(Cin, 2, 2, Cout).permute(0, 3, 1, 2)
    for acc in (0, 1):
        grad = Guarded((Cin, Cout, 2, 2), fill=g0.cuda())
        _call("ub2_convt_wgrad_reduce", _p(part.cuda()), splits, Cin, Cout, _p(grad.t), acc, _s())
        assert grad.ok()
        rref = p64 + (g0.double() if acc else 0)
        log[f"wgrad fold acc{acc}"] = _check(grad.t.cpu(), rref, _tol32(pt + (g0.double().abs() if acc else 0), splits + acc),
                                             "fold")
    record(f"bf16 kernels shuffle/convt C{C} {N}x{h}x{w} in {Ho}x{Wo}", **log)


# =============================================================================================== 64-bit offsets
@GPU
def test_bn_offsets_past_2_pow_31():
    """(33, 256, 256, 1024) bf16 = 2.2e9 elements: bn_act (relu, pool, a and pidx) and bn_bwd_apply (dA and the
    pooled gradient routed through pidx); the last rows of the last image and a seeded sample of pixels against
    float64 computed on the device for just those pixels."""
    N, H, W, C = 33, 256, 256, 1024
    assert N * H * W * C > 2 ** 31
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory, {free / 1e9:.1f} GB free")
    gen = torch.Generator(device="cuda").manual_seed(21)
    y = torch.empty((N, H, W, C), device="cuda", dtype=BF16)
    for i in range(0, N, 4):
        y[i:i + 4] = torch.randn((min(4, N - i), H, W, C), device="cuda", generator=gen).to(BF16)
    sc = torch.rand(C, device="cuda", generator=gen) + 0.5
    sh = torch.randn(C, device="cuda", generator=gen) * 0.3
    a = torch.empty_like(y)
    Hp, Wp = H // 2, W // 2
    p = torch.empty((N, Hp, Wp, C), device="cuda", dtype=BF16)
    idx = torch.empty((N, Hp, Wp, C), device="cuda", dtype=torch.uint8)
    _call("ub2_bn_act", _p(y), C, _p(sc), _p(sh), _p(a), C, _p(p), C, _p(idx), N, H, W, C, 1, _s())
    pixels = N * H * W
    gs = torch.Generator().manual_seed(22)
    flat = torch.cat([torch.arange(pixels - 2 * W, pixels), torch.randint(0, pixels, (512,), generator=gs)]).cuda()
    yf, af = y.view(pixels, C), a.view(pixels, C)
    z = yf[flat].double() * sc.double() + sh.double()
    ref = z.clamp_min(0)
    e_a = _check(af[flat], ref, _tol_bf(ref.cpu(), _tol32(z.abs().cpu(), 1)), "bn_act 64-bit")
    pp = torch.cat([torch.arange(N * Hp * Wp - Wp, N * Hp * Wp), torch.randint(0, N * Hp * Wp, (512,), generator=gs)]).cuda()
    n, hp, wp = pp // (Hp * Wp), (pp // Wp) % Hp, pp % Wp
    win = torch.stack([a[n, 2 * hp + r, 2 * wp + c] for r in (0, 1) for c in (0, 1)], 1).float()     # (P, 4, C)
    mx = win.max(1).values
    first = (win == mx.unsqueeze(1)).float().argmax(1)
    assert torch.equal(p.view(-1, C)[pp].float(), mx)
    assert torch.equal(idx.view(-1, C)[pp].long(), first)
    del win
    # backward apply: dA and dP routed, relu mask of y, coefficients A, B, C; dy written over a
    dA = torch.empty_like(y)
    for i in range(0, N, 4):
        dA[i:i + 4] = torch.randn((min(4, N - i), H, W, C), device="cuda", generator=gen).to(BF16)
    dP = torch.randn((N, Hp, Wp, C), device="cuda", generator=gen).to(BF16)
    coef = torch.stack([torch.rand(C, device="cuda", generator=gen) + 0.5, torch.randn(C, device="cuda", generator=gen) * 0.1,
                        torch.randn(C, device="cuda", generator=gen) * 0.1])
    _call("ub2_bn_bwd_apply", _p(dA), C, _p(dP), C, _p(idx), _p(y), C, _p(sc), _p(sh), _p(coef), _p(a), C, N, H, W, C, 1, _s())
    n, h, w_ = flat // (H * W), (flat // W) % H, flat % W
    inside = ((h // 2) < Hp) & ((w_ // 2) < Wp)
    ppi = (n * Hp + (h // 2).clamp_max(Hp - 1)) * Wp + (w_ // 2).clamp_max(Wp - 1)
    pos = ((h % 2) * 2 + (w_ % 2)).unsqueeze(1)
    routed = torch.where((idx.view(-1, C)[ppi].long() == pos) & inside.unsqueeze(1), dP.view(-1, C)[ppi].double(),
                         torch.zeros((), device="cuda", dtype=F64))
    gsum = (dA.view(-1, C)[flat].double() + routed) * (z > 0)
    A, B, Cc = coef.double()
    ref = A * gsum + B * yf[flat].double() + Cc
    terms = (A * gsum).abs() + (B * yf[flat].double()).abs() + Cc.abs()
    e_b = _check(af[flat], ref, _tol_bf(ref.cpu(), _tol32(terms.cpu(), 3)), "bn_bwd_apply 64-bit")
    record("bf16 kernels 64-bit offsets 33x256x256x1024", bn_act_worst_over_bound=e_a, bn_bwd_apply_worst_over_bound=e_b)
    del y, a, p, idx, dA, dP
    torch.cuda.empty_cache()
