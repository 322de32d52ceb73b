"""fp32 / TF32 mode with ``bilinear=False``: the ConvTranspose2d(C, C/2, 2, stride 2) + F.pad up-sampling of
Up / AttentionUp (layers.py:81, :98-102, :217-221), from the kernels of csrc/shuffle.cu to whole networks.

* the host-side argument checks of the four fp32 entry points (no ``gpu`` mark, child process without a device);
* the kernels one at a time against exact references: the pixel shuffle and its transpose are copies (bit-exact),
  the weight pack is a copy (bit-exact), the bias gradient is a reduction gated at ``2u * steps * sum|terms|`` with
  ``steps`` read off the launch geometry, as in test_fp32_kernels_gpu.py; every launch writes inside NaN guard
  bands and every reduction repeats bit for bit;
* the layer alone against float64 ``conv_transpose2d`` + ``F.pad`` on the same TF32-representable operands: eval
  (one TF32 pass, output rounded to TF32) rel-L2 <= 1e-3, training output and dx (3xTF32) <= 1e-5, dW (bf16
  hi/lo) <= 1e-4, db within the reduction bound;
* Up / AttentionUp modules through ``check_module_f32`` and whole networks against the fp32 oracle, including
  deep supervision, the input gradient, frozen up-sampling parameters and the batch-sharded trainer.

Every measured number goes to the parity log."""
import copy
import os
import subprocess
import sys

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import unet_oracle as O
from parity_log import record
from test_fp32_kernels_gpu import Guarded, _bits, _call, _gen, _p, _randn, _rel_l2, _rows, _s, _within
from test_fp32_train_gpu import ACTIVE, _tf32, check_module_f32
from test_input_grad_gpu import _all_active, _gouts, _net_id
from test_modules_gpu import _build, _x, cosine, rel_l2

GPU = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64 = torch.float32, torch.float64
TOL = 1e-3


@pytest.fixture
def tf32_mode():
    import unet
    unet.set_precision("tf32")
    yield
    unet.set_precision("bf16")


# =============================================================================================== host checks
CHILD = r'''
import ctypes, sys
sys.path.insert(0, sys.argv[1] + "/unet-segment-pytorch_b200")
from unet import _C
lib = _C.lib()
P = 1 << 20                      # a 16-byte-aligned fake device address: the calls below must never use it
Q = P + 4                        # 4-byte aligned only
# the entry points under test, with their parameters as include/unetb200.h declares them
SIG = {name: _C.SIGNATURES[name] for name in ("ub2_f32_shuffle2x2_fwd", "ub2_f32_shuffle2x2_bwd", "ub2_f32_pack_convt_weight")}
rows = lambda N=2, h=4, w=4, C=16, Ho=8, Wo=8: lib.ub2_f32_shuffle2x2_rows(N, h, w, C, Ho, Wo)
R = rows()
assert R > 0 and rows(C=1024) > 0 and rows(N=1, h=1, w=1, C=4, Ho=2, Wo=2) > 0
GEOM = dict(N=2, h=4, w=4, C=16, Ho=8, Wo=8)
BASE = {
 "ub2_f32_shuffle2x2_fwd": dict(GEOM, ld_t=64, ld_out=16),
 "ub2_f32_shuffle2x2_bwd": dict(GEOM, ld_dout=16, ld_dt=64, rows=R),
 "ub2_f32_pack_convt_weight": dict(Cin=32, Cout=16),
}
def call(name, **kw):
    vals = []
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
FWD, BWD, PACK = "ub2_f32_shuffle2x2_fwd", "ub2_f32_shuffle2x2_bwd", "ub2_f32_pack_convt_weight"
BAD = []
for name in (FWD, BWD):
    BAD += [(name, dict(N=0), S), (name, dict(N=-3), S), (name, dict(h=0), S), (name, dict(w=-1), S), (name, dict(C=0), S),
            (name, dict(C=-4), S), (name, dict(C=6), S), (name, dict(C=1028, ld_t=4112, ld_out=1028, ld_dout=1028, ld_dt=4112), S),
            (name, dict(Ho=7), S), (name, dict(Wo=7), S), (name, dict(Ho=0), S)]
BAD += [
 # channel strides below the row, NULL required pointers
 (FWD, dict(ld_t=60), S), (FWD, dict(ld_out=12), S), (FWD, dict(t=None), S), (FWD, dict(out=None), S),
 (BWD, dict(ld_dout=12), S), (BWD, dict(ld_dt=60), S), (BWD, dict(dout=None), S), (BWD, dict(dt=None), S),
 (BWD, dict(dbias=None), S),                                   # a bias gradient without its output
 (PACK, dict(Cin=0), S), (PACK, dict(Cout=0), S), (PACK, dict(Cout=-1), S),
 (PACK, dict(w=None), S), (PACK, dict(fwd=None), S), (PACK, dict(scale4=None), S), (PACK, dict(shift4=None), S),
 # strides and alignment
 (FWD, dict(ld_t=66), A), (FWD, dict(ld_out=18), A), (FWD, dict(t=Q), A), (FWD, dict(out=Q), A),
 (BWD, dict(ld_dout=18), A), (BWD, dict(ld_dt=66), A), (BWD, dict(dout=Q), A), (BWD, dict(dt=Q), A),
 (BWD, dict(partials=Q), A), (BWD, dict(dbias=P + 2), A),
 (PACK, dict(w=P + 2), A), (PACK, dict(bias=P + 2), A), (PACK, dict(fwd=P + 2), A), (PACK, dict(scale4=P + 2), A),
 (PACK, dict(shift4=P + 2), A),
 # workspace rows
 (BWD, dict(rows=R + 1), WS), (BWD, dict(rows=R - 1), WS), (BWD, dict(rows=0), WS),
]
ROWS_BAD = [dict(N=0), dict(h=0), dict(w=-1), dict(C=0), dict(C=6), dict(C=1028), dict(Ho=7), dict(Wo=7)]
GOOD = [(name, {}) for name in SIG] + [
 # the NULLs the modules pass: no bias gradient (dbias and rows are then ignored), no bias
 (BWD, dict(partials=None, dbias=None, rows=0)), (BWD, dict(partials=None, rows=12345)), (PACK, dict(bias=None)),
 # edges that are valid
 (FWD, dict(ld_t=68, ld_out=20)), (FWD, dict(C=4, ld_t=16, ld_out=4)), (FWD, dict(C=1024, ld_t=4096, ld_out=1024)),
 (FWD, dict(Ho=11, Wo=9)), (FWD, dict(N=1, h=1, w=1, Ho=2, Wo=2)),
 (BWD, dict(ld_dout=48, ld_dt=68)), (BWD, dict(C=4, ld_dout=4, ld_dt=16, rows=rows(C=4))),
 (BWD, dict(C=1024, ld_dout=1024, ld_dt=4096, rows=rows(C=1024))), (BWD, dict(Ho=11, Wo=9, rows=rows(Ho=11, Wo=9))),
 (BWD, dict(N=1, h=1, w=1, C=4, Ho=2, Wo=2, ld_dout=4, ld_dt=16, rows=rows(N=1, h=1, w=1, C=4, Ho=2, Wo=2))),
 (PACK, dict(Cin=1, Cout=1)), (PACK, dict(Cin=1024, Cout=512)),
]
for name, kw, want in BAD:
    rc = call(name, **kw)
    print(name, sorted(kw.items()), rc, want, "OK" if rc == want else "WRONG", flush=True)
for kw in ROWS_BAD:
    rc = rows(**kw)
    print("ub2_f32_shuffle2x2_rows", sorted(kw.items()), rc, S, "OK" if rc == S else "WRONG", flush=True)
for name, kw in GOOD:
    rc = call(name, **kw)
    print(name, "valid", sorted(kw.items()), rc, "positive", "OK" if rc > 0 else "WRONG", flush=True)
print("DONE", len(BAD) + len(ROWS_BAD), len(GOOD), flush=True)
'''


def test_convt_entry_points_check_arguments_on_the_host():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")      # argument checks only, also on a GPU box
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, env=env)
    lines = r.stdout.strip().splitlines()
    assert r.returncode == 0 and lines and lines[-1].startswith("DONE"), (r.returncode, lines[-3:], r.stderr[-2000:])
    wrong = [l for l in lines if l.endswith("WRONG")]
    assert not wrong, wrong
    _, nbad, ngood = lines[-1].split()
    assert sum(l.endswith("OK") for l in lines) == int(nbad) + int(ngood) >= 80


# =============================================================================================== kernels
def _pads(h, w, Ho, Wo):
    return (Ho - 2 * h) // 2, (Wo - 2 * w) // 2       # F.pad's [d // 2, d - d // 2]


def _shuffle_ref(t, C, Ho, Wo):
    """t (N,h,w,>=4C) -> (N,Ho,Wo,C): out[n, 2y+i+py, 2x+j+px, co] = t[n, y, x, (i*2+j)*C + co], zeros elsewhere."""
    N, h, w = t.shape[:3]
    py, px = _pads(h, w, Ho, Wo)
    out = torch.zeros((N, Ho, Wo, C), dtype=t.dtype, device=t.device)
    out[:, py:py + 2 * h, px:px + 2 * w] = (t[..., :4 * C].reshape(N, h, w, 2, 2, C).permute(0, 1, 3, 2, 4, 5)
                                           .reshape(N, 2 * h, 2 * w, C))
    return out


def _unshuffle_ref(dout, h, w, C):
    """dout (N,Ho,Wo,>=C) -> dt (N,h,w,4C): the transpose of _shuffle_ref (the padding is dropped)."""
    N, Ho, Wo = dout.shape[:3]
    py, px = _pads(h, w, Ho, Wo)
    core = dout[:, py:py + 2 * h, px:px + 2 * w, :C]
    return core.reshape(N, h, 2, w, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(N, h, w, 4 * C)


SHUFFLE_FWD = [  # N, h, w, C, Ho - 2h, Wo - 2w, ld_t - 4C, ld_out - C
    (2, 3, 5, 4, 0, 0, 0, 0), (1, 4, 3, 12, 1, 3, 8, 4), (2, 5, 7, 64, 3, 1, 16, 12), (1, 2, 3, 1024, 1, 0, 4, 4),
    (3, 1, 1, 12, 3, 3, 0, 8), (2, 16, 16, 64, 1, 1, 0, 0)]


@GPU
@pytest.mark.parametrize("N,h,w,C,dh,dw,et,eo", SHUFFLE_FWD)
def test_shuffle_forward_is_a_copy(N, h, w, C, dh, dw, et, eo):
    """ub2_f32_shuffle2x2_fwd bit for bit: even and odd padding, channel strides above 4C (t) and C (out); the
    columns of out beyond C stay untouched."""
    Ho, Wo, ld_t, ld_out = 2 * h + dh, 2 * w + dw, 4 * C + et, C + eo
    g = _gen(N * h * w + C + dh + dw)
    tf = _randn((N, h, w, ld_t), g)
    t = Guarded((N, h, w, ld_t), fill=tf.cuda())
    out = Guarded((N, Ho, Wo, ld_out))
    _call("ub2_f32_shuffle2x2_fwd", _p(t.t), ld_t, _p(out.t), ld_out, N, h, w, C, Ho, Wo, _s())
    assert out.ok() and t.ok(), "guard bands"
    got = out.t.cpu()
    assert torch.equal(_bits(got[..., :C]), _bits(_shuffle_ref(tf, C, Ho, Wo)))
    assert torch.isnan(got[..., C:]).all()
    assert torch.equal(_bits(t.t.cpu()), _bits(tf))


SHUFFLE_BWD = [  # N, h, w, C, Ho - 2h, Wo - 2w, ld_dout (dout is a channel slice), ld_dt - 4C, bias gradient
    (2, 3, 5, 4, 0, 0, 12, 0, True), (1, 4, 3, 12, 1, 3, 28, 4, True), (2, 5, 7, 64, 3, 1, 192, 0, True),
    (1, 2, 3, 1024, 1, 0, 1088, 4, True), (2, 32, 32, 256, 1, 1, 512, 0, True), (8, 64, 64, 64, 0, 0, 128, 0, True),
    (2, 5, 7, 64, 3, 1, 128, 8, False)]


@GPU
@pytest.mark.parametrize("N,h,w,C,dh,dw,ld_do,et,bias", SHUFFLE_BWD)
def test_shuffle_backward_and_bias_gradient(N, h, w, C, dh, dw, ld_do, et, bias):
    """ub2_f32_shuffle2x2_bwd: dt bit for bit from a dout that is a channel slice of a wider tensor (the concat's
    data gradient), and the bias gradient accumulated (+=) into a non-zero dbias, within 2u * steps * sum|terms|
    with steps = the sequential fp32 additions of one thread plus the two final roundings; run twice, it repeats
    bit for bit.  Without partials, dbias is not touched."""
    Ho, Wo, ld_dt = 2 * h + dh, 2 * w + dw, 4 * C + et
    g = _gen(N * h * w + C + ld_do)
    df = _randn((N, Ho, Wo, ld_do), g)
    db0 = _randn((C,), g)
    dout = Guarded((N, Ho, Wo, ld_do), fill=df.cuda())
    rows = _rows("ub2_f32_shuffle2x2_rows", N, h, w, C, Ho, Wo) if bias else 0
    results = []
    for _ in range(2):
        dt = Guarded((N, h, w, ld_dt))
        part = Guarded((max(rows, 1), C), F64)
        db = Guarded((C,), fill=db0.cuda())
        _call("ub2_f32_shuffle2x2_bwd", _p(dout.t), ld_do, _p(dt.t), ld_dt, _p(part.t if bias else None), rows, _p(db.t),
              N, h, w, C, Ho, Wo, _s())
        assert dt.ok() and part.ok() and db.ok() and dout.ok(), "guard bands"
        results.append((dt.t.cpu(), db.t.cpu()))
    (dt0, dbg), (dt1, dbg1) = results
    assert torch.equal(_bits(dt0[..., :4 * C]), _bits(_unshuffle_ref(df, h, w, C)))
    assert torch.isnan(dt0[..., 4 * C:]).all()
    assert torch.equal(_bits(dbg), _bits(dbg1)), "bias gradient not repeatable"
    if not bias:
        assert torch.equal(_bits(dbg), _bits(db0))
        return
    core = _unshuffle_ref(df, h, w, C).double().reshape(-1, 4, C)
    ref = db0.double() + core.sum((0, 1))
    terms = db0.double().abs() + core.abs().sum((0, 1))
    lanes = max(256 // (C // 4), 1)
    k = -(-(N * h * w * 4) // (rows * lanes))                # sequential fp32 adds per thread
    e = _within(dbg, ref, terms, k + 2, ("dbias", N, h, w, C))
    record(f"fp32 convt shuffle bwd {N}x{h}x{w} C{C} pad {dh}/{dw} ld {ld_do}", dbias_worst_over_2u=e, steps=k + 2)


@GPU
@pytest.mark.parametrize("Cin,Cout", [(128, 64), (12, 4), (1024, 512), (36, 20)])
@pytest.mark.parametrize("with_bias", [True, False])
def test_pack_convt_weight_is_exact(Cin, Cout, with_bias):
    """ub2_f32_pack_convt_weight: the unrounded (4*Cout, Cin) 1x1 weight with row (i*2+j)*Cout + co, scale4 = 1 and
    shift4 = the bias tiled four times (zeros without a bias), bit for bit."""
    g = _gen(Cin * Cout + with_bias)
    w = _randn((Cin, Cout, 2, 2), g)
    b = _randn((Cout,), g)
    fwd = Guarded((4 * Cout, Cin))
    sc, sh = Guarded((4 * Cout,)), Guarded((4 * Cout,))
    _call("ub2_f32_pack_convt_weight", _p(w.cuda()), _p(b.cuda() if with_bias else None), _p(fwd.t), _p(sc.t), _p(sh.t),
          Cin, Cout, _s())
    assert fwd.ok() and sc.ok() and sh.ok(), "guard bands"
    assert torch.equal(_bits(fwd.t.cpu()), _bits(w.permute(2, 3, 1, 0).reshape(4 * Cout, Cin)))
    assert torch.equal(sc.t.cpu(), torch.ones(4 * Cout))
    assert torch.equal(_bits(sh.t.cpu()), _bits(b.repeat(4) if with_bias else torch.zeros(4 * Cout)))


@GPU
def test_shuffle_offsets_past_2_pow_31():
    """(33, 128, 128, 4*1024) -> (33, 257, 257, 1024) fp32: the output is 2.2e9 elements.  The forward is checked
    image by image against the exact shuffle, the backward of its output (no bias gradient) must give t back."""
    N, h, w, C = 33, 128, 128, 1024
    Ho, Wo = 2 * h + 1, 2 * w + 1
    assert N * Ho * Wo * C > 2 ** 31
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory, {free / 1e9:.1f} GB free")
    gen = torch.Generator(device="cuda").manual_seed(13)
    t = torch.empty((N, h, w, 4 * C), device="cuda")
    for i in range(0, N, 4):
        t[i:i + 4].normal_(generator=gen)
    out = torch.empty((N, Ho, Wo, C), device="cuda")
    _call("ub2_f32_shuffle2x2_fwd", _p(t), 4 * C, _p(out), C, N, h, w, C, Ho, Wo, _s())
    for i in range(N):
        assert torch.equal(_bits(out[i:i + 1]), _bits(_shuffle_ref(t[i:i + 1], C, Ho, Wo))), i
    dt = torch.empty_like(t)
    _call("ub2_f32_shuffle2x2_bwd", _p(out), C, _p(dt), 4 * C, _p(None), 0, _p(None), N, h, w, C, Ho, Wo, _s())
    assert torch.equal(_bits(dt), _bits(t))
    record("fp32 convt shuffle 64-bit offsets 33x128x128 C1024 -> 257x257", out_elements=N * Ho * Wo * C)
    del t, out, dt
    torch.cuda.empty_cache()


# =============================================================================================== the layer alone
LAYER = [(2, 128, 8, 8, 16, 16), (1, 128, 6, 9, 13, 19), (2, 64, 5, 7, 11, 14), (1, 256, 4, 4, 8, 8)]


def _layer_ref(x, w, b, Ho, Wo):
    y = F.conv_transpose2d(x, w, b, stride=2)
    dy, dx = Ho - y.shape[2], Wo - y.shape[3]
    return F.pad(y, [dx // 2, dx - dx // 2, dy // 2, dy - dy // 2])


def _layer_operands(N, Cin, h, w, seed):
    g = _gen(seed)
    mod = nn.ConvTranspose2d(Cin, Cin // 2, kernel_size=2, stride=2)
    with torch.no_grad():
        mod.weight.copy_(_tf32(_randn(mod.weight.shape, g, (Cin * 4) ** -0.5)))
        mod.bias.copy_(_tf32(_randn(mod.bias.shape, g, 0.1)))
    return mod, _tf32(_randn((N, Cin, h, w), g))


@GPU
@pytest.mark.parametrize("N,Cin,h,w,Ho,Wo", LAYER)
def test_layer_eval(N, Cin, h, w, Ho, Wo):
    """fp32.conv_transpose2x2 under no_grad: one TF32 pass with the output rounded to TF32, against float64 on the
    same TF32-representable operands: rel-L2 <= 1e-3."""
    from unet import fp32
    mod, x = _layer_operands(N, Cin, h, w, N * Cin + h * w + Ho)
    with torch.no_grad():
        ref = _layer_ref(x.double(), mod.weight.double(), mod.bias.double(), Ho, Wo)
    m = copy.deepcopy(mod).cuda().eval()
    with torch.no_grad():
        got = fp32.conv_transpose2x2(m, x.cuda(), Ho, Wo)
    assert got.shape == ref.shape and got.dtype == F32
    e = _rel_l2(got.cpu(), ref)
    record(f"fp32 convt layer eval {N}x{Cin}x{h}x{w} -> {Ho}x{Wo}", out_rel_l2=e)
    assert e <= TOL, e


@GPU
@pytest.mark.parametrize("N,Cin,h,w,Ho,Wo", LAYER)
def test_layer_training(N, Cin, h, w, Ho, Wo):
    """The training path (ConvTranspose2x2F32) against float64 autograd: output and dx (3xTF32) rel-L2 <= 1e-5, dW
    (bf16 hi/lo) <= 1e-4, db within 2u * steps * sum|terms| of the float64 sum."""
    from unet import fp32
    mod, x = _layer_operands(N, Cin, h, w, N * Cin + h * w + Wo)
    g = _gen(Ho * Wo + Cin)
    gout = _randn((N, Cin // 2, Ho, Wo), g)
    xr = x.double().requires_grad_(True)
    wr, br = mod.weight.detach().double().requires_grad_(True), mod.bias.detach().double().requires_grad_(True)
    ref = _layer_ref(xr, wr, br, Ho, Wo)
    ref.backward(gout.double())
    m = copy.deepcopy(mod).cuda().train()
    xc = x.cuda().requires_grad_(True)
    out = fp32.conv_transpose2x2(m, xc, Ho, Wo)
    out.backward(gout.cuda())
    e_o, e_x, e_w = _rel_l2(out.detach().cpu(), ref.detach()), _rel_l2(xc.grad.cpu(), xr.grad), _rel_l2(m.weight.grad.cpu(), wr.grad)
    cout = Cin // 2
    rows = _rows("ub2_f32_shuffle2x2_rows", N, h, w, cout, Ho, Wo)
    k = -(-(N * h * w * 4) // (rows * max(256 // (cout // 4), 1)))
    py, px = _pads(h, w, Ho, Wo)
    terms = gout[:, :, py:py + 2 * h, px:px + 2 * w].double().abs().sum((0, 2, 3))
    e_b = _within(m.bias.grad, br.grad, terms, k + 1, "db")
    record(f"fp32 convt layer train {N}x{Cin}x{h}x{w} -> {Ho}x{Wo}", out_rel_l2=e_o, dx_rel_l2=e_x, dw_rel_l2=e_w,
           db_worst_over_2u=e_b)
    assert e_o <= 1e-5 and e_x <= 1e-5, (e_o, e_x)
    assert e_w <= 1e-4, e_w


# =============================================================================================== modules
@GPU
@ACTIVE
@pytest.mark.parametrize("training", [True, False])
def test_up_transposed(training, all_active, tf32_mode):
    from unet.models.layers import Up
    check_module_f32(Up(128, 64, False), lambda x1, x2, sd, tr: O.up_block(x1, x2, sd, "m", False, False, tr),
                     [_x((2, 128, 8, 8), 51), _x((2, 64, 16, 16), 52)], training, all_active=all_active)


@GPU
@ACTIVE
@pytest.mark.parametrize("training", [True, False])
def test_up_transposed_padded(training, all_active, tf32_mode):
    from unet.models.layers import Up
    check_module_f32(Up(128, 64, False), lambda x1, x2, sd, tr: O.up_block(x1, x2, sd, "m", False, False, tr),
                     [_x((1, 128, 6, 9), 53), _x((1, 64, 13, 19), 54)], training, all_active=all_active)


@GPU
@ACTIVE
@pytest.mark.parametrize("training", [True, False])
def test_attention_up_transposed(training, all_active, tf32_mode):
    """x1 feeds both the gate (as g, gate_channels = in_channels) and the transposed convolution: its gradient is
    the sum of the two."""
    from unet.models.layers import AttentionUp
    check_module_f32(AttentionUp(128, 64, False), lambda x1, x2, sd, tr: O.up_block(x1, x2, sd, "m", True, False, tr),
                     [_x((2, 128, 8, 8), 55), _x((2, 64, 16, 16), 56)], training, all_active=all_active)


# =============================================================================================== networks
@GPU
@pytest.mark.parametrize("attention,base,n,hw", [(True, 32, 2, 64), (False, 32, 2, 64), (True, 64, 1, 512)])
def test_network_eval_within_1e3(attention, base, n, hw, tf32_mode):
    model, sd, _ = _build(attention, base, 42, bilinear=False)
    model = model.cuda().eval()
    x, _ = O.synthetic_batch(n, hw, hw, seed=1234)
    with torch.no_grad():
        logits = model(x.cuda()).cpu()
    ref = O.unet_forward(x, sd, attention=attention, bilinear=False, training=False)
    e = rel_l2(logits, ref)
    record(f"tf32 eval bilinear=False attention={attention} base {base} {n}x1x{hw}x{hw}", logits_rel_l2=e)
    assert logits.dtype == torch.float32 and logits.shape == ref.shape
    assert e <= TOL, e


@GPU
@pytest.mark.parametrize("attention", [True, False])
def test_train_step_end_to_end(attention, tf32_mode):
    """One fp32-mode training step with bilinear=False against the fp32 oracle's: loss within 1e-5 relative,
    logits within 1e-3, every parameter gradient's cosine >= 0.995 (see test_fp32_train_gpu)."""
    from unet.utils.loss import DiceBCELoss
    model, sd, _ = _build(attention, 32, 22, bilinear=False)
    x, t = O.synthetic_batch(2, 64, 64, seed=6, fg_fraction=0.05)
    model = model.cuda().train()
    logits = model(x.cuda())
    loss = DiceBCELoss()(logits, t.cuda())
    loss.backward()
    ref_loss, ref_logits, ref_grads = O.train_grads(x, t, O.clone_state(sd), attention=attention, bilinear=False)
    e = rel_l2(logits, ref_logits)
    errs = {k: rel_l2(p.grad, ref_grads[k]) for k, p in model.named_parameters() if p.numel() > 1}
    cos = sorted(cosine(p.grad, ref_grads[k]) for k, p in model.named_parameters() if p.numel() > 1)
    up = sorted(v for k, v in errs.items() if ".up." in k)
    srt = sorted(errs.values())
    record(f"tf32-train e2e step bilinear=False attention={attention} base 32 2x64x64", logits_rel_l2=e, loss=loss.item(),
           loss_oracle=ref_loss.item(), grad_rel_l2_median=srt[len(srt) // 2], grad_rel_l2_max=srt[-1],
           up_grad_rel_l2_max=up[-1], grad_cos_min=cos[0])
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert e <= TOL and cos[0] >= 0.995, (e, cos[0])


@GPU
@pytest.mark.parametrize("bilinear", [True, False])
def test_deep_supervision_outputs_and_loss(bilinear, tf32_mode):
    """deep_supervision=True in TF32 training mode: the four outputs within 1e-3 of the oracle's and
    DeepSupervisionLoss within 1e-5 relative of the oracle's loss on the oracle's outputs; every head gets a
    finite, non-zero gradient."""
    from unet.utils.loss import DeepSupervisionLoss, DiceBCELoss
    model, sd, _ = _build(True, 32, 31, deep_supervision=True, bilinear=bilinear)
    x, t = O.synthetic_batch(2, 64, 64, seed=7, fg_fraction=0.05)
    model = model.cuda().train()
    outs = model(x.cuda())
    assert isinstance(outs, list) and len(outs) == 4 and all(o.shape == (2, 2, 64, 64) for o in outs)
    loss = DeepSupervisionLoss(DiceBCELoss())(outs, t.cuda())
    ref_outs = O.unet_forward(x, O.clone_state(sd), attention=True, bilinear=bilinear, deep_supervision=True, training=True)
    ref_loss = O.deep_supervision_loss(ref_outs, t)
    errs = [rel_l2(o, r) for o, r in zip(outs, ref_outs)]
    record(f"tf32 deep supervision bilinear={bilinear} base 32 2x64x64", outputs_rel_l2=errs, loss=loss.item(),
           loss_oracle=ref_loss.item())
    assert max(errs) <= TOL, errs
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    loss.backward()
    heads = [p for n, p in model.named_parameters() if n.startswith("ds_out")]
    assert len(heads) == 6 and all(p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0
                                   for p in heads)


NETS = [(True, 32, {"bilinear": False}), (False, 32, {"bilinear": False}), (True, 32, {"deep_supervision": True}),
        (True, 32, {"deep_supervision": True, "bilinear": False})]


@GPU
@pytest.mark.parametrize("net", NETS, ids=[_net_id(p) for p in NETS])
def test_network_input_grad_fp32_all_active(net):
    """dL/dx in TF32 mode, eval, every ReLU active, for the bilinear=False and deep-supervision networks: within
    1e-3 of the fp32 oracle, or 1.5 times the stem weight gradient's error where the upstream gradient already
    carries more (the gate of test_input_grad_gpu.test_network_input_grad_fp32_all_active)."""
    import unet
    attention, bf, kw = net
    model, sd, cfg = _build(attention, bf, 31, **kw)
    sd = _all_active(sd)
    model.load_state_dict(sd)
    x, _ = O.synthetic_batch(2, 64, 64, seed=8)
    stem = "inc.double_conv.0.weight"
    unet.set_precision("tf32")
    try:
        model = model.cuda().eval()
        gouts = _gouts(model, x, 5)
        xc = x.cuda().requires_grad_(True)
        (model(xc) * gouts[0].cuda()).sum().backward()
        got, got_w = xc.grad.cpu(), dict(model.named_parameters())[stem].grad.cpu()
    finally:
        unet.set_precision("bf16")
    xo = x.clone().requires_grad_(True)
    w = dict(sd)
    w[stem] = sd[stem].clone().requires_grad_(True)
    (O.unet_forward(xo, w, attention=attention, bilinear=cfg["bilinear"], training=False) * gouts[0]).sum().backward()
    e, e_w = rel_l2(got, xo.grad), rel_l2(got_w, w[stem].grad)
    gate = max(TOL, 1.5 * e_w)
    record(f"input-grad network fp32 all-active [{_net_id(net)}-eval] 2x1x64x64", rel_l2_vs_fp32=e,
           stem_weight_grad_rel_l2_vs_fp32=e_w, gate=gate)
    assert e <= gate, (e, e_w)


@GPU
def test_frozen_upsampling_parameters(tf32_mode):
    """Training step with every ConvTranspose2d parameter (up*.up.*) frozen: the input gradient and every other
    parameter's gradient are bit-identical to the step with them trainable, and the frozen ones get no .grad."""
    model, _, _ = _build(True, 32, 33, bilinear=False)
    x, _ = O.synthetic_batch(2, 64, 64, seed=9)
    model = model.cuda().train()
    grads = []
    for freeze in (False, True):
        m = copy.deepcopy(model)
        for n, p in m.named_parameters():
            p.requires_grad_(not (freeze and ".up." in n))
        xc = x.cuda().requires_grad_(True)
        m(xc).sum().backward()
        grads.append((xc.grad, {n: p.grad for n, p in m.named_parameters()}))
    (gx, free), (gx_f, frozen) = grads
    up = [n for n in frozen if ".up." in n]
    assert len(up) == 8 and all(frozen[n] is None for n in up)
    assert all(free[n] is not None for n in up)
    assert torch.equal(gx, gx_f) and gx.abs().sum() > 0
    for n, gr in frozen.items():
        if n not in up:
            assert gr is not None and torch.equal(gr, free[n]), n


@GPU
def test_trainer_runs_in_tf32_mode(tf32_mode):
    """BatchShardedTrainer (gradient buckets, FusedAdamW) on AttentionUNet(bilinear=False) in TF32 mode: two steps,
    finite losses, and every ConvTranspose2d parameter moved."""
    from unet.models import AttentionUNet
    from unet.optim import FusedAdamW
    from unet.parallel import BatchShardedTrainer
    from unet.utils.loss import DiceBCELoss
    torch.manual_seed(3)
    model = AttentionUNet(1, 2, False, 32).cuda()
    tr = BatchShardedTrainer(model, DiceBCELoss(), FusedAdamW(model.parameters(), lr=1e-3), grad_clip=1.0)
    x, t = O.synthetic_batch(2, 64, 64, seed=9, fg_fraction=0.05)
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    losses = [tr.step(x.cuda(), t.cuda()).item() for _ in range(2)]
    assert all(torch.isfinite(torch.tensor(l)) for l in losses)
    up = [n for n in before if ".up." in n]
    assert len(up) == 8
    moved = {n: not torch.equal(before[n], p) for n, p in model.named_parameters() if n in up}
    record("tf32 trainer AttentionUNet(1, 2, False, 32) 2x64x64", losses=losses)
    assert all(moved.values()), moved
