"""Gradients with respect to the network input: the stem convolution's data gradient (ub2_conv_in_dgrad /
ub2_f32_conv_in_dgrad) and everything built on it.

* host: every bad argument is refused before the device is touched (no ``gpu`` mark);
* kernels: both entry points against float64 ``torch.nn.grad.conv2d_input`` on the same operands over a shape
  grid that reaches both variants (Cin = 1 with W % 4 == 0 and aligned pointers: the register-window kernel;
  everything else: the general one), channel slices of dy, a dx pointer off 16-byte alignment; bit-identical
  repeats; canary bands around dx; a dy of more than 2^31 elements;
* modules and whole networks: ``x.requires_grad_()`` through DoubleConv, UNet and AttentionUNet in both
  precisions, train and eval, against the oracle's autograd; frozen parameters (saliency maps); a two-stage
  cascade whose first stage trains through the second; CUDA-graph capture of forward + backward to the input.
Every measured number goes to the parity log."""
import copy
import os
import subprocess
import sys

import pytest
import torch

from oracle import unet_oracle as O
from parity_log import record
from test_modules_gpu import _build, _x, check_module, cosine, rel_l2

GPU = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HW_GRID = [(1, 1), (3, 5), (17, 33), (64, 64), (32, 36)]


# --------------------------------------------------------------------------- host-side argument checks
CHILD = r'''
import ctypes, sys
sys.path.insert(0, sys.argv[1] + "/unet-segment-pytorch_b200")
from unet import _C
lib = _C.lib()
P = 1 << 20                      # a 16-byte-aligned fake device address: the calls below must never use it
for name in ("ub2_conv_in_dgrad", "ub2_f32_conv_in_dgrad"):
    getattr(lib, name).restype = ctypes.c_int
    getattr(lib, name).argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_void_p]
def call(name, dy=P, ld=64, w=P, dx=P, N=2, Cin=1, H=8, W=8, Cout=64):
    return getattr(lib, name)(dy, ld, w, dx, N, Cin, H, W, Cout, None)
bad = {
    "N=0": (dict(N=0), -1), "N<0": (dict(N=-3), -1), "H=0": (dict(H=0), -1), "W=0": (dict(W=0), -1),
    "H<0": (dict(H=-1), -1), "W<0": (dict(W=-8), -1), "Cout=0": (dict(Cout=0, ld=8), -1),
    "Cout<0": (dict(Cout=-8), -1), "Cin=0": (dict(Cin=0), -1), "Cin<0": (dict(Cin=-1), -1),
    "ld<Cout": (dict(ld=32), -1), "dy NULL": (dict(dy=None), -1), "w NULL": (dict(w=None), -1),
    "dx NULL": (dict(dx=None), -1), "dx misaligned": (dict(dx=P + 2), -2), "w misaligned": (dict(w=P + 2), -2),
}
bf16 = dict(bad, **{"Cin>4": (dict(Cin=5), -1), "Cout%8": (dict(Cout=12, ld=16), -1), "ld%8": (dict(ld=68), -2),
                    "Cout/8>256": (dict(Cout=2056, ld=2056), -1), "dy odd": (dict(dy=P + 1), -2),
                    "N*H*W*Cin>=2e9": (dict(N=8000, H=512, W=512), -1),
                    "smem>48KB": (dict(Cin=4, Cout=512, ld=512), -1)})
f32 = dict(bad, **{"Cout%4": (dict(Cout=6, ld=8), -1), "ld%4": (dict(ld=66), -2), "dy misaligned": (dict(dy=P + 2), -2),
                   "smem>48KB": (dict(Cin=15, Cout=128, ld=128), -1)})
for name, cases in (("ub2_conv_in_dgrad", bf16), ("ub2_f32_conv_in_dgrad", f32)):
    for what, (kw, want) in cases.items():
        rc = call(name, **kw)
        print(name, what, rc, want, "OK" if rc == want else "WRONG", flush=True)
    # valid arguments pass the checks and only then fail for want of a device (a CUDA error code, > 0)
    for kw in (dict(), dict(Cin=3, W=9), dict(Cin=4, Cout=16, ld=16) if name == "ub2_conv_in_dgrad" else dict(Cin=7, Cout=20, ld=20)):
        rc = call(name, **kw)
        print(name, "valid", kw, rc, "positive", "OK" if rc > 0 else "WRONG", flush=True)
print("DONE", flush=True)
'''


def test_entry_points_refuse_bad_arguments_on_the_host():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")      # argument checks only, also on a GPU box
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, env=env)
    lines = r.stdout.strip().splitlines()
    assert r.returncode == 0 and lines and lines[-1] == "DONE", (r.returncode, lines[-3:], r.stderr[-2000:])
    wrong = [l for l in lines if l.endswith("WRONG")]
    assert not wrong, wrong
    assert sum(l.endswith("OK") for l in lines) >= 45


# --------------------------------------------------------------------------- kernels
def _ref(dy, w, cin):
    n, h, wd, _ = dy.shape
    return torch.nn.grad.conv2d_input((n, cin, h, wd), w.double().cpu(), dy.double().cpu().permute(0, 3, 1, 2),
                                      padding=1)


def _raw(dy, w, dx, cin):
    """The entry point on a caller-provided dx (possibly misaligned or inside a guard band)."""
    from unet import _C
    from unet import kernels as K
    from unet._C import ptr, stream
    f32 = dy.dtype == torch.float32
    n, h, wd, cout, ld = (K._nhwc32 if f32 else K._nhwc)(dy)
    _C.call("ub2_f32_conv_in_dgrad" if f32 else "ub2_conv_in_dgrad", ptr(dy), ld, ptr(w), ptr(dx), n, cin, h, wd,
            cout, stream())
    return dx


def _operands(n, cin, h, w, cout, dtype, seed, ld=None):
    g = torch.Generator().manual_seed(seed)
    ld = ld or cout
    full = torch.randn((n, h, w, ld), generator=g).to(dtype).cuda()
    wt = (torch.randn((cout, cin, 3, 3), generator=g) / (9 * cin) ** 0.5).cuda()
    return full[..., :cout], wt


def _parity(dy, w, cin, dx=None):
    from unet import kernels as K
    got = _raw(dy, w, dx, cin) if dx is not None else K.conv_in_dgrad(dy, w, cin)
    ref = _ref(dy, w, cin)
    diff = (got.double().cpu() - ref).abs()
    e = (diff.norm() / (ref.norm() + 1e-30)).item()
    return e, diff.max().item(), ref.abs().max().item()


@GPU
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("cout", [16, 48, 64])
@pytest.mark.parametrize("cin", [1, 2, 3, 4])
def test_kernel_parity(dtype, cin, cout):
    worst = (0.0, None)
    for n in (1, 3):
        for h, w in HW_GRID:
            dy, wt = _operands(n, cin, h, w, cout, dtype, seed=cin * 1000 + cout * 10 + n + h * w)
            e, dmax, rmax = _parity(dy, wt, cin)
            if e > worst[0]:
                worst = (e, (n, h, w, dmax, rmax))
            assert e <= 1e-5, (n, cin, h, w, cout, e)
    record(f"input-grad kernel parity [{'bf16' if dtype == torch.bfloat16 else 'fp32'}-Cin{cin}-Cout{cout}]",
           worst_rel_l2=worst[0], worst_case_nhw=list(worst[1][:3]) if worst[1] else None,
           worst_abs_err=worst[1][3] if worst[1] else 0.0, max_abs_ref=worst[1][4] if worst[1] else 0.0)


@GPU
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_kernel_parity_channel_slice_and_misaligned_dx(dtype):
    log = {}
    for cin, (h, w), cout, ld in ((1, (32, 36), 48, 64), (1, (17, 33), 16, 48), (3, (64, 64), 64, 128)):
        dy, wt = _operands(2, cin, h, w, cout, dtype, seed=7 + cout, ld=ld)
        assert dy.stride(2) == ld
        log[f"slice Cin{cin} {h}x{w} Cout{cout} ld{ld}"] = e = _parity(dy, wt, cin)[0]
        assert e <= 1e-5, (cin, h, w, cout, ld, e)
        # dx 4 bytes past a 16-byte boundary: the general variant
        buf = torch.empty(2 * cin * h * w + 1, device="cuda", dtype=torch.float32)
        dx = buf[1:].view(2, cin, h, w)
        assert dx.data_ptr() % 16 == 4
        log[f"dx+4B Cin{cin} {h}x{w} Cout{cout} ld{ld}"] = e = _parity(dy, wt, cin, dx=dx)[0]
        assert e <= 1e-5, ("misaligned dx", cin, h, w, cout, ld, e)
    if dtype == torch.float32:
        for n, (h, w) in ((1, (1, 1)), (3, (17, 33)), (2, (64, 64))):
            dy, wt = _operands(n, 7, h, w, 20, dtype, seed=70 + h)
            log[f"Cin7 Cout20 {n}x{h}x{w}"] = e = _parity(dy, wt, 7)[0]
            assert e <= 1e-5, (n, h, w, e)
        dy, wt = _operands(2, 1, 32, 64, 20, dtype, seed=77)      # Cout/4 = 5: the shared-memory fold
        log["Cin1 Cout20 2x32x64"] = e = _parity(dy, wt, 1)[0]
        assert e <= 1e-5, e
    record(f"input-grad kernel parity slices/misaligned [{dtype}]", **log)


@GPU
def test_variant_choice():
    """The shape grid reaches both variants: Cin 1, W % 4 == 0 and aligned pointers take the register-window
    kernel, anything else the general one (kernel names from the profiler)."""
    from torch.profiler import ProfilerActivity, profile
    from unet import kernels as K
    cases = []
    for dtype in (torch.bfloat16, torch.float32):
        dy, wt = _operands(1, 1, 16, 64, 64, dtype, 1)
        cases.append((lambda dy=dy, wt=wt: K.conv_in_dgrad(dy, wt, 1), True))
        dy48, wt48 = _operands(1, 1, 16, 64, 48, dtype, 1)
        cases.append((lambda dy=dy48, wt=wt48: K.conv_in_dgrad(dy, wt, 1), True))
        dx = torch.empty(16 * 64 + 1, device="cuda")[1:].view(1, 1, 16, 64)
        cases.append((lambda dy=dy, wt=wt, dx=dx: _raw(dy, wt, dx, 1), False))
        dy3, wt3 = _operands(1, 1, 16, 66, 64, dtype, 1)
        cases.append((lambda dy=dy3, wt=wt3: K.conv_in_dgrad(dy, wt, 1), False))
        dy2, wt2 = _operands(1, 2, 16, 64, 64, dtype, 1)
        cases.append((lambda dy=dy2, wt=wt2: K.conv_in_dgrad(dy, wt, 2), False))
    for fn, fast in cases:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "conv_in_dgrad" in e.name]
        assert len(names) == 1, names
        assert ("conv_in_dgrad4_kernel" in names[0]) == fast, names[0]


@GPU
def test_kernel_is_deterministic():
    from unet import kernels as K
    for dtype in (torch.bfloat16, torch.float32):
        for n, cin, h, w, cout in ((3, 1, 64, 64, 48), (2, 1, 64, 128, 64), (2, 3, 17, 33, 64)):
            dy, wt = _operands(n, cin, h, w, cout, dtype, seed=5)
            a, b = K.conv_in_dgrad(dy, wt, cin), K.conv_in_dgrad(dy, wt, cin)
            assert torch.equal(a, b), (dtype, n, cin, h, w, cout)


@GPU
def test_dx_writes_stay_inside_dx():
    """dx in the middle of a sentinel-filled buffer: odd shapes (general variant) and W % 4 == 0 (register-window
    variant, 16-byte-aligned dx) in both precisions; the bands on either side stay untouched."""
    guard = 1024                  # floats, 4 KiB
    for dtype in (torch.bfloat16, torch.float32):
        for n, cin, h, w, cout in ((1, 1, 3, 5, 16), (3, 2, 17, 33, 48), (2, 1, 32, 36, 64), (3, 1, 8, 4, 48),
                                   (1, 4, 64, 64, 16)):
            if dtype == torch.bfloat16 and cin > 4:
                continue
            dy, wt = _operands(n, cin, h, w, cout, dtype, seed=11)
            numel = n * cin * h * w
            buf = torch.full((guard + numel + guard,), float("nan"), device="cuda")
            sentinel = buf.clone()
            dx = buf[guard:guard + numel].view(n, cin, h, w)
            e, _, _ = _parity(dy, wt, cin, dx=dx)
            torch.cuda.synchronize()
            assert e <= 1e-5, (dtype, n, cin, h, w, cout, e)
            lo, hi = buf[:guard], buf[guard + numel:]
            assert torch.equal(lo.view(torch.int32), sentinel[:guard].view(torch.int32)), (dtype, n, cin, h, w)
            assert torch.equal(hi.view(torch.int32), sentinel[guard + numel:].view(torch.int32)), (dtype, n, cin, h, w)


@GPU
def test_offsets_past_2_pow_31():
    """bf16 dy of 130 x 512^2 x 64 (2.2e9 elements, 4.4 GB): images 0, 64 and 129 against the per-image
    reference, through both variants (aligned dx: register window; dx 4 bytes off: general)."""
    from unet import kernels as K
    n, h, w, cout = 130, 512, 512, 64
    assert n * h * w * cout > 2 ** 31
    wt = (torch.randn((cout, 1, 3, 3), generator=torch.Generator().manual_seed(3)) / 3).cuda()
    dy = torch.empty((n, h, w, cout), device="cuda", dtype=torch.bfloat16)
    gen = torch.Generator(device="cuda").manual_seed(4)
    for i in range(0, n, 16):
        dy[i:i + 16].normal_(generator=gen)
    fast = K.conv_in_dgrad(dy, wt, 1)
    buf = torch.empty(n * h * w + 1, device="cuda")
    general = _raw(dy, wt, buf[1:].view(n, 1, h, w), 1)
    torch.cuda.synchronize()
    log = {}
    for i in (0, 64, 129):
        ref = _ref(dy[i:i + 1], wt, 1)
        for tag, got in (("fast", fast), ("general", general)):
            e = ((got[i:i + 1].double().cpu() - ref).norm() / ref.norm()).item()
            log[f"{tag} image {i}"] = e
            assert e <= 1e-5, (tag, i, e)
    record("input-grad kernel 64-bit offsets 130x512x512x64 bf16", **log)
    del dy, fast, general, buf
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------- modules
@GPU
@pytest.mark.parametrize("cin,cout", [(1, 64), (3, 48)])
@pytest.mark.parametrize("training", [True, False])
def test_double_conv_stem_input_grad(cin, cout, training):
    from unet.models.layers import DoubleConv
    check_module(DoubleConv(cin, cout), lambda x, sd, tr: O.double_conv(x, sd, "m", tr), [_x((2, cin, 32, 32), 2)],
                 training, input_needs_grad=True, tag=f"input-grad DoubleConv({cin},{cout}) training={training}")


@GPU
@pytest.mark.parametrize("all_active", [True, False], ids=["all-active", "random"])
@pytest.mark.parametrize("cin,cout", [(1, 64), (3, 48)])
@pytest.mark.parametrize("training", [True, False])
def test_double_conv_stem_input_grad_fp32(cin, cout, training, all_active):
    import unet
    from test_fp32_train_gpu import check_module_f32
    from unet.models.layers import DoubleConv
    unet.set_precision("tf32")
    try:
        check_module_f32(DoubleConv(cin, cout), lambda x, sd, tr: O.double_conv(x, sd, "m", tr),
                         [_x((2, cin, 32, 32), 2)], training, input_needs_grad=True, all_active=all_active,
                         tag=f"input-grad DoubleConv({cin},{cout}) training={training}")
    finally:
        unet.set_precision("bf16")


# --------------------------------------------------------------------------- whole network
def _all_active(sd):
    """Every BatchNorm bias +8 (the gate's psi BatchNorm, which feeds a sigmoid, stays): no ReLU near a decision."""
    for k in sd:
        if k.endswith(".bias") and k.replace(".bias", ".running_mean") in sd and ".psi." not in k:
            sd[k].fill_(8.0)
    return sd


def _net_input_grad(model, x, gouts):
    xc = x.cuda().requires_grad_(True)
    out = model(xc)
    outs = out if isinstance(out, (list, tuple)) else [out]
    loss = sum((o * g.cuda()).sum() for o, g in zip(outs, gouts))
    (gx,) = torch.autograd.grad(loss, xc)
    return gx


def _oracle_input_grad(sd, x, gouts, training, storage=False, **cfg):
    xo = x.clone().requires_grad_(True)
    with O.bf16_storage(storage):
        out = O.unet_forward(xo, O.clone_state(sd), training=training, **cfg)
    outs = out if isinstance(out, (list, tuple)) else [out]
    loss = sum((o * g).sum() for o, g in zip(outs, gouts))
    (gx,) = torch.autograd.grad(loss, xo)
    return gx


def _gouts(model, x, seed):
    with torch.no_grad():
        out = model(x.cuda())
    outs = out if isinstance(out, (list, tuple)) else [out]
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(o.shape, generator=g).to(torch.bfloat16).float() for o in outs]


NETS = [(True, 32, {}), (True, 16, {}), (False, 32, {}), (False, 16, {}),
        (True, 32, {"deep_supervision": True}), (False, 32, {"bilinear": False})]


def _net_id(p):
    attention, bf, kw = p
    return f"{'attention' if attention else 'unet'}-{bf}" + "".join(f"-{k}={v}" for k, v in kw.items())


@GPU
@pytest.mark.parametrize("all_active", [False, True], ids=["random", "all-active"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("net", NETS, ids=[_net_id(p) for p in NETS])
def test_network_input_grad_bf16(net, training, all_active):
    """dL/dx of the whole bf16 network against the oracle's autograd.  The bf16-storage oracle (the product's
    rounding points) vs the fp32 oracle is the floor that any bf16 implementation sits at.  Where that floor is
    within 2e-2 the CUDA result takes the module gates: rel-L2 <= 2e-2 vs the bf16-storage oracle, cosine >= 0.995
    vs fp32.  Where it is larger — random parameters in train mode: ReLU decisions taken on batch statistics flip
    between any two correct implementations, measured 0.62 rel-L2 between the two oracles for AttentionUNet-32 —
    the CUDA result is gated relative to the floor: no further than 1.5 floors from either oracle.  The all-active
    parameters (every BatchNorm bias +8, no ReLU near a decision) keep the module gates in every mode."""
    attention, bf, kw = net
    model, sd, cfg = _build(attention, bf, 31, **kw)
    if all_active:
        sd = _all_active(sd)
        model.load_state_dict(sd)
    ocfg = {k: v for k, v in cfg.items() if k in ("bilinear", "deep_supervision")}
    x, _ = O.synthetic_batch(2, 64, 64, seed=8)
    model = model.cuda().train(training)
    gouts = _gouts(copy.deepcopy(model), x, 5)       # a copy: its train-mode forward moves only its own BN buffers
    got = _net_input_grad(model, x, gouts).cpu()
    ref = _oracle_input_grad(sd, x, gouts, training, attention=attention, **ocfg)
    st = _oracle_input_grad(sd, x, gouts, training, storage=True, attention=attention, **ocfg)
    floor, floor_cos = rel_l2(st, ref), cosine(st, ref)
    e_model, e_fp32, c_fp32 = rel_l2(got, st), rel_l2(got, ref), cosine(got, ref)
    relative = floor > 2e-2
    record(f"input-grad network bf16 [{_net_id(net)}-{'train' if training else 'eval'}"
           f"{'-all-active' if all_active else ''}] 2x1x64x64",
           rel_l2_vs_bf16_model=e_model, cos_vs_fp32=c_fp32, rel_l2_vs_fp32=e_fp32,
           floor_rel_l2_bf16_model_vs_fp32=floor, floor_cos_bf16_model_vs_fp32=floor_cos,
           gated_relative_to_floor=relative)
    assert torch.isfinite(got).all()
    if relative:
        assert e_model <= 1.5 * floor and e_fp32 <= 1.5 * floor, (e_model, e_fp32, floor)
    else:
        assert e_model <= 2e-2, (e_model, floor)
        assert c_fp32 >= 0.995, (c_fp32, floor_cos)


@GPU
@pytest.mark.parametrize("net", NETS[:4], ids=[_net_id(p) for p in NETS[:4]])
def test_network_input_grad_fp32_all_active(net):
    """fp32 / TF32 mode, eval, every ReLU active: dL/dx within 1e-3 of the fp32 oracle.

    The stem's data gradient dx and its weight gradient are both computed from the same upstream gradient dy of
    the stem, which every other block of the network produces.  So the stem weight gradient's error against the
    oracle measures the error that dy already carries into the stem: where it exceeds the 1e-3 gate, dx is held to
    1.5 times that error instead, which still fails a wrong data-gradient kernel (the kernel alone is checked at
    1e-5 above) but does not charge it for the blocks in front of it.  Both numbers are logged."""
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
    (O.unet_forward(xo, w, attention=attention, training=False) * gouts[0]).sum().backward()
    e, e_w = rel_l2(got, xo.grad), rel_l2(got_w, w[stem].grad)
    gate = max(1e-3, 1.5 * e_w)
    record(f"input-grad network fp32 all-active [{_net_id(net)}-eval] 2x1x64x64", rel_l2_vs_fp32=e,
           stem_weight_grad_rel_l2_vs_fp32=e_w, gate=gate)
    assert e <= gate, (e, e_w)


@GPU
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_frozen_parameters_saliency(precision):
    """Eval mode with every parameter frozen (a saliency map of a trained model): the input gradient is
    bit-identical to the one with trainable parameters, no parameter gets a .grad, BN buffers stay."""
    import unet
    model, _, _ = _build(True, 32, 33)
    x, _ = O.synthetic_batch(2, 64, 64, seed=9)
    unet.set_precision(precision)
    try:
        model = model.cuda().eval()
        buffers = {k: v.clone() for k, v in model.named_buffers()}
        xa = x.cuda().requires_grad_(True)
        (ga,) = torch.autograd.grad(model(xa).sum(), xa)
        for p in model.parameters():
            p.requires_grad_(False)
        xb = x.cuda().requires_grad_(True)
        (gb,) = torch.autograd.grad(model(xb).sum(), xb)
    finally:
        unet.set_precision("bf16")
    assert torch.equal(ga, gb)
    assert ga.abs().sum() > 0
    assert all(p.grad is None for p in model.parameters())
    for k, v in model.named_buffers():
        assert torch.equal(v, buffers[k]), k


@GPU
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_two_stage_cascade_trains_the_first_stage(precision):
    """Stage 2 = UNet(n_channels=3) on cat(x, softmax(stage1(x))): one training step (train mode) reaches stage 1,
    and its parameter gradients match the same composition of oracle calls.  Every BatchNorm bias is +8 (no ReLU
    near a decision): in bf16 train mode at random init, ReLU flips make two correct implementations disagree
    (SURVEY App. C), and this test is about the arithmetic that carries the gradient through the stem."""
    import unet
    from unet.models import UNet
    cfg1 = dict(n_channels=1, n_classes=2, bilinear=True, base_features=16, attention=False)
    cfg2 = dict(n_channels=3, n_classes=2, bilinear=True, base_features=16, attention=False)
    sd1, sd2 = _all_active(O.synthetic_state_dict(41, **cfg1)), _all_active(O.synthetic_state_dict(42, **cfg2))
    s1, s2 = UNet(1, 2, True, 16), UNet(3, 2, True, 16)
    s1.load_state_dict(sd1)
    s2.load_state_dict(sd2)
    x, _ = O.synthetic_batch(2, 64, 64, seed=10)
    g = torch.Generator().manual_seed(6)
    gout = torch.randn((2, 2, 64, 64), generator=g).to(torch.bfloat16).float()
    unet.set_precision(precision)
    try:
        s1, s2 = s1.cuda().train(), s2.cuda().train()
        opt = torch.optim.SGD(list(s1.parameters()) + list(s2.parameters()), lr=1e-3)
        xc = x.cuda()
        out = s2(torch.cat([xc, torch.softmax(s1(xc), 1)], 1))
        (out * gout.cuda()).sum().backward()
        grads = {k: p.grad.detach().cpu().clone() for k, p in s1.named_parameters()}
        before = [p.detach().clone() for p in s1.parameters()]
        opt.step()
        moved = any(not torch.equal(a, b) for a, b in zip(before, s1.parameters()))
    finally:
        unet.set_precision("bf16")
    assert moved

    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd1.items()
              if v.is_floating_point() and not k.endswith(("running_mean", "running_var"))}
    w1 = dict(O.clone_state(sd1), **params)
    o1 = O.unet_forward(x, w1, attention=False, training=True)
    o2 = O.unet_forward(torch.cat([x, torch.softmax(o1, 1)], 1), O.clone_state(sd2), attention=False, training=True)
    (o2 * gout).sum().backward()
    scale = max(float(p.grad.norm()) for p in params.values())
    gate = 0.995 if precision == "bf16" else 0.999
    cos, skipped = {}, []
    for k, got in grads.items():
        r = params[k].grad
        assert torch.isfinite(got).all(), k
        if float(r.norm()) < 1e-5 * scale:      # zero in exact arithmetic (a bias in front of a train-mode BN)
            skipped.append(k)
            continue
        cos[k] = cosine(got, r)
    worst = min(cos, key=cos.get)
    record(f"input-grad cascade [{precision}] stage-1 parameter gradients all-active", cos_min=cos[worst],
           cos_min_param=worst, cos_median=sorted(cos.values())[len(cos) // 2], zero_in_exact_arithmetic=skipped)
    assert len(cos) > 20
    assert cos[worst] >= gate, (worst, cos[worst])


@GPU
def test_graph_captured_saliency_equals_eager():
    """Eval forward + backward to the input of AttentionUNet, captured with torch.cuda.graph and replayed: bit-
    identical to eager (the new path neither synchronises nor allocates outside the graph's pool)."""
    model, _, _ = _build(True, 32, 34)
    model = model.cuda().eval()
    for p in model.parameters():
        p.requires_grad_(False)
    x, _ = O.synthetic_batch(2, 64, 64, seed=12)
    xs = x.cuda().requires_grad_(True)

    def step():
        (gx,) = torch.autograd.grad(model(xs).sum(), xs)
        return gx

    eager = step().clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    with torch.no_grad():
        xs.copy_(torch.flip(x, [3]).cuda())
    graph.replay()
    flipped = static.clone()
    with torch.no_grad():
        xs.copy_(x.cuda())
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static, eager)
    assert not torch.equal(flipped, eager)
