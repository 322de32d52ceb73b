"""Channel counts that are not multiples of 16: the per-tap tensor-core kernels pad K (input channels, multiples of 8
per source) and N (output channels, multiples of 8) internally, and the modules route such layers to them.

Kernels: every case against a float64 convolution of the same rounded operands, at test_conv_gpu.py's tolerance.
Input channels past a source's count hold NaN in memory: they must be read through the tensor map's zero fill.
Output buffers have a channel stride above Cout, filled with a sentinel that must survive.
Modules and whole networks: against the oracle, with the gates of test_modules_gpu.py / test_fp32_train_gpu.py."""
import itertools

import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O
from parity_log import record
from test_fp32_train_gpu import check_module_f32
from test_modules_gpu import _x, check_module, cosine, rel_l2

pytestmark = pytest.mark.gpu

N, H, W = 2, 11, 13          # odd sizes: masked pixel tiles
SENTINEL = -12352.0          # exactly representable in bf16


def _tf32(x):
    i = x.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _padded(x, dtype, extra=8):
    """(N,H,W,C) values in a buffer whose channel stride is the next multiple of 8 plus `extra`, the rest NaN."""
    c = x.shape[3]
    ld = (c + 7) // 8 * 8 + extra
    buf = torch.full((*x.shape[:3], ld), float("nan"), dtype=dtype, device="cuda")
    buf[..., :c] = x.to(dtype).cuda()
    return buf[..., :c]


def _ref(xs, w, taps):
    """float64 conv of NHWC sources (concatenated) with OIHW w -> NHWC."""
    x = torch.cat([t.double().cpu() for t in xs], 3).permute(0, 3, 1, 2)
    return F.conv2d(x, w.double().cpu(), padding=1 if taps == 9 else 0).permute(0, 2, 3, 1)


def _close(got, ref, what):
    got = got.double().cpu()
    err = (got - ref).abs()
    bad = (err > 2.0 ** -7 * ref.abs() + 2e-2).sum().item()
    assert bad == 0, f"{what}: {bad} / {ref.numel()} mismatches, max err {err.max().item():.4g}"


def _fwd_pack(w):
    cout, cin, k, _ = w.shape
    return w.permute(0, 2, 3, 1).reshape(cout, k * k, cin).contiguous()


SHAPES = [(c0, c1, cout, taps) for c0, c1, cout, taps in itertools.product((8, 24, 40), (0, 8, 24), (8, 24, 40, 72), (1, 9))]


@pytest.mark.parametrize("cout", [8, 24, 72])
@pytest.mark.parametrize("taps", [1, 9])
def test_five_channel_source(cout, taps):
    """C0 = 5, C1 = 3: the weight gradient pads each source to whole A sub-boxes and takes any count.  The forward
    kernel reads each source's weight-pack columns with TMA, whose boxes start on 16 bytes: it refuses on the host
    (the modules zero-pad such a network input to 8 channels instead)."""
    from unet import kernels as K
    g = torch.Generator().manual_seed(cout + taps)
    k = 3 if taps == 9 else 1
    xs = [torch.randn(N, H, W, c, generator=g).to(torch.bfloat16) for c in (5, 3)]
    dev = [_padded(x, torch.bfloat16) for x in xs]
    w = torch.randn(cout, 8, k, k, generator=g).to(torch.bfloat16)
    with pytest.raises(RuntimeError, match=r"code -2"):
        K.conv_fwd(dev[0], _fwd_pack(w).cuda(), taps, x1=dev[1])
    dy = torch.randn(N, H, W, cout, generator=g).to(torch.bfloat16)
    part = K.conv_wgrad(dev[0], _padded(dy, torch.bfloat16), taps, x1=dev[1])
    assert K.last_conv_variant() == 11
    gw = torch.empty((cout, 8, k, k), device="cuda")
    K.wgrad_reduce(part, cout, 8, taps, gw)
    xr = torch.cat([t.double() for t in xs], 3).permute(0, 3, 1, 2)
    wr = w.double().requires_grad_(True)
    F.conv2d(xr, wr, padding=k // 2).backward(dy.double().permute(0, 3, 1, 2))
    e = (gw.double().cpu() - wr.grad).abs().max().item()
    assert e <= 1e-4 * wr.grad.abs().max().item() + 1e-4, f"weight gradient max err {e:.3g}"


@pytest.mark.parametrize("c0,c1,cout,taps", SHAPES)
def test_kernels(c0, c1, cout, taps):
    from unet import kernels as K
    g = torch.Generator().manual_seed(c0 * 1000 + c1 * 100 + cout + taps)
    k = 3 if taps == 9 else 1
    ctot = c0 + c1
    xs = [torch.randn(N, H, W, c, generator=g).to(torch.bfloat16) for c in (c0, c1) if c]
    w = (torch.randn(cout, ctot, k, k, generator=g) / (taps * ctot) ** 0.5).to(torch.bfloat16)
    dev = [_padded(x, torch.bfloat16) for x in xs]
    x1 = dev[1] if c1 else None
    wf = _fwd_pack(w).cuda()
    ref = _ref(xs, w, taps)

    # forward with BatchNorm statistics, into a guard-banded output
    ldo = cout + 16
    out = torch.full((N, H, W, ldo), SENTINEL, dtype=torch.bfloat16, device="cuda")
    y, st = K.conv_fwd(dev[0], wf, taps, x1=x1, out=out[..., :cout], stats=True)
    assert K.last_conv_variant() == 1
    _close(y, ref, "forward")
    assert (out[..., cout:] == SENTINEL).all(), "forward wrote past Cout"
    o = y.double().cpu().reshape(-1, cout)
    s = st.sum(0).cpu()
    assert torch.allclose(s[0], o.sum(0), rtol=1e-4, atol=1e-2)
    assert torch.allclose(s[1], (o * o).sum(0), rtol=1e-4, atol=1e-2)

    # eval epilogue: per-channel affine + ReLU
    scale = torch.rand(cout, generator=g) + 0.5
    shift = torch.randn(cout, generator=g)
    out.fill_(SENTINEL)
    K.conv_fwd(dev[0], wf, taps, x1=x1, out=out[..., :cout], scale=scale.cuda(), shift=shift.cuda(), relu=True)
    _close(out[..., :cout], torch.relu(ref * scale.double() + shift.double()), "affine+relu")
    assert (out[..., cout:] == SENTINEL).all()

    # accumulate into the destination
    base = torch.randn(N, H, W, cout, generator=g).to(torch.bfloat16)
    out[..., :cout] = base.cuda()
    K.conv_fwd(dev[0], wf, taps, x1=x1, out=out[..., :cout], accumulate=True)
    _close(out[..., :cout], ref + base.double(), "accumulate")
    assert (out[..., cout:] == SENTINEL).all()

    # weight gradient + fold
    dy = torch.randn(N, H, W, cout, generator=g).to(torch.bfloat16)
    dyd = _padded(dy, torch.bfloat16)
    part = K.conv_wgrad(dev[0], dyd, taps, x1=x1)
    assert K.last_conv_variant() == 11
    gw = torch.empty((cout, ctot, k, k), device="cuda")
    K.wgrad_reduce(part, cout, ctot, taps, gw)
    xr = torch.cat([t.double() for t in xs], 3).permute(0, 3, 1, 2).requires_grad_(True)
    wr = w.double().requires_grad_(True)
    F.conv2d(xr, wr, padding=k // 2).backward(dy.double().permute(0, 3, 1, 2))
    e = (gw.double().cpu() - wr.grad).abs().max().item()
    assert e <= 1e-4 * wr.grad.abs().max().item() + 1e-4, f"weight gradient max err {e:.3g}"

    # data gradient of the (virtual) concat: output split over two guard-banded tensors
    _, wd = K.pack_conv_weight(w.float().cuda().contiguous(), want_fwd=False)
    dref = xr.grad.permute(0, 2, 3, 1)
    b0 = torch.full((N, H, W, c0 + 8), SENTINEL, dtype=torch.bfloat16, device="cuda")
    b1 = torch.full((N, H, W, c1 + 8), SENTINEL, dtype=torch.bfloat16, device="cuda") if c1 else None
    K.conv_fwd(dyd, wd, taps, out=b0[..., :c0], out1=b1[..., :c1] if c1 else None, split=c0)
    assert K.last_conv_variant() == 1
    _close(b0[..., :c0], dref[..., :c0], "dgrad split 0")
    assert (b0[..., c0:] == SENTINEL).all()
    if c1:
        _close(b1[..., :c1], dref[..., c0:], "dgrad split 1")
        assert (b1[..., c1:] == SENTINEL).all()

    # the TF32 instance (fp32 inference): operands rounded to TF32 on both sides, output rounded to TF32
    xt = [_tf32(torch.randn(N, H, W, c, generator=g)) for c in (c0, c1) if c]
    wt = _tf32(torch.randn(cout, ctot, k, k, generator=g) / (taps * ctot) ** 0.5)
    dt = [_padded(x, torch.float32) for x in xt]
    yt = K.conv_fwd_tf32(dt[0], dt[1] if c1 else None, _fwd_pack(wt).cuda(), cout, taps)
    assert K.last_conv_variant() == 1
    rt = _ref(xt, wt, taps)
    e = (yt.double().cpu() - rt).abs()
    assert (e <= 2.0 ** -10 * rt.abs() + 1e-4 * rt.abs().max()).all(), f"tf32 max err {e.max().item():.3g}"


# ------------------------------------------------------------------------------------------------ modules
@pytest.fixture(params=["bf16", "tf32"])
def precision(request):
    import unet
    unet.set_precision(request.param)
    yield request.param
    unet.set_precision("bf16")


@pytest.fixture
def all_active_bf16(monkeypatch):
    """check_module with every BatchNorm bias +8, so that no ReLU sits near a decision.  With random parameters the
    24-channel DoubleConv / Down sit as far from the bf16-storage oracle (input gradient 5-7 % rel-L2) as that oracle
    sits from the fp32 one (ReLU decisions taken on batch statistics flip between any two implementations);
    all-active parameters make the bf16 gates discriminating (measured: every gradient cosine >= 0.9998)."""
    import test_modules_gpu as M
    orig = M.randomise

    def randomise(module, seed):
        module = orig(module, seed)
        with torch.no_grad():
            for mod in module.modules():
                if isinstance(mod, torch.nn.BatchNorm2d):
                    mod.bias.fill_(8.0)
        return module

    monkeypatch.setattr(M, "randomise", randomise)


def _check(precision, module, oracle_fn, inputs, training=True):
    if precision == "bf16":
        check_module(module, oracle_fn, inputs, training)
    else:
        check_module_f32(module, oracle_fn, inputs, training, all_active=True)


def test_double_conv_24(all_active_bf16, precision):
    from unet.models.layers import DoubleConv
    _check(precision, DoubleConv(24, 24), lambda x, sd, tr: O.double_conv(x, sd, "m", tr), [_x((2, 24, 48, 44), 1)])


def test_down_24_48(all_active_bf16, precision):
    """bf16 in eval mode: with all-active parameters the train-mode running-mean gate (atol 2e-3) measures the bf16
    rounding of large pre-activations, not the kernels; DoubleConv above covers train mode."""
    from unet.models.layers import Down
    _check(precision, Down(24, 48), lambda x, sd, tr: O.down(x, sd, "m", tr), [_x((2, 24, 64, 62), 2)],
           training=precision != "bf16")


@pytest.mark.parametrize("bilinear", [True, False])
def test_up_48_24(precision, bilinear):
    from unet.models.layers import Up
    c_low = 24 if bilinear else 48
    _check(precision, Up(48, 24, bilinear), lambda x1, x2, sd, tr: O.up_block(x1, x2, sd, "m", False, bilinear, tr),
           [_x((2, c_low, 20, 21), 3), _x((2, 24, 40, 43), 4)])


def test_attention_up_48_24(precision):
    """AttentionUp(48, 24): the gate has 12 inter-channels (zero-padded to 16)."""
    from unet.models.layers import AttentionUp
    m = AttentionUp(48, 24, True)
    assert m.attention.W_g[0].weight.shape[0] == 12
    _check(precision, m, lambda x1, x2, sd, tr: O.up_block(x1, x2, sd, "m", True, True, tr),
           [_x((2, 24, 20, 20), 5), _x((2, 24, 40, 40), 6)])


# ------------------------------------------------------------------------------------------------ networks
NETS = [  # attention, n_channels, n_classes, bilinear, base_features, deep_supervision
    (True, 1, 2, True, 24, False),
    (False, 1, 2, False, 24, False),
    (True, 1, 2, True, 8, False),
    (True, 1, 2, False, 40, True),
    (True, 5, 2, True, 32, False),
    (False, 7, 3, True, 16, False),
]


def _net_id(p):
    a, nc, ncl, bil, bf, ds = p
    return f"{'attention' if a else 'unet'}-{nc}ch-{ncl}cls-{'bilinear' if bil else 'convt'}-{bf}" + ("-ds" if ds else "")


def _build_net(p, seed):
    from unet.models import AttentionUNet, UNet
    attention, nc, ncl, bil, bf, ds = p
    cfg = dict(n_channels=nc, n_classes=ncl, bilinear=bil, base_features=bf, attention=attention)
    if ds:
        cfg["deep_supervision"] = True
    sd = O.synthetic_state_dict(seed, **cfg)
    model = AttentionUNet(nc, ncl, bil, bf, deep_supervision=ds) if attention else UNet(nc, ncl, bil, bf)
    model.load_state_dict(sd, strict=True)
    return model, sd, {k: v for k, v in cfg.items() if k in ("bilinear", "deep_supervision")}


@pytest.mark.parametrize("net", NETS, ids=[_net_id(p) for p in NETS])
def test_network(net, precision):
    from unet.utils.loss import DeepSupervisionLoss, DiceBCELoss
    attention, nc, ncl = net[:3]
    model, sd, ocfg = _build_net(net, 51)
    x, t = O.synthetic_batch(2, 64, 64, seed=13, n_channels=nc, fg_fraction=0.05)
    model = model.cuda().eval()
    with torch.no_grad():
        logits = model(x.cuda())
    ref = O.unet_forward(x, sd, attention=attention, training=False, **ocfg)
    assert logits.shape == ref.shape == (2, ncl, 64, 64)
    e = rel_l2(logits, ref)
    assert e <= (2e-2 if precision == "bf16" else 1e-3), f"eval logits rel-L2 {e:.3e}"

    model.train()
    out = model(x.cuda())
    loss = DeepSupervisionLoss(DiceBCELoss())(out, t.cuda())
    loss.backward()
    ref_loss, _, ref_grads = O.train_grads(x, t, O.clone_state(sd), attention=attention, **ocfg)
    cos = {k: cosine(p.grad, ref_grads[k]) for k, p in model.named_parameters() if p.numel() > 1}
    record(f"channels network [{_net_id(net)}] [{precision}]", eval_logits_rel_l2=e, loss=loss.item(),
           loss_oracle=ref_loss.item(), grad_cos_min=min(cos.values()))
    assert abs(loss.item() - ref_loss.item()) <= (5e-2 if precision == "bf16" else 1e-4) * abs(ref_loss.item())
    for k, p in model.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape and torch.isfinite(p.grad).all(), k
    if precision == "tf32":
        assert min(cos.values()) >= 0.999, min(cos, key=cos.get)
    got_sd = model.state_dict()
    assert list(got_sd.keys()) == list(sd.keys())
    assert all(got_sd[k].shape == sd[k].shape for k in sd)


def test_input_grad_five_channels(precision):
    """dL/dx of AttentionUNet(n_channels=5) in eval, every ReLU active (BatchNorm biases +8): against the oracle's
    autograd, with test_input_grad_gpu.py's gates (bf16: relative to the bf16-storage oracle; tf32: 1e-3, or 1.5 times
    the stem weight gradient's error, which measures what the upstream gradient already carries into the stem)."""
    net = (True, 5, 2, True, 32, False)
    model, sd, ocfg = _build_net(net, 52)
    for k in sd:
        if k.endswith(".bias") and k.replace(".bias", ".running_mean") in sd and ".psi." not in k:
            sd[k].fill_(8.0)
    model.load_state_dict(sd)
    model = model.cuda().eval()
    x, _ = O.synthetic_batch(2, 64, 64, seed=14, n_channels=5)
    g = torch.randn(2, 2, 64, 64, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).float()
    xc = x.cuda().requires_grad_(True)
    (model(xc) * g.cuda()).sum().backward()
    got = xc.grad
    stem = "inc.double_conv.0.weight"
    got_w = dict(model.named_parameters())[stem].grad
    assert got.dtype == x.dtype and got.shape == x.shape

    def oracle(storage, want_w=False):
        xo = x.clone().requires_grad_(True)
        w = O.clone_state(sd)
        w[stem].requires_grad_(True)
        with O.bf16_storage(storage):
            (O.unet_forward(xo, w, attention=True, training=False, **ocfg) * g).sum().backward()
        return (xo.grad, w[stem].grad) if want_w else xo.grad

    if precision == "bf16":
        e = rel_l2(got, oracle(True))
        record("channels input-grad n_channels=5 [bf16]", rel_l2_vs_bf16_model=e, cos_vs_fp32=cosine(got, oracle(False)))
        assert e <= 2e-2 and cosine(got, oracle(False)) >= 0.995
    else:
        ref, ref_w = oracle(False, want_w=True)
        e, e_w = rel_l2(got, ref), rel_l2(got_w, ref_w)
        record("channels input-grad n_channels=5 [tf32]", rel_l2_vs_fp32=e, stem_weight_grad_rel_l2_vs_fp32=e_w)
        assert e <= max(1e-3, 1.5 * e_w), (e, e_w)


def test_trainer_graph_and_one_launch_pack():
    """BatchShardedTrainer with a captured step on AttentionUNet(base_features=24): graph replays are bit-identical
    to eager steps, and every conv weight the tensor cores read unpadded comes from the one-launch pack."""
    from unet.models import AttentionUNet
    from unet.optim import FusedAdamW
    from unet.parallel import BatchShardedTrainer
    from unet.utils.loss import DiceBCELoss

    x, t = O.synthetic_batch(2, 64, 64, seed=9, fg_fraction=0.05)
    x, t = x.cuda(), t.cuda()
    results = []
    for use_graph in (False, True):
        torch.manual_seed(3)
        model = AttentionUNet(1, 2, True, 24).cuda()
        tr = BatchShardedTrainer(model, DiceBCELoss(), FusedAdamW(model.parameters(), lr=1e-3), grad_clip=1.0,
                                 cuda_graph=use_graph, graph_warmup=2)
        losses = [tr.step(x, t).item() for _ in range(5)]   # 2 warm-up steps, then 3 captured / replayed ones
        results.append((losses, [p.detach().clone() for p in model.parameters()]))
        packed = [m.weight for m in model.modules() if isinstance(m, torch.nn.Conv2d)
                  and m.weight.shape[0] % 8 == 0 and m.weight.shape[1] % 8 == 0]
        assert len(packed) == 23
        assert all(tr._packer.get(w) is not None for w in packed)
    (l0, p0), (l1, p1) = results
    assert l0 == l1, (l0, l1)
    assert all(torch.equal(a, b) for a, b in zip(p0, p1))


@pytest.mark.parametrize("precision_name", ["bf16", "tf32"])
def test_unsupported_width_is_a_clear_error(precision_name):
    import unet
    from unet.models import AttentionUNet
    model = AttentionUNet(1, 2, True, 12)
    model.load_state_dict(O.synthetic_state_dict(1, n_channels=1, n_classes=2, bilinear=True, base_features=12,
                                                 attention=True))
    model = model.cuda().eval()
    unet.set_precision(precision_name)
    try:
        with pytest.raises(RuntimeError, match=r"12 channels.*multiple of 8"):
            with torch.no_grad():
                model(torch.zeros(1, 1, 32, 32, device="cuda"))
    finally:
        unet.set_precision("bf16")
