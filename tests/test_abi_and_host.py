"""CPU: the C-ABI library loads and exports every symbol include/unetb200.h declares, and the
host-side mirror of the reference interface behaves (no compute calls: there is no GPU here)."""
import copy
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import unet_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "unetb200.h")) as f:
        text = f.read()
    return sorted(set(re.findall(r"\b(ub2_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from unet import _C
    lib = _C.lib()
    names = _declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/unetb200.h but not exported"
    assert lib.ub2_version() >= 100


def test_header_declares_every_exported_symbol():
    import subprocess
    from unet import _C
    out = subprocess.run(["nm", "-D", "--defined-only", _C.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r"\b(ub2_[a-z0-9_]+)\b", out)))
    assert exported == _declared_symbols()


def test_every_entry_point_is_typed_from_the_header():
    """lib() sets restype and argtypes of every prototype from include/unetb200.h, once: SIGNATURES is that
    table and the loaded functions carry it."""
    from unet import _C
    lib = _C.lib()
    assert sorted(_C.SIGNATURES) == _declared_symbols() and len(_C.SIGNATURES) == 89
    for name, params in _C.SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is ctypes.c_int, name
        assert fn.argtypes == [t for _, t in params], name
        assert all(p.isidentifier() and p not in ("in", "from", "lambda") for p, _ in params), name
    assert _C.SIGNATURES["ub2_version"] == []
    assert _C.SIGNATURES["ub2_seg_stats_blocks"] == [("N", ctypes.c_int), ("HW", ctypes.c_longlong)]
    assert [t for _, t in _C.SIGNATURES["ub2_bn_finalize"]][3::7] == [ctypes.c_double, ctypes.c_float]
    assert _C.SIGNATURES["ub2_conv_fwd"][-1] == ("stream", ctypes.c_void_p)


def test_wrongly_typed_arguments_raise_before_the_call():
    """With argtypes from the header a float for an int, or for a pointer, is refused by ctypes (ArgumentError)
    instead of reaching C as garbage; a refused _C.call counts no launch."""
    from unet import _C
    lib = _C.lib()
    assert lib.ub2_outc_rows(4, 64, 64, 64) > 0
    with pytest.raises(ctypes.ArgumentError):
        lib.ub2_outc_rows(4.0, 64, 64, 64)
    with pytest.raises(ctypes.ArgumentError):
        lib.ub2_f32_channel_rows(4096, 16.0)
    with pytest.raises(ctypes.ArgumentError):
        lib.ub2_resize_planes_fwd(0.5, None, 1, 1, 1, 1, 1, None)
    with pytest.raises(TypeError):
        lib.ub2_outc_rows(4, 64, 64)
    launches = _C.LAUNCHES
    with pytest.raises(ctypes.ArgumentError):
        _C.call("ub2_f32_scalar_stats", None, 64.0, None, 1, None)
    assert _C.LAUNCHES == launches


@pytest.mark.parametrize("decl,error", [
    ("int ub2_f(float* x, short n, void* stream);", "unknown parameter type"),
    ("int ub2_f(const float*, int n);", "unnamed parameter"),
    ("int ub2_f(int);", "unnamed parameter"),
    ("long ub2_f(int n);", "not an int-returning prototype"),
    ("int ub2_f(int n); int ub2_f(int m);", "declared twice"),
])
def test_header_parser_refuses_what_it_cannot_type(tmp_path, decl, error):
    from unet import _C
    hdr = tmp_path / "unetb200.h"
    hdr.write_text("/* int ub2_comment(void); */\nint ub2_ok(const long long* p, long long n, double d);\n" + decl + "\n")
    with pytest.raises(RuntimeError, match=error):
        _C._parse_header(str(hdr))
    hdr.write_text("/* int ub2_comment(void); */\nint ub2_ok(const long long* p, long long n, double d);\n")
    assert _C._parse_header(str(hdr)) == {"ub2_ok": [("p", ctypes.c_void_p), ("n", ctypes.c_longlong), ("d", ctypes.c_double)]}
    with pytest.raises(RuntimeError, match="missing.h"):
        _C._parse_header(str(tmp_path / "missing.h"))


def test_only_kernels_py_launches():
    """Every launch goes through a wrapper of unet/kernels.py: no other module of the package calls _C.call."""
    import ast
    pkg = os.path.join(ROOT, "unet-segment-pytorch_b200", "unet")
    callers = set()
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                path = os.path.join(dirpath, f)
                with open(path) as fh:
                    tree = ast.parse(fh.read(), path)
                for node in ast.walk(tree):
                    if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "call"
                            and isinstance(node.func.value, ast.Name) and node.func.value.id == "_C"):
                        callers.add(os.path.relpath(path, pkg))
    assert callers == {"kernels.py"}


def test_state_dict_layout_and_default_init_match_reference():
    from unet.models import AttentionUNet, UNet
    for attention, kw in ((True, {}), (False, {}), (True, {"deep_supervision": True}), (True, {"bilinear": False})):
        cls = AttentionUNet if attention else UNet
        m = cls(1, 2, base_features=16, **kw)
        shapes = O.state_dict_shapes(base_features=16, attention=attention, **kw)
        sd = m.state_dict()
        assert list(sd.keys()) == list(shapes.keys())
        assert all(tuple(sd[k].shape) == tuple(shapes[k]) for k in shapes)
    # same seed -> bit-identical default initialisation as the reference constructor
    fp = torch.load(os.path.join(GOLD, "init_fingerprint.pt"), weights_only=False)
    torch.manual_seed(42)
    m = AttentionUNet(1, 2, True, 16)
    for k, v in m.state_dict().items():
        s, head = fp[k]
        assert v.double().sum().item() == s and torch.equal(v.flatten()[:4], head), k
    assert m.get_num_params() == sum(p.numel() for p in m.parameters())
    assert AttentionUNet().get_num_params() == 17_612_458


def test_modules_survive_deepcopy_and_refuse_cpu_compute():
    from unet.models import AttentionUNet
    from unet.utils.loss import DiceBCELoss
    from unet.utils.metrics import SegmentationMetrics
    m = AttentionUNet(1, 2, True, 16)
    c = copy.deepcopy(m)
    c.load_state_dict(m.state_dict(), strict=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 1, 32, 32))
    with pytest.raises(RuntimeError, match="CUDA"):
        DiceBCELoss()(torch.zeros(1, 2, 8, 8), torch.zeros(1, 8, 8, dtype=torch.long))
    with pytest.raises(RuntimeError, match="CUDA"):
        SegmentationMetrics(2).update(torch.zeros(1, 2, 8, 8), torch.zeros(1, 8, 8, dtype=torch.long))


def test_loss_combination_from_statistics():
    """The O(N*C) part of the losses (host side of the ABI) against the oracle, with the pixel
    statistics computed by plain torch here."""
    from unet.utils import loss as L
    g = torch.load(os.path.join(GOLD, "loss.pt"), weights_only=False)
    z, t = g["z"], g["t"]
    p = torch.softmax(z, 1)
    y = torch.nn.functional.one_hot(t, 2).permute(0, 3, 1, 2).float()
    cnt = y.sum((2, 3))
    ce = (-torch.log_softmax(z, 1) * y).sum((2, 3))
    inter, psum = (p * y).sum((2, 3)), p.sum((2, 3))
    dice = L._dice_from_stats(cnt, inter, psum, 1.0, 'mean', True)
    bce = L._balanced_ce_from_stats(cnt, ce, 0.3, 1e-6)
    assert abs(dice.item() - g["dice"]["value"]) < 1e-5
    assert abs(bce.item() - g["balanced_ce"]["value"]) < 1e-5


def test_metrics_host_side():
    from unet.utils.metrics import SegmentationMetrics
    for g in torch.load(os.path.join(GOLD, "metrics.pt"), weights_only=False):
        m = SegmentationMetrics(g["c"], ignore_index=g["ignore"])
        assert m.compute()["mean_iou"] == 0.0
        m.confusion_matrix = g["cm"].numpy()
        res = m.compute()
        for k, v in g["result"].items():
            assert res[k] == v
        assert m.get_confusion_matrix().dtype == np.int64
        m.reset()
        assert m.confusion_matrix.sum() == 0


def test_input_pipeline_host_side():
    """Flip bits are reproducible from the seed, and the device pipeline refuses a CPU device."""
    from unet.data import DeviceBatchPipeline
    from unet.data.device import draw_flags, prepare_batch
    a = draw_flags(64, torch.Generator().manual_seed(5), 0.5, 0.3)
    b = draw_flags(64, torch.Generator().manual_seed(5), 0.5, 0.3)
    assert a.dtype == torch.uint8 and torch.equal(a, b) and int(a.max()) <= 3
    assert 10 < int((a & 1).sum()) < 54 and 3 < int((a >> 1).sum()) < 40
    assert int(draw_flags(16, torch.Generator().manual_seed(1), 0.0, 0.0).sum()) == 0
    assert int(draw_flags(16, torch.Generator().manual_seed(1), 1.0, 1.0).min()) == 3
    with pytest.raises(RuntimeError, match="CUDA"):
        DeviceBatchPipeline([], "cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        prepare_batch(torch.zeros(1, 16, 16, dtype=torch.uint8))


def test_host_side_argument_checks():
    """Constructor-level behaviour that needs no GPU: bad arguments raise, CPU models are refused
    by the engines that only exist for the CUDA path."""
    import torch.nn as nn
    from unet.inference import InferenceEngine
    from unet.models import AttentionUNet
    from unet.parallel import BatchShardedTrainer
    lin = nn.Linear(2, 2)
    with pytest.raises(ValueError, match="accumulation_steps"):
        BatchShardedTrainer(lin, nn.MSELoss(), torch.optim.SGD(lin.parameters(), lr=0.1), accumulation_steps=0)
    tr = BatchShardedTrainer(lin, nn.MSELoss(), torch.optim.SGD(lin.parameters(), lr=0.1), accumulation_steps=2)
    assert tr.accumulation_steps == 2 and tr.world == 1 and len(tr.buckets) == 1
    # gradients live in one flat bucket, every view on a 128-byte boundary
    assert all(p.grad is not None and p.grad.data_ptr() % 128 == tr.buckets[0].flat.data_ptr() % 128
               for p in lin.parameters())
    engine = InferenceEngine(AttentionUNet(1, 2, True, 16))      # building on the CPU is allowed (train.py:306)
    with pytest.raises(RuntimeError, match="CUDA"):
        engine(torch.zeros(1, 1, 32, 32))
    with pytest.raises(RuntimeError, match="CUDA"):
        engine.predict(torch.zeros(1, 32, 32, dtype=torch.uint8))


def test_workspace_queries_and_argument_errors_on_the_host():
    """The *_rows / *_blocks queries are pure host arithmetic (no device needed): positive counts for
    valid shapes, UB2_ERR_SHAPE (-1) for degenerate or unsupported ones, and entry points reject NULL /
    unsupported arguments before touching the device."""
    from unet import _C
    lib = _C.lib()
    assert lib.ub2_adamw_chunk_elems() == 16384
    good = (4, 512, 512, 64)
    queries = [lib.ub2_outc_rows, lib.ub2_conv_in_rows, lib.ub2_gate_rows, lib.ub2_gate_strip_rows,
               lambda n, h, w, c: lib.ub2_bn_bwd_rows(n, h, w, c, 0), lambda n, h, w, c: lib.ub2_bn_bwd_rows(n, h, w, c, 1)]
    for q in queries:
        assert 0 < q(*good) <= 148 * 16
        for bad in ((0, 512, 512, 64), (4, 0, 512, 64), (4, 512, 0, 64), (-1, 8, 8, 8), (4, 512, 512, 60), (4, 512, 512, 0)):
            assert q(*bad) == -1, bad
    assert lib.ub2_seg_stats_blocks(4, 512 * 512) > 0
    assert lib.ub2_seg_stats_blocks(0, 512 * 512) == -1 and lib.ub2_seg_stats_blocks(2, 0) == -1
    assert lib.ub2_prepare_batch(None, None, None, 1, 8, 8, 0.5, 0.5, None, None, None) == -1
    assert lib.ub2_predict_mask(None, 1, 2, 64, 0.5, None, None, None) == -1
    assert lib.ub2_resize_planes_fwd(None, None, 0, 1, 1, 1, 1, None) == -1
    assert lib.ub2_resize_planes_bwd(None, None, 2, 0, 1, 1, 1, None) == -1


def test_convolution_kernels_are_tcgen05_tma_code():
    """The built library's convolution kernels contain the SASS that tcgen05.mma / tcgen05.ld / TMA compile
    to on sm_100a (UTCHMMA, LDTM, UTMALDG: /opt/skills/guides/B200_PROFILING.md), and no legacy HMMA:
    the tensor-core path is the Blackwell one, not a recompiled mma.sync kernel."""
    import shutil
    import subprocess
    from unet import _C
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([tool, "-sass", _C.LIB_PATH], capture_output=True, text=True).stdout
    per_kernel, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            per_kernel[name] = set()
            continue
        if name:
            for op in ("UTCHMMA", "LDTM", "UTMALDG", "UTCBAR"):
                if op in line:
                    per_kernel[name].add(op)
            if re.search(r"(?<![A-Z])HMMA", line):     # mma.sync / wmma
                per_kernel[name].add("legacy HMMA")
    conv = {k: v for k, v in per_kernel.items() if re.search(r"conv_(fwd|fwd2|halo|halo2|wgrad|wgrad2|wgrad_halo|wgrad_halo2)_kernel", k)}
    assert len(conv) >= 12
    for k, ops in conv.items():
        assert {"UTCHMMA", "LDTM", "UTMALDG", "UTCBAR"} <= ops, (k, ops)
    assert not any("legacy HMMA" in ops for ops in per_kernel.values())


def test_side_stream_fork_join_bookkeeping(monkeypatch):
    """ops.SideStream on fake streams (no GPU here): the side stream waits for the main stream before each fork, the
    main stream joins the previous fork before the next one, and the tensors a fork reads stay referenced until
    that join — the caching allocator recycles a freed block in main-stream order only."""
    import weakref
    from unet import ops
    log = []

    class FakeStream:
        def __init__(self, name="side", device=None):
            self.name, self.device = name, device

        def wait_stream(self, other):
            log.append((self.name, "waits", other.name))

    class FakeCtx:
        def __init__(self, s):
            self.s = s

        def __enter__(self):
            log.append(("enter", self.s.name))

        def __exit__(self, *a):
            log.append(("exit", self.s.name))

    main = FakeStream("main")
    monkeypatch.setattr(torch.cuda, "Stream", lambda device=None: FakeStream("side", device))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: main)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: FakeCtx(s))

    class Blob:   # stands for a tensor (weak-referenceable)
        pass

    side = ops.SideStream("cuda:0")
    a, dy = Blob(), Blob()
    ra, rdy = weakref.ref(a), weakref.ref(dy)
    out = side.run(lambda: log.append("wgrad-1") or "partials-1", a, dy)
    assert out == "partials-1"
    assert log == [("side", "waits", "main"), ("enter", "side"), "wgrad-1", ("exit", "side")]
    del a, dy
    assert ra() is not None and rdy() is not None          # still referenced: the side stream may be reading them
    del log[:]
    side.run(lambda: log.append("wgrad-2"), Blob())
    # the main stream joined fork 1 BEFORE fork 2 was queued, and fork 1's operands were released at that join
    assert log[0] == ("main", "waits", "side") and log[1] == ("side", "waits", "main") and "wgrad-2" in log
    assert ra() is None and rdy() is None
    del log[:]
    side.join()
    side.join()                                             # idempotent: nothing outstanding after the first
    assert log == [("main", "waits", "side")]
    # module-level join is a no-op without an installed side stream
    assert ops.WGRAD_SIDE is None
    ops.wgrad_join()
