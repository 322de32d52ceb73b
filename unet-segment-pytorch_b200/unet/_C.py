"""ctypes binding of libunetb200.so (the C ABI declared in include/unetb200.h).

There is no CPU or eager-PyTorch fallback: if the library is missing, or a
tensor is not on a CUDA device, the ops raise.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG = os.path.dirname(_HERE)
# UB2_LIB: another build of the same library (same-box A/B runs of a kernel change, tools/ab_lib.sh)
LIB_PATH = os.environ.get("UB2_LIB") or os.path.join(_PKG, "lib", "libunetb200.so")

_lib = None
_lock = threading.Lock()

ERRORS = {
    -1: "unsupported shape",
    -2: "pointer/stride alignment",
    -3: "workspace too small",
    -4: "driver entry point / tensor-map encode failed",
    -5: "not an sm_100 device",
}


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; build it in-tree if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                import importlib.util

                spec = importlib.util.spec_from_file_location("_ub2_build", os.path.join(_PKG, "build.py"))
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                mod.build()
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"libunetb200.so not found at {LIB_PATH} and could not be built")
            _lib = ctypes.CDLL(LIB_PATH)
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f"{what}: {ERRORS.get(rc, 'error')} (code {rc})")
    raise RuntimeError(f"{what}: CUDA error {rc}")


# Device of the tensors of the call being assembled (per host thread: forward runs on the main thread,
# backward on autograd's).  Every wrapper builds its argument list with ptr(...) first and stream() last,
# so stream() hands out the current stream OF THAT DEVICE and call() launches with that device current —
# a model on cuda:1 works while cuda:0 is the process's current device (the reference's
# get_device('cuda:1') pattern).  Tensors of two devices in one call raise.
_tls = threading.local()


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return ctypes.c_void_p(0)
    if not t.is_cuda:
        raise RuntimeError("unet-b200 ops need CUDA tensors: there is no CPU fallback")
    idx = t.device.index
    prev = getattr(_tls, "device", None)
    if prev is None:
        _tls.device = idx
    elif prev != idx:
        _tls.device = None
        raise RuntimeError(f"unet-b200 op received tensors on cuda:{prev} and cuda:{idx}")
    return ctypes.c_void_p(t.data_ptr())


def stream() -> ctypes.c_void_p:
    idx = getattr(_tls, "device", None)
    return ctypes.c_void_p(torch.cuda.current_stream(idx).cuda_stream)


# kernels launched per entry point (default 1); used for the bench's `gpu_launches` claim
_KERNELS_PER_CALL = {"ub2_conv_in_wgrad": 2, "ub2_outc_bwd": 2, "ub2_seg_stats": 2, "ub2_wgrad_reduce_multi": 2,
                     "ub2_shuffle2x2_bwd": 2, "ub2_f32_shuffle2x2_bwd": 2}
LAUNCHES = 0


# When set to a list, call() appends (entry point, start event, end event, work) per launch; ``work`` is
# the wrapper's (algorithmic FLOPs, algorithmic bytes) claim for the call or None.  bench.py's per-kernel
# roofline table is built from it (eager pass only: a replayed graph has no host hooks).
PROFILE = None


def call(name: str, *args, work=None) -> None:
    global LAUNCHES
    fn = getattr(lib(), name)
    fn.restype = ctypes.c_int
    idx = getattr(_tls, "device", None)
    _tls.device = None
    prof = PROFILE
    if idx is not None and idx != torch.cuda.current_device():
        with torch.cuda.device(idx):
            rc = fn(*args)
    elif prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(idx))
        rc = fn(*args)
        e1.record(torch.cuda.current_stream(idx))
        prof.append((name, e0, e1, work))
    else:
        rc = fn(*args)
    check(rc, name)
    LAUNCHES += _KERNELS_PER_CALL.get(name, 1)


c_int = ctypes.c_int
c_float = ctypes.c_float
c_double = ctypes.c_double
c_longlong = ctypes.c_longlong
byref = ctypes.byref
