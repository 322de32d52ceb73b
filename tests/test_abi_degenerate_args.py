"""CPU: no entry point of include/unetb200.h may crash on degenerate arguments.

Every prototype is called with NULL pointers and plausible sizes (8, 16, 64) where one integer
argument at a time is 0 or negative.  On a box without a GPU a call that passes its argument checks
fails later with a CUDA error code, which is fine; what must never happen is a host-side division by
zero or NULL dereference before the checks (the calls run in a child process so that a crash is
reported as a failure, with the offending call, instead of killing pytest)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import ctypes, sys
sys.path.insert(0, sys.argv[1] + "/unet-segment-pytorch_b200")
from unet import _C
lib = _C.lib()
FIXED = {ctypes.c_void_p: None, ctypes.c_float: 0.5, ctypes.c_double: 1.0}   # NULL pointers; integers vary
calls = 0
for name, args in _C.SIGNATURES.items():
    if not args or name == "ub2_set_conv_mode":
        continue
    fn = getattr(lib, name)
    ints = [i for i, (_, t) in enumerate(args) if t not in FIXED]
    for base in (8, 16, 64):
        for z in [None] + ints:
            for zv in (0, -3):
                vals = [base] * len(args)
                if z is not None: vals[z] = zv
                print(name, vals, flush=True)
                fn(*[FIXED.get(t, v) for (_, t), v in zip(args, vals)])
                calls += 1
                if z is None: break
print("CALLS", calls, flush=True)
'''


def test_no_entry_point_crashes_on_degenerate_arguments():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")      # argument checks only, also on a GPU box
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, env=env)
    lines = r.stdout.strip().splitlines()
    assert r.returncode == 0, f"crashed (rc {r.returncode}) in: {lines[-1] if lines else '?'}"
    m = re.match(r"CALLS (\d+)", lines[-1])
    assert m and int(m.group(1)) > 1000
