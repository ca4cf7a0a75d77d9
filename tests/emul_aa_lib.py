"""Test-side loader of tests/host_emul/libhostemul_aa.so: the refine rule of adaptive supersampling and the accumulator
slots it reads (ntracer_b200/csrc/trace_core.cuh: refine_pixel, halo_pixel, corner_slot), compiled for the host.
Test infrastructure only; the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_aa.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_aa.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, 'emul_aa.cpp')] + [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_aa.so'))
        _lib = C.CDLL(path)
        _lib.emul_refine_mask.restype = C.c_longlong
        _lib.emul_refine_mask.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_float, C.c_void_p]
    return _lib


def refine_mask(view_rgb, t, window=None, trf=0, trs=1, compact=False):
    """The device's refine mask of one launch over the plain frame `view_rgb` (h, w, 3) of the whole view: window =
    (x0, y0, win_w, win_h) (default: the view), tile rows trf, trf + trs, ... of it -> (mask (win_h, win_w) uint8 with
    the rows the launch does not own left 0, halo pixels traced)."""
    rgb = np.ascontiguousarray(view_rgb, dtype=np.float32)
    vh, vw = rgb.shape[:2]
    x0, y0, ww, wh = window or (0, 0, vw, vh)
    mask = np.zeros((wh, ww), np.uint8)
    n = lib().emul_refine_mask(rgb.ctypes.data, vw, vh, x0, y0, ww, wh, trf, trs, int(compact), float(t), mask.ctypes.data)
    return mask, int(n)
