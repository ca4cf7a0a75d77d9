"""Test-side loader of tests/host_emul/libhostemul_ss.so: the host-emulated frame driver (tests/host_emul/emul.cpp) with
a supersampling factor, running the product's ss_pixel_color (ntracer_b200/csrc/trace_core.cuh) for the primary pass.
Test infrastructure only; the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_ss.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_ss.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, f) for f in ('emul_ss.cpp', 'emul.cpp')] + \
               [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h', 'arena_pack.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_ss.so'))
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def render_ss(sc, w, h, ss, cam=None, generic=False):
    """A w x h frame supersampled with factor ss (ntr_scene_set_supersampling) -> (rgb, counters)."""
    d, keep = _capi.make_desc(sc)
    if cam is None:
        cam = (sc['cam_origin'], sc['cam_axes'])
    o = np.ascontiguousarray(cam[0], dtype=np.float32)
    a = np.ascontiguousarray(cam[1], dtype=np.float32)
    rgb = np.zeros((h, w, 3), dtype=np.float32)
    cnt = np.zeros(9, dtype=np.uint64)
    if lib().emul_render_ss(C.byref(d), _p(o), _p(a), w, h, int(ss), int(generic), _p(rgb), _p(cnt)) != 0:
        raise ValueError('supersampling factor out of range')
    names = [n for n, _ in _capi.Counters._fields_]
    return rgb, {n: int(v) for n, v in zip(names, cnt)}
