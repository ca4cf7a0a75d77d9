"""Test-side loader of tests/host_emul/libhostemul_views.so: the primary pass of a batch of views at factor 1 (the product's
ss_pixel_color as the NTR_F_VIEWS kernels run it) next to the plain primary pass, on the host (tests/host_emul/emul.cpp).
Test infrastructure only; the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_views.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None
COUNTERS = ('reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests', 'solid_tests', 'shaded_hits', 'truncated_hit_lists')


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_views.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, f) for f in ('emul_views.cpp', 'emul.cpp')] + \
               [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h', 'arena_pack.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_views.so'))
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def factor1(sc, w, h, cam=None, generic=False, exact=True):
    """A w x h frame at factor 1 through the plain primary path and through ss_pixel_color (exact=True: as the NTR_F_VIEWS
    kernels run it; False: as the NTR_F_SS kernels do) -> dict(plain, views: (h, w, 3) float32, plain_counters,
    views_counters, plain_records, views_records, same_records)."""
    d, keep = _capi.make_desc(sc)
    if cam is None:
        cam = (sc['cam_origin'], sc['cam_axes'])
    o = np.ascontiguousarray(cam[0], dtype=np.float32)
    a = np.ascontiguousarray(cam[1], dtype=np.float32)
    plain = np.zeros((h, w, 3), np.float32)
    views = np.zeros((h, w, 3), np.float32)
    cnt = np.zeros(14, np.uint64)
    rec = np.zeros(3, np.uint64)
    lib().emul_views_factor1(C.byref(d), _p(o), _p(a), w, h, int(generic), int(exact), _p(plain), _p(views), _p(cnt), _p(rec))
    return dict(plain=plain, views=views, plain_counters=dict(zip(COUNTERS, map(int, cnt[:7]))),
                views_counters=dict(zip(COUNTERS, map(int, cnt[7:]))), plain_records=int(rec[0]), views_records=int(rec[1]),
                same_records=bool(rec[2]))
