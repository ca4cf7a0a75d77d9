"""Test-side loader of tests/host_emul/libhostemul_aov.so: the AOV capture of the NTR_F_VIEWS | NTR_F_AOV kernels (the
product's ss_pixel_color with a PrimaryAov) on the host (tests/host_emul/emul_aov.cpp).  Test infrastructure only; the product
never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_aov.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None
COUNTERS = ('reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests', 'solid_tests', 'shaded_hits', 'truncated_hit_lists')


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_aov.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, f) for f in ('emul_aov.cpp', 'emul.cpp')] + \
               [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h', 'arena_pack.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_aov.so'))
        _lib = C.CDLL(path)
        _lib.emul_aov_sample0_mismatches.restype = C.c_longlong
        _lib.emul_aov_sample0_mismatches.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_int]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cam(sc, cam):
    if cam is None:
        cam = (sc['cam_origin'], sc['cam_axes'])
    return np.ascontiguousarray(cam[0], dtype=np.float32), np.ascontiguousarray(cam[1], dtype=np.float32)


def aov_pass(sc, w, h, ss=1, cam=None, generic=False):
    """A w x h view at factor ss through ss_pixel_color as the views kernels run it, without and with the AOV capture ->
    dict(ids, depth: (h, w), normals, dirs: (h, w, dim) -- dirs: every pixel's plain primary ray --, plain, aov: (h, w, 3)
    float32 colours, plain_counters, aov_counters, plain_records, aov_records, same_records)."""
    d, keep = _capi.make_desc(sc)
    o, a = _cam(sc, cam)
    dim = int(sc['dim'])
    ids = np.zeros((h, w), np.int32)
    depth = np.zeros((h, w), np.float32)
    normals = np.zeros((h, w, dim), np.float32)
    dirs = np.zeros((h, w, dim), np.float32)
    plain = np.zeros((h, w, 3), np.float32)
    aov = np.zeros((h, w, 3), np.float32)
    cnt = np.zeros(14, np.uint64)
    rec = np.zeros(3, np.uint64)
    lib().emul_aov_pass(C.byref(d), _p(o), _p(a), w, h, ss, int(generic), _p(ids), _p(depth), _p(normals), _p(dirs),
                        _p(plain), _p(aov), _p(cnt), _p(rec))
    return dict(ids=ids, depth=depth, normals=normals, dirs=dirs, plain=plain, aov=aov,
                plain_counters=dict(zip(COUNTERS, map(int, cnt[:7]))), aov_counters=dict(zip(COUNTERS, map(int, cnt[7:]))),
                plain_records=int(rec[0]), aov_records=int(rec[1]), same_records=bool(rec[2]))


def sample0_mismatches(dim, cam, fov, w, h, ss):
    """pixels of a w x h view whose sample (0, 0) at factor ss is not their plain primary ray bit for bit"""
    o = np.ascontiguousarray(cam[0], dtype=np.float32)
    a = np.ascontiguousarray(cam[1], dtype=np.float32)
    return int(lib().emul_aov_sample0_mismatches(dim, _p(o), _p(a), fov, w, h, ss))
