"""Test-side loader of tests/host_emul/libhostemul_rays.so: the primary pass of a batch of caller-given rays (the product's
given_ray_color as render_rays_kernel runs it) on the host, next to the plain primary pass and as a whole rays call
(tests/host_emul/emul_rays.cpp).  Test infrastructure only; the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_rays.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None
COUNTERS = ('reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests', 'solid_tests', 'shaded_hits', 'truncated_hit_lists')


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_rays.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, f) for f in ('emul_rays.cpp', 'emul.cpp')] + \
               [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h', 'arena_pack.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_rays.so'))
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def vs_plain(sc, w, h, cam=None, generic=False):
    """A w x h frame's primary pass through the plain path and through the ray-fed pass with the camera's own rays ->
    dict(plain, rays: (h, w, 3) float32, origins, dirs: (h * w, D) the rays, plain_counters, rays_counters,
    plain_records, rays_records, same_records)."""
    d, keep = _capi.make_desc(sc)
    if cam is None:
        cam = (sc['cam_origin'], sc['cam_axes'])
    o = np.ascontiguousarray(cam[0], dtype=np.float32)
    a = np.ascontiguousarray(cam[1], dtype=np.float32)
    D = int(sc['dim'])
    plain = np.zeros((h, w, 3), np.float32)
    rays = np.zeros((h, w, 3), np.float32)
    rr = np.zeros((h * w, 2, D), np.float32)
    cnt = np.zeros(14, np.uint64)
    rec = np.zeros(3, np.uint64)
    lib().emul_rays_vs_plain(C.byref(d), _p(o), _p(a), w, h, int(generic), _p(plain), _p(rays), _p(rr), _p(cnt), _p(rec))
    return dict(plain=plain, rays=rays, origins=rr[:, 0].copy(), dirs=rr[:, 1].copy(),
                plain_counters=dict(zip(COUNTERS, map(int, cnt[:7]))), rays_counters=dict(zip(COUNTERS, map(int, cnt[7:]))),
                plain_records=int(rec[0]), rays_records=int(rec[1]), same_records=bool(rec[2]))


def render_rays(sc, origins, dirs, generic=False):
    """A whole rays call on the host -> dict(rgb (n, 3), ids, depth (n,), normals (n, D), counters)"""
    d, keep = _capi.make_desc(sc)
    o = np.ascontiguousarray(origins, dtype=np.float32)
    di = np.ascontiguousarray(dirs, dtype=np.float32)
    n, D = o.shape[0], int(sc['dim'])
    rgb = np.zeros((n, 3), np.float32)
    ids = np.zeros(n, np.int32)
    depth = np.zeros(n, np.float32)
    normals = np.zeros((n, D), np.float32)
    cnt = np.zeros(7, np.uint64)
    lib().emul_render_rays(C.byref(d), C.c_uint32(n), _p(o), _p(di), int(generic), _p(rgb), _p(ids), _p(depth), _p(normals),
                           _p(cnt))
    return dict(rgb=rgb, ids=ids, depth=depth, normals=normals, counters=dict(zip(COUNTERS, map(int, cnt))))
