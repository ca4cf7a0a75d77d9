"""Test-side loader of tests/host_emul/libhostemul_proj.so: projected frames (ntr_scene_set_projection) on the host -- the
product's ray generator, the primary pass of the NTR_F_PROJ builds and the refine rule between the rounds of an adaptive
frame (tests/host_emul/emul_proj.cpp).  Test infrastructure only; the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi
from ntracer_b200.backend import PROJECTIONS

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'libhostemul_proj.so')
_CSRC = os.path.join(os.path.dirname(_DIR), '..', 'ntracer_b200', 'csrc')
_lib = None
COUNTERS = ('reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests', 'solid_tests', 'shaded_hits', 'truncated_hit_lists')


def build(out=_SO):
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    subprocess.run([gxx, '-std=c++17', '-O2', '-fPIC', '-shared', '-fvisibility=hidden',
                    '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-o', out,
                    os.path.join(_DIR, 'emul_proj.cpp')], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, f) for f in ('emul_proj.cpp', 'emul.cpp')] + \
               [os.path.join(_CSRC, f) for f in ('trace_core.cuh', 'device_types.h', 'arena_pack.h')]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'libhostemul_proj.so'))
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cam(sc, cam):
    if cam is None:
        cam = (sc['cam_origin'], sc['cam_axes'])
    return np.ascontiguousarray(cam[0], dtype=np.float32), np.ascontiguousarray(cam[1], dtype=np.float32)


def camera_rays(sc, w, h, kind, param, cam=None, generic=False):
    """The w x h view's rays under projection (kind, param) -> (origins, dirs) float32 (w * h, D), ray y * w + x = pixel (x, y)"""
    d, keep = _capi.make_desc(sc)
    o, a = _cam(sc, cam)
    D = int(sc['dim'])
    ro = np.zeros((w * h, D), np.float32)
    rd = np.zeros((w * h, D), np.float32)
    lib().emul_camera_rays(C.byref(d), _p(o), _p(a), w, h, PROJECTIONS.index(kind), C.c_float(param or 0.0), int(generic),
                           _p(ro), _p(rd))
    return ro, rd


def render(sc, w, h, kind, param, ss=1, threshold=None, cam=None, generic=False):
    """A projected w x h frame at factor ss (adaptive with a threshold) -> dict(rgb (h, w, 3) float32, mask (h, w) uint8 (zeros
    when not adaptive), primary_rays, counters)"""
    d, keep = _capi.make_desc(sc)
    o, a = _cam(sc, cam)
    rgb = np.zeros((h, w, 3), np.float32)
    mask = np.zeros((h, w), np.uint8)
    cnt = np.zeros(8, np.uint64)
    rc = lib().emul_render_proj(C.byref(d), _p(o), _p(a), w, h, ss, C.c_float(-1.0 if threshold is None else threshold),
                                PROJECTIONS.index(kind), C.c_float(param or 0.0), int(generic), _p(rgb), _p(mask), _p(cnt))
    assert rc == 0
    return dict(rgb=rgb, mask=mask, primary_rays=int(cnt[0]), counters=dict(zip(COUNTERS, map(int, cnt[1:]))))


def vs_rays(sc, w, h, kind, param, cam=None, generic=False):
    """The projected factor-1 pass and the ray-fed pass over its own camera rays -> dict(frame, rays: (h, w, 3) float32,
    origins, dirs, frame_counters, rays_counters, frame_records, rays_records, same_records)"""
    d, keep = _capi.make_desc(sc)
    o, a = _cam(sc, cam)
    D = int(sc['dim'])
    frame = np.zeros((h, w, 3), np.float32)
    rays = np.zeros((h, w, 3), np.float32)
    ro = np.zeros((w * h, D), np.float32)
    rd = np.zeros((w * h, D), np.float32)
    cnt = np.zeros(14, np.uint64)
    rec = np.zeros(3, np.uint64)
    lib().emul_proj_vs_rays(C.byref(d), _p(o), _p(a), w, h, PROJECTIONS.index(kind), C.c_float(param or 0.0), int(generic),
                            _p(frame), _p(rays), _p(ro), _p(rd), _p(cnt), _p(rec))
    return dict(frame=frame, rays=rays, origins=ro, dirs=rd,
                frame_counters=dict(zip(COUNTERS, map(int, cnt[:7]))), rays_counters=dict(zip(COUNTERS, map(int, cnt[7:]))),
                frame_records=int(rec[0]), rays_records=int(rec[1]), same_records=bool(rec[2]))
