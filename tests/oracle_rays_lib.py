"""Test-side loader of tests/host_emul/liboracle_rays.so: the oracle (oracle/ntr_oracle.c, the C restatement of the
reference) for a batch of caller-given primary rays, built from tests/host_emul/oracle_rays.c.  Test infrastructure only;
the product never loads it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from ntracer_b200 import _capi

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_emul')
_SO = os.path.join(_DIR, 'liboracle_rays.so')
_ORACLE = os.path.join(os.path.dirname(_DIR), '..', 'oracle', 'ntr_oracle.c')
_lib = None


def build(out=_SO):
    cc = '/usr/bin/gcc' if os.path.exists('/usr/bin/gcc') else 'gcc'
    cmd = [cc, '-O2', '-std=c11', '-fPIC', '-fvisibility=hidden', '-shared', '-o', out, os.path.join(_DIR, 'oracle_rays.c'), '-lm']
    # as oracle/Makefile: OpenMP where the compiler has it, serial otherwise
    if subprocess.run(cmd[:1] + ['-fopenmp'] + cmd[1:], capture_output=True).returncode != 0:
        subprocess.run(cmd[:1] + ['-Wno-unknown-pragmas'] + cmd[1:], check=True)
    return out


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_DIR, 'oracle_rays.c'), _ORACLE]
        path = _SO
        if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
            # a tree that cannot be written to (a read-only checkout) gets the library in a temporary directory
            path = build() if os.access(_DIR, os.W_OK) else build(os.path.join(tempfile.mkdtemp(), 'liboracle_rays.so'))
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def ray_colors(sc, origins, dirs):
    """The colour of caller-given primary rays as the reference computes it (ray_color at depth 0 with no source, or the
    BoxScene's colour) and their opaque hits -> dict(rgb (n, 3), ids, dist, t0 (aabb_distance; -1: the ray misses the scene
    box), undefined (per ray, as oracle_lib.render_float's mask), counters)."""
    d, keep = _capi.make_desc(sc)
    origins = np.ascontiguousarray(origins, dtype=np.float32)
    dirs = np.ascontiguousarray(dirs, dtype=np.float32)
    n = origins.shape[0]
    rgb = np.zeros((n, 3), np.float32)
    ids = np.zeros(n, np.int32)
    dist = np.zeros(n, np.float32)
    t0 = np.zeros(n, np.float32)
    undefined = np.zeros(n, np.uint8)
    cnt = _capi.Counters()
    lib().oracle_ray_colors(C.byref(d), C.c_uint32(n), _p(origins), _p(dirs), _p(rgb), _p(ids), _p(dist), _p(t0),
                            _p(undefined), C.byref(cnt))
    return dict(rgb=rgb, ids=ids, dist=dist, t0=t0, undefined=undefined, counters=cnt.as_dict())
