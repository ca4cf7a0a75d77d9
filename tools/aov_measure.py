"""Per-pixel AOVs of a views call against what a caller can do without them (DESIGN section 10).

For c2, c4b and c4 at 1920x1080 and 640x480 (s = 1, and s = 2 on c4b) it renders the first 32 cameras of the 160-step
rotation of `polytope.py --benchmark` (stream.rotation_cameras) three ways, alternating them rep after rep:
  (a) DeviceScene.render_views (frames only);
  (b) DeviceScene.render_views_aovs with ids, depth and normals in the same launches;
  (c) render_views plus a primary_hit_ids loop over the views (ids and depth only: no normals without AOVs).
Each into pinned host buffers (wall clock around the calls) and, for (a) and (b), into device tensors (CUDA events of the
call, the first launch to the last).  It checks that the frames of (a) and (b) agree and that the ids and depth of (b) are
those of (c).  The GPU's name and power limit are read in the same run.

    python tools/aov_measure.py [--out profiles/aov_measure.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.views_measure import gpu_info, scene, spread  # noqa: E402

SIZES = ((1920, 1080), (640, 480))
POINTS = [(c, w, h, 1) for c in ('c2', 'c4b', 'c4') for w, h in SIZES] + [('c4b', w, h, 2) for w, h in SIZES]


def measure_point(config, w, h, ss, n, reps):
    import torch
    from ntracer_b200 import _capi, stream
    from ntracer_b200.backend import DeviceScene, aov_struct
    sc = scene(config)
    dim = int(sc['dim'])
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    fb, npix = fmt.pitch * h, w * h
    cams = stream.rotation_cameras(sc['cam_origin'], sc['cam_axes'], 160)[:n]
    out = {'config': config, 'width': w, 'height': h, 'ss': ss, 'views': n,
           'aov_bytes_per_launch_view': npix * (8 + 4 * dim)}
    pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory()
    with DeviceScene(sc) as ds:
        ds.set_supersampling(ss)
        frames_a, frames_b = pin(n * fb, torch.uint8), pin(n * fb, torch.uint8)
        host = {'ids': pin((n, h, w), torch.int32), 'depth': pin((n, h, w), torch.float32),
                'normals': pin((n, h, w, dim), torch.float32)}
        ids_c, depth_c = np.zeros((n, h, w), np.int32), np.zeros((n, h, w), np.float32)
        dev = torch.zeros(n * fb, dtype=torch.uint8, device='cuda')
        dev_aov = {k: torch.zeros(v.shape, dtype=v.dtype, device='cuda') for k, v in host.items()}
        st = torch.cuda.current_stream().cuda_stream
        o = np.ascontiguousarray(np.stack([c[0] for c in cams]), np.float32)
        ax = np.ascontiguousarray(np.stack([c[1] for c in cams]), np.float32)
        import ctypes as C
        a_host = aov_struct({k: (t.data_ptr(), t.numel()) for k, t in host.items()})

        def run_a():
            t0 = time.perf_counter()
            ds.render_views(fmt, cams, frames_a.numpy())
            return time.perf_counter() - t0

        def run_b():
            t0 = time.perf_counter()
            _capi.check(ds._lib.ntr_render_views_aovs(ds._h, n, o.ctypes.data, ax.ctypes.data, C.byref(fmt), frames_b.data_ptr(),
                                                      frames_b.numel(), C.byref(a_host)))
            return time.perf_counter() - t0

        def run_c():
            t0 = time.perf_counter()
            ds.render_views(fmt, cams, frames_a.numpy())
            for k, (co, ca) in enumerate(cams):
                ds.set_camera(co, ca)
                i, d = ds.primary_hit_ids(w, h)
                ids_c[k], depth_c[k] = i, d
            return time.perf_counter() - t0

        def dev_a():
            ds.render_views_device(fmt, cams, dev.data_ptr(), dev.numel(), st)
            torch.cuda.synchronize()
            return ds.last_kernel_ms()

        def dev_b():
            ds.render_views_aovs_device(fmt, cams, dev.data_ptr(), dev.numel(), dev_aov, st)
            torch.cuda.synchronize()
            return ds.last_kernel_ms()

        runs = (run_a, run_b, run_c, dev_a, dev_b)
        for f in runs:
            f()                                     # warm-up: modules, queues, schedules, sort sizes
        res = {f.__name__: [] for f in runs}
        for _ in range(reps):
            for f in runs:
                res[f.__name__].append(f())
        out['a_render_views_host_fps'] = spread([n / t for t in res['run_a']])
        out['b_render_views_aovs_host_fps'] = spread([n / t for t in res['run_b']])
        out['c_render_views_plus_hit_ids_host_fps'] = spread([n / t for t in res['run_c']])
        out['a_render_views_device_kernel_ms_per_frame'] = spread([ms / n for ms in res['dev_a']])
        out['b_render_views_aovs_device_kernel_ms_per_frame'] = spread([ms / n for ms in res['dev_b']])
        ds.render_views(fmt, cams, frames_a.numpy())
        out['max_abs_diff_frames_a_b'] = int(np.abs(frames_a.numpy().astype(np.int16) - frames_b.numpy().astype(np.int16)).max())
        out['ids_equal_b_c'] = bool(np.array_equal(host['ids'].numpy(), ids_c))
        out['depth_equal_b_c'] = bool(np.array_equal(host['depth'].numpy().view(np.uint32), depth_c.view(np.uint32)))
        out['device_aovs_equal_host'] = all(bool(np.array_equal(dev_aov[k].cpu().numpy(), host[k].numpy())) for k in host)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'aov_measure.json'))
    ap.add_argument('--views', type=int, default=32)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    res = {'gpu': gpu_info(), 'views': args.views, 'reps': args.reps,
           'note': 'frames/s: wall clock around the whole call into pinned host buffers, median over the reps; kernel ms: '
                   'CUDA events from the first launch to the last of the call, per frame, device destinations'}
    res['points'] = [measure_point(c, w, h, ss, args.views, args.reps) for c, w, h, ss in POINTS]
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
