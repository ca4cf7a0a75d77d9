#!/usr/bin/env python3
"""Cost of projected frames (Scene.set_projection, DESIGN section 12), on one GPU.

For c2 ({5,3,3}) and c4 ({5/2,3,3} with reflections and transparency) at 1920x1080 and 640x480:
  (a) an orthographic and an equirectangular frame (render_float) against render_rays_device of the same camera rays
      (DeviceScene.camera_rays_device): the native frame generates its rays, the ray-fed call reads 2 x D floats per ray;
  (b) the perspective frame of the same scene (report only);
  (c) views throughput: 32 orthographic views of the rotation (stream.rotation_cameras) into device memory.
Kernel time is ntr_last_kernel_ms (CUDA events around the call's launches).  Each point is the median of --reps calls after
--warmup calls, and the spread (max - min) of the kernel times is reported beside it.  The card's name and power limit are
read in the same run.  Writes one JSON document (stdout, or --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENES = {'c2': 'cell120', 'c4': 'ggs120:refl_transp'}


def timed(fn, ds, warmup, reps):
    for _ in range(warmup):
        fn()
    ms, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        ms.append(ds.last_kernel_ms())
    return {'kernel_ms': statistics.median(ms), 'kernel_spread_ms': max(ms) - min(ms), 'wall_ms': statistics.median(wall)}


def ortho_camera(sc):
    """the scene's camera axes, moved back along fwd so that the image plane lies outside the scene box; half width: the box"""
    lo, hi = np.asarray(sc['boundary'], np.float64)
    ax = np.asarray(sc['cam_axes'], np.float32)
    r = float(np.linalg.norm(hi - lo))
    return ((lo + hi) / 2 - ax[2] * r).astype(np.float32), ax, float(np.max(hi - lo)) * 0.6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from ntracer_b200 import _capi, stream
    from ntracer_b200.backend import DeviceScene
    from tests import fixtures as fx
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    out = {'gpu': q[0] if q else 'unknown', 'reps': args.reps, 'warmup': args.warmup, 'points': [], 'views': []}
    for cfg, fixture in SCENES.items():
        name, _, var = fixture.partition(':')
        sc, g = fx.load(name)
        if var:
            sc = fx.variant(sc, g, var)
        oc, ax, half = ortho_camera(sc)
        with DeviceScene(sc) as ds:
            for w, h in ((1920, 1080), (640, 480)):
                n = w * h
                point = {'config': cfg, 'width': w, 'height': h}
                ds.set_camera(sc['cam_origin'], sc['cam_axes'])
                ds.set_projection('perspective')
                point['b_perspective_frame'] = timed(lambda: ds.render_float(w, h), ds, args.warmup, args.reps)
                for kind, param, cam in (('orthographic', half, (oc, ax)),
                                         ('equirectangular', 2 * np.pi, (sc['cam_origin'], sc['cam_axes']))):
                    ds.set_camera(*cam)
                    ds.set_projection(kind, param)
                    frame = timed(lambda: ds.render_float(w, h), ds, args.warmup, args.reps)
                    to = torch.empty((n, ds.dim), device='cuda')
                    td = torch.empty((n, ds.dim), device='cuda')
                    ds.camera_rays_device(w, h, to, td)
                    rgb = torch.empty((n, 3), device='cuda')

                    def call():
                        ds.render_rays_device(to, td, rgb)
                        torch.cuda.synchronize()
                    rays = timed(call, ds, args.warmup, args.reps)
                    img = ds.render_float(w, h).reshape(-1, 3)
                    point['a_' + kind] = {'frame': frame, 'render_rays_device': rays,
                                          'frame_over_rays': frame['kernel_ms'] / rays['kernel_ms'],
                                          'max_abs_diff_frame_vs_rays': float(np.abs(rgb.cpu().numpy() - img).max())}
                print(json.dumps(point), flush=True)
                out['points'].append(point)
            # (c) 32 orthographic views of the rotation, every one moved back along its fwd axis, into device memory
            lo, hi = np.asarray(sc['boundary'], np.float64)
            r = float(np.linalg.norm(hi - lo))
            cams = [((lo + hi) / 2 - np.asarray(a, np.float64)[2] * r, np.asarray(a, np.float32))
                    for _, a in stream.rotation_cameras(sc['cam_origin'], sc['cam_axes'], 160)[:32]]
            cams = [(o.astype(np.float32), a) for o, a in cams]
            ds.set_projection('orthographic', half)
            for w, h in ((1920, 1080), (640, 480)):
                fmt = _capi.make_image_format(w, h, _capi.RGB8)
                dst = torch.empty(len(cams) * fmt.pitch * h, dtype=torch.uint8, device='cuda')

                def views():
                    ds.render_views_device(fmt, cams, dst.data_ptr(), dst.numel())
                    torch.cuda.synchronize()
                t = timed(views, ds, 1, 3)
                v = {'config': cfg, 'width': w, 'height': h, 'views': len(cams), 'call': t,
                     'views_per_s': len(cams) / (t['wall_ms'] / 1e3)}
                print(json.dumps(v), flush=True)
                out['views'].append(v)
    text = json.dumps(out, indent=1)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    else:
        print(text)


if __name__ == '__main__':
    main()
