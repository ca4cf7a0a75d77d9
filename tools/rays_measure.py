#!/usr/bin/env python3
"""Cost of shading caller-given rays (DeviceScene.render_rays, DESIGN section 11), on one GPU.

For c2 ({5,3,3}) and c4 ({5/2,3,3} with reflections and transparency) at 1920x1080 and 640x480:
  (a) the camera's own primary rays in pixel order, against render_float of the same view: the cost of feeding rays
      instead of generating them;
  (b) the same rays randomly shuffled: how much the caller's ray order matters;
  (c) an orthographic view: parallel rays along the camera's forward axis from a plane as wide as the scene box.
Kernel time is ntr_last_kernel_ms (CUDA events around the call's launches); Mrays/s counts the primary rays only.  Each
point is the median of --reps calls after --warmup calls.  Writes one JSON document (stdout, or --out)."""
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


def camera_rays(sc, w, h):
    """flat_origin_ray_source (tracer.hpp:60-76) for every pixel, row-major -> (origins, dirs)"""
    D = int(sc['dim'])
    fov = float(np.asarray(sc['params'])[0])
    half_w, half_h = np.float32(w / 2), np.float32(h / 2)
    fov_i = np.float32(np.tan(np.float32(fov) / 2)) / half_w
    ys, xs = np.mgrid[0:h, 0:w]
    fx = (fov_i * (xs.astype(np.float32) - half_w)).reshape(-1, 1)
    fy = (fov_i * (ys.astype(np.float32) - half_h)).reshape(-1, 1)
    ax = np.asarray(sc['cam_axes'], np.float32)
    d = ax[2][None] + ax[0][None] * fx - ax[1][None] * fy
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = np.broadcast_to(np.asarray(sc['cam_origin'], np.float32), (w * h, D))
    return np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)


def ortho_rays(sc, w, h):
    D = int(sc['dim'])
    lo, hi = np.asarray(sc['boundary'], np.float32)
    r = float(np.linalg.norm(hi - lo)) / 2
    c = (lo + hi) / 2
    ax = np.asarray(sc['cam_axes'], np.float32)
    ys, xs = np.mgrid[0:h, 0:w]
    u = ((xs + 0.5) / w * 2 - 1).reshape(-1, 1) * r
    v = ((ys + 0.5) / h * 2 - 1).reshape(-1, 1) * r * h / w
    o = c[None] - 2 * r * ax[2][None] + ax[0][None] * u - ax[1][None] * v
    d = np.broadcast_to(ax[2], (w * h, D))
    return np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)


def timed(fn, ds, warmup, reps):
    for _ in range(warmup):
        fn()
    ms, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        ms.append(ds.last_kernel_ms())
    return statistics.median(ms), statistics.median(wall)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from ntracer_b200.backend import DeviceScene
    from tests import fixtures as fx
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    out = {'gpu': q[0] if q else 'unknown', 'reps': args.reps, 'warmup': args.warmup, 'points': []}
    for cfg, fixture in SCENES.items():
        name, _, var = fixture.partition(':')
        sc, g = fx.load(name)
        if var:
            sc = fx.variant(sc, g, var)
        with DeviceScene(sc) as ds:
            for w, h in ((1920, 1080), (640, 480)):
                n = w * h
                point = {'config': cfg, 'width': w, 'height': h, 'rays': n}
                ms, wall = timed(lambda: ds.render_float(w, h), ds, args.warmup, args.reps)
                point['render_float'] = {'kernel_ms': ms, 'wall_ms': wall, 'mrays_s': n / ms / 1e3}
                o, d = camera_rays(sc, w, h)
                perm = np.random.default_rng(1).permutation(n)
                oo, od = ortho_rays(sc, w, h)
                for key, (ro, rd) in (('a_camera_rays', (o, d)), ('b_shuffled', (o[perm], d[perm])), ('c_orthographic', (oo, od))):
                    to = torch.from_numpy(np.ascontiguousarray(ro)).cuda()
                    td = torch.from_numpy(np.ascontiguousarray(rd)).cuda()
                    rgb = torch.empty((n, 3), device='cuda')

                    def call():
                        ds.render_rays_device(to, td, rgb)
                        torch.cuda.synchronize()
                    ms, wall = timed(call, ds, args.warmup, args.reps)
                    point[key] = {'kernel_ms': ms, 'wall_ms': wall, 'mrays_s': n / ms / 1e3}
                    hms, hwall = timed(lambda: ds.render_rays(ro, rd), ds, 1, 3)
                    point[key]['host_arrays_wall_ms'] = hwall
                    if key == 'a_camera_rays':
                        img = ds.render_float(w, h).reshape(-1, 3)
                        got = rgb.cpu().numpy()
                        point[key]['max_abs_diff_vs_render_float'] = float(np.abs(got - img).max())
                print(json.dumps(point), flush=True)
                out['points'].append(point)
    text = json.dumps(out, indent=1)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    else:
        print(text)


if __name__ == '__main__':
    main()
