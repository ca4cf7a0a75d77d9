"""A batch of camera views in one call against the frame-by-frame camera path (DESIGN section 9).

For c2, c4b and c4 at 1920x1080 and 640x480 it renders the first 32 cameras of the 160-step rotation of
`polytope.py --benchmark` (stream.rotation_cameras) three ways, alternating them rep after rep:
  (a) stream.render_sequence into two pinned host buffers (ntr_render_begin / ntr_render_end, two frames in flight);
  (b) DeviceScene.render_views into one pinned host buffer (ntr_render_views);
  (c) DeviceScene.render_views_device into device memory: device time from the first launch to the last (CUDA events).
It reports frames/s, kernel ms per frame, launches per frame and whether the frames of (a) and (b) agree (max |difference|
in 8-bit levels: 0 for frames without reflection passes, <= 1 with them), the median over the reps and the spread.

The block order of a views launch (tile-major with the views inner, shipped; view-major, rejected in DESIGN section 9) was
compared on c2 and c4 at 1920x1080 with --only-views --configs c2,c4 --sizes 1920x1080 under NTR_B200_LIB=<a build whose
fetch decodes the view outermost>, alternating with the shipped library.
On a box with several GPUs, group render_views of 64 views of c4 at 1920x1080 over N = 2/4/8 devices is compared with
one GPU's render_views and with a loop of per-frame ntr_group_render calls.  The GPU's name and power limit are read in
the same run.

    python tools/views_measure.py [--out profiles/views_measure.json]
"""
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

SIZES = ((1920, 1080), (640, 480))
CONFIGS = ('c2', 'c4b', 'c4')


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out
    except Exception as e:          # noqa: BLE001 -- reported, not fatal
        return ['nvidia-smi failed: %s' % e]


def scene(config):
    import bench
    name = bench.CONFIGS[config][0]
    sc, _ = bench.load_fixture(name)
    return sc


def spread(xs):
    return {'median': statistics.median(xs), 'min': min(xs), 'max': max(xs), 'reps': len(xs)}


def measure_point(config, w, h, n, reps, only_views=False):
    import torch
    from ntracer_b200 import _capi, stream
    from ntracer_b200.backend import DeviceScene
    sc = scene(config)
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    fb = fmt.pitch * h
    cams = stream.rotation_cameras(sc['cam_origin'], sc['cam_axes'], 160)[:n]
    out = {'config': config, 'width': w, 'height': h, 'views': n}
    with DeviceScene(sc) as ds:
        bufs = [torch.zeros(fb, dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
        seq = torch.zeros(n * fb, dtype=torch.uint8).pin_memory().numpy()
        batch = torch.zeros(n * fb, dtype=torch.uint8).pin_memory().numpy()
        dev = torch.zeros(n * fb, dtype=torch.uint8, device='cuda')
        st = torch.cuda.current_stream().cuda_stream

        def run_a():
            def sink(k, b):
                seq[k * fb:(k + 1) * fb] = b
            l0 = ds.launch_count()
            t0 = time.perf_counter()
            stream.render_sequence(ds, fmt, cams, bufs, sink)
            return time.perf_counter() - t0, ds.launch_count() - l0

        def run_b():
            l0 = ds.launch_count()
            t0 = time.perf_counter()
            ds.render_views(fmt, cams, batch)
            return time.perf_counter() - t0, ds.launch_count() - l0

        def run_c():
            ds.render_views_device(fmt, cams, dev.data_ptr(), dev.numel(), st)
            torch.cuda.synchronize()
            return ds.last_kernel_ms()

        for f in ((run_b, run_c) if only_views else (run_a, run_b, run_c)):
            f()                                     # warm-up: modules, queues, schedules, sort sizes
        a, b, c = [], [], []
        for _ in range(reps):
            if not only_views:
                a.append(run_a())
            b.append(run_b())
            c.append(run_c())
        if not only_views:
            out['a_render_sequence'] = {'frames_per_s': spread([n / t for t, _ in a]), 'launches_per_frame': a[-1][1] / n}
        out['b_render_views'] = {'frames_per_s': spread([n / t for t, _ in b]), 'launches_per_frame': b[-1][1] / n}
        out['c_render_views_device'] = {'kernel_ms_per_frame': spread([ms / n for ms in c])}
        if not only_views:
            out['max_abs_diff_a_b'] = int(np.abs(seq.astype(np.int16) - batch.astype(np.int16)).max())
            dev_frames = dev.cpu().numpy()
            out['max_abs_diff_b_c'] = int(np.abs(dev_frames.astype(np.int16) - batch.astype(np.int16)).max())
            # kernel ms per frame of (a): the same frames one at a time through ntr_render_device (device events)
            ks = []
            for o, ax in cams:
                ds.set_camera(o, ax)
                ds.render_device(fmt, dev.data_ptr(), fb, st)
                torch.cuda.synchronize()
                ks.append(ds.last_kernel_ms())
            out['a_kernel_ms_per_frame_single'] = statistics.mean(ks)
    return out


def measure_groups(n=64, w=1920, h=1080, reps=3):
    import torch
    from ntracer_b200 import _capi, stream
    from ntracer_b200.backend import DeviceGroup, DeviceScene, device_count
    ndev = device_count()
    if ndev < 2:
        return 'not measured: %d GPU on this box' % ndev
    sc = scene('c4')
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    fb = fmt.pitch * h
    cams = stream.rotation_cameras(sc['cam_origin'], sc['cam_axes'], 160)[:n]
    out = torch.zeros(n * fb, dtype=torch.uint8).pin_memory().numpy()
    res = {'config': 'c4', 'width': w, 'height': h, 'views': n}
    with DeviceScene(sc) as ds:
        ds.render_views(fmt, cams[:4], out)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            ds.render_views(fmt, cams, out)
            ts.append(time.perf_counter() - t0)
        one = n / statistics.median(ts)
        res['one_gpu_render_views_fps'] = one
    for g_n in (2, 4, 8):
        if g_n > ndev:
            res['N=%d' % g_n] = 'not measured: %d GPUs on this box' % ndev
            continue
        with DeviceGroup(sc, g_n) as g:
            g.render_views(fmt, cams[:g_n], out)
            tv, tl = [], []
            frame = out[:fb]
            for _ in range(reps):
                t0 = time.perf_counter()
                g.render_views(fmt, cams, out)
                tv.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                for o, ax in cams:
                    g.set_camera(o, ax)
                    g.render(fmt, frame)
                tl.append(time.perf_counter() - t0)
            fv, fl = n / statistics.median(tv), n / statistics.median(tl)
            res['N=%d' % g_n] = {'group_render_views_fps': fv, 'group_render_loop_fps': fl,
                                 'render_views_scaling_efficiency': fv / (g_n * one),
                                 'render_loop_scaling_efficiency_vs_one_gpu_views': fl / (g_n * one)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'views_measure.json'))
    ap.add_argument('--views', type=int, default=32)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--configs', default=','.join(CONFIGS))
    ap.add_argument('--sizes', default=','.join('%dx%d' % s for s in SIZES))
    ap.add_argument('--only-views', action='store_true', help='(b) and (c) only, printed as one JSON line')
    args = ap.parse_args()
    sizes = [tuple(int(v) for v in s.split('x')) for s in args.sizes.split(',')]
    configs = args.configs.split(',')
    if args.only_views:
        print(json.dumps([measure_point(c, w, h, args.views, args.reps, only_views=True) for c in configs for w, h in sizes]))
        return
    res = {'gpu': gpu_info(), 'views': args.views, 'reps': args.reps,
           'note': 'frames/s: wall clock around the whole call (host buffers pinned); kernel ms: CUDA events from the first '
                   'launch to the last of the call, per frame; a_kernel_ms_per_frame_single: the same frames one at a time '
                   'through ntr_render_device'}
    res['points'] = [measure_point(c, w, h, args.views, args.reps) for c in configs for w, h in sizes]
    res['groups'] = measure_groups()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
