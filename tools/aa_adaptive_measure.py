"""Cost and error of adaptive supersampling (Scene.set_supersampling(s, threshold) / ntr_scene_set_supersampling_threshold)
on the GPU.

For each measured point (scene, frame size W x H) and factor s it times, alternating them, the plain frame (factor 1), the
fully supersampled frame (factor s) and, for every threshold t, the adaptive frame (factor s, threshold t), each on a
DeviceScene of its own.  Kernel time is ntr_last_kernel_ms (CUDA events around the frame's kernels), best and median over
the timed repetitions after warm-up.  The refined share is the refine mask's count over W x H.  The error is that of the
adaptive frame against the full-SS frame, both packed to 8-bit RGB: the mean absolute difference in 8-bit steps and the
share of channel values more than 2 steps apart.  The card's name and power limit are read in the same run and written
beside the numbers.

    python tools/aa_adaptive_measure.py OUT_DIR [--reps 5] [--warmup 2] [--points c2:1920x1080,...] [--factors 2,4]
        [--thresholds 1,4,16]     (thresholds in 8-bit steps: t = n / 255)
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from aa_measure import SCENES, card_info, rays, stats  # noqa: E402

POINTS = 'c2:1920x1080,c4b:1920x1080,c4b:3840x2160,c4:1920x1080'


def timed(ds, fmt, host):
    ds.render(fmt, host)
    return ds.last_kernel_ms()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('out_dir')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--points', default=POINTS)
    ap.add_argument('--factors', default='2,4')
    ap.add_argument('--thresholds', default='1,4,16')
    args = ap.parse_args()
    if args.reps < 5:
        ap.error('--reps must be at least 5')
    import torch
    import bench
    from ntracer_b200 import _capi
    from ntracer_b200.backend import DeviceScene
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures on the GPU only')
    os.makedirs(args.out_dir, exist_ok=True)
    factors = [int(f) for f in args.factors.split(',')]
    steps = [int(n) for n in args.thresholds.split(',')]
    result = {'card': card_info(), 'reps': args.reps, 'warmup': args.warmup, 'thresholds_in_8bit_steps': steps, 'points': []}
    for point in args.points.split(','):
        cfg, _, size = point.partition(':')
        w, h = (int(v) for v in size.split('x'))
        sc, _ = bench.load_fixture(SCENES[cfg])
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        host = torch.zeros(fmt.pitch * h, dtype=torch.uint8).pin_memory().numpy()
        for s in factors:
            devs = [DeviceScene(sc, 0) for _ in range(2 + len(steps))]       # plain, full, adaptive per threshold
            try:
                for k, d in enumerate(devs):
                    d.set_supersampling(1 if k == 0 else s)
                    if k >= 2:
                        d.set_supersampling_threshold(steps[k - 2] / 255)
                for _ in range(args.warmup):
                    for d in devs:
                        timed(d, fmt, host)
                ms = [[] for _ in devs]
                for _ in range(args.reps):      # alternating: every mode sees the same state of the shared machine
                    for k, d in enumerate(devs):
                        ms[k].append(timed(d, fmt, host))
                full = devs[1].render(fmt).astype(np.int32)
                plain = devs[0].render(fmt).astype(np.int32)
                row = {'config': cfg, 'fixture': SCENES[cfg], 'width': w, 'height': h, 'factor': s,
                       'plain': {'kernel_ms': stats(ms[0]), 'counters': devs[0].counters()},
                       'full_ss': {'kernel_ms': stats(ms[1]), 'counters': devs[1].counters()},
                       'plain_vs_full_ss': {'mean_8bit_steps': float(np.abs(plain - full).mean()),
                                            'share_over_2_steps': float((np.abs(plain - full) > 2).mean())},
                       'adaptive': []}
                for k in range(2, len(devs)):
                    img = devs[k].render(fmt).astype(np.int32)
                    _, n = devs[k].refine_mask()
                    cnt = devs[k].counters()
                    a = {'threshold_8bit_steps': steps[k - 2], 'kernel_ms': stats(ms[k]), 'counters': cnt,
                         'refined_share': n / (w * h),
                         'vs_full_ss': {'mean_8bit_steps': float(np.abs(img - full).mean()),
                                        'share_over_2_steps': float((np.abs(img - full) > 2).mean())},
                         'kernel_ratio_to_full_ss_best': min(ms[k]) / min(ms[1]),
                         'kernel_ratio_to_full_ss_median': statistics.median(ms[k]) / statistics.median(ms[1]),
                         'Mrays_per_s': rays(cnt) / min(ms[k]) / 1e3}
                    row['adaptive'].append(a)
                    print('%-4s %dx%d s=%d t=%2d/255  kernel ms plain %.3f  full %.3f  adaptive %.3f (x%.3f of full)  '
                          'refined %.2f %%  vs full: mean %.3f, >2 steps %.3f %%'
                          % (cfg, w, h, s, steps[k - 2], min(ms[0]), min(ms[1]), min(ms[k]), a['kernel_ratio_to_full_ss_best'],
                             100 * a['refined_share'], a['vs_full_ss']['mean_8bit_steps'],
                             100 * a['vs_full_ss']['share_over_2_steps']), flush=True)
                result['points'].append(row)
            finally:
                for d in devs:
                    d.close()
        del host
    result['card_after'] = card_info()
    with open(os.path.join(args.out_dir, 'aa_adaptive_measure.json'), 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
