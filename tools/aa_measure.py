"""Cost of supersampled anti-aliasing (Scene.set_supersampling / ntr_scene_set_supersampling) on the GPU.

For each measured point (scene, frame size W x H, factor s) it times two renders of the same rays, alternating them:
  * the supersampled frame: ntr_render of W x H with factor s (the NTR_F_SS primary pass);
  * the reference cost: a 1-spp ntr_render of the sW x sH view, what a user had to do before (then shrink on the host).
Kernel time is ntr_last_kernel_ms (CUDA events around the frame's kernels), end-to-end time is the host clock around
ntr_render into pinned memory; both are best and median over the timed repetitions after warm-up.  Rays/s are the
frame's primary + shadow + reflection rays (device counters) over the kernel time.  The card's name and power limit are
read in the same run and written beside the numbers.

    python tools/aa_measure.py OUT_DIR [--reps 5] [--warmup 2] [--points c2:1920x1080,...] [--factors 1,2,3,4]
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

SCENES = {'c2': 'cell120', 'c4': 'ggs120:refl_transp', 'c4b': 'ssc120:refl_transp'}
POINTS = 'c2:1920x1080,c4b:1920x1080,c4b:3840x2160,c4:1920x1080'


def card_info():
    import torch
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
    except (OSError, subprocess.SubprocessError) as e:
        info['nvidia_smi'] = 'unavailable: %s' % e
    return info


def rays(cnt):
    return cnt['primary_rays'] + cnt['shadow_rays'] + cnt['reflection_rays']


def measure(ds, fmt, factor, host):
    ds.set_supersampling(factor)
    t0 = time.perf_counter()
    ds.render(fmt, host)
    e2e = (time.perf_counter() - t0) * 1e3
    return ds.last_kernel_ms(), e2e, ds.counters()


def stats(v):
    return {'best': min(v), 'median': statistics.median(v), 'all': v}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('out_dir')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--points', default=POINTS)
    ap.add_argument('--factors', default='1,2,3,4')
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
    result = {'card': card_info(), 'reps': args.reps, 'warmup': args.warmup, 'points': []}
    for point in args.points.split(','):
        cfg, _, size = point.partition(':')
        w, h = (int(v) for v in size.split('x'))
        sc, _ = bench.load_fixture(SCENES[cfg])
        with DeviceScene(sc, 0) as ss_dev, DeviceScene(sc, 0) as big_dev:
            for s in factors:
                fmt = _capi.make_image_format(w, h, _capi.RGB8)
                big_fmt = _capi.make_image_format(s * w, s * h, _capi.RGB8)
                host = torch.zeros(fmt.pitch * h, dtype=torch.uint8).pin_memory().numpy()
                big_host = torch.zeros(big_fmt.pitch * s * h, dtype=torch.uint8).pin_memory().numpy()
                for _ in range(args.warmup):
                    measure(ss_dev, fmt, s, host)
                    measure(big_dev, big_fmt, 1, big_host)
                k_ss, e_ss, k_big, e_big = [], [], [], []
                for _ in range(args.reps):          # alternating: both see the same state of the shared machine
                    k, e, c_ss = measure(ss_dev, fmt, s, host)
                    k_ss.append(k); e_ss.append(e)
                    k, e, c_big = measure(big_dev, big_fmt, 1, big_host)
                    k_big.append(k); e_big.append(e)
                row = {
                    'config': cfg, 'fixture': SCENES[cfg], 'width': w, 'height': h, 'factor': s,
                    'ss': {'kernel_ms': stats(k_ss), 'e2e_ms': stats(e_ss), 'counters': c_ss,
                           'Mrays_per_s': rays(c_ss) / min(k_ss) / 1e3},
                    'big_view_1spp': {'width': s * w, 'height': s * h, 'kernel_ms': stats(k_big), 'e2e_ms': stats(e_big),
                                      'counters': c_big, 'Mrays_per_s': rays(c_big) / min(k_big) / 1e3},
                }
                row['kernel_ratio_best'] = min(k_ss) / min(k_big)
                row['kernel_ratio_median'] = statistics.median(k_ss) / statistics.median(k_big)
                result['points'].append(row)
                print('%-4s %dx%d s=%d  kernel ms ss %.3f / big %.3f (ratio %.3f)  e2e ms ss %.2f / big %.2f  Mrays/s %.0f'
                      % (cfg, w, h, s, min(k_ss), min(k_big), row['kernel_ratio_best'], min(e_ss), min(e_big),
                         row['ss']['Mrays_per_s']), flush=True)
                del host, big_host
    result['card_after'] = card_info()
    with open(os.path.join(args.out_dir, 'aa_measure.json'), 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
