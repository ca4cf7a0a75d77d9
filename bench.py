#!/usr/bin/env python3
"""bench.py -- headline benchmark of the render path (BASELINE.json: Mrays/s and frame time).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c4|c4b|c2|...] [--impl ours|reference] [--dump-outputs DIR]

A step = one frame of the workload.  The workload is the frame BASELINE.json's metric and north star are quoted on
(configs[3]): the great grand stellated 120-cell {5/2,3,3} as a CompositeScene over the reference's own k-d tree
(tests/golden/ggs120.npz), 3840x2160, PointLight + GlobalLight, shadows, reflections depth 4, 12 transparent cells,
RGB8 output.  The line also carries `secondary`: the same measurement for {5/2,5,3} (the symbol BASELINE.json spells,
c4b) and for configs[1] (c2, 1920x1080 {5,3,3}).  N>1 (launched with torchrun, one rank per GPU): the same frame
partitioned by interleaved 32-pixel tile rows, scene replicated, every rank storing its rows into one frame on rank
0's GPU over NVLink.

One JSON line is printed by rank 0; see the prompt contract for the keys.  `value` = device-resident
throughput (kernels only, CUDA events), `e2e` = the same metric through ntr_render with a HOST destination
buffer (camera upload + D2H of the frame inside the timed region).  `cpu_baseline` / `--impl reference` time
the reference's own multithreaded CPU renderer (oracle/_ref) on this box's host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (fixture, width, height, description)
    'c1': ('box4', 640, 480, "config 1: 4-D tesseract BoxScene 640x480"),
    'c2': ('cell120', 1920, 1080, "config 2: 4-D 120-cell {5,3,3} CompositeScene 1920x1080, PointLight+GlobalLight, shadows on"),
    'c3': ('solids6', 1920, 1080, "config 3 stand-in: 6-D solids (2 hypercubes, 2 hyperspheres; SURVEY 8d C3), 1920x1080, reflections depth 4, PointLight, shadows, fixed-dim path"),
    'c4': ('ggs120:refl_transp', 3840, 2160, "config 4: great grand stellated 120-cell {5/2,3,3} 3840x2160, lights, shadows, reflectivity 0.3 depth 4, 12 of 120 cells opacity 0.5"),
    'c5': ('soup10:1000000', 3840, 2160, "config 5: 10-D synthetic simplex soup, 1,000,000 TrianglePrototypes (SURVEY 8d C5 generator, seed 1234), fixed 10-D kernel family (NTR_FORCE_GENERIC=1: the run-time-dimension family), 3840x2160, camera light only; tree from this repo's native builder (max_depth 17)"),
    'c5s': ('soup10:16000', 3840, 2160, "config 5 reduced: the same 10-D soup generator with 16,000 simplexes (what the reference CPU renderer can be timed on), 3840x2160"),
    'c4b': ('ssc120:refl_transp', 3840, 2160, "config 4 as BASELINE.json spells its symbol: small stellated 120-cell {5/2,5,3} (7,200 simplexes, leaves <= 48 items), 3840x2160, lights, shadows, reflectivity 0.3 depth 4, 12 transparent cells (opacity 0.5)"),
    'c4o': ('ggs120', 3840, 2160, "config 4 (opaque variant): great grand stellated 120-cell {5/2,3,3} 3840x2160, lights, shadows, reflectivity 0.3 depth 4"),
}
# BASELINE.json's metric, verbatim.  `value` is the Mrays/s half (rays of a frame / frame time; frames with bounce passes
# count their reflection / transparency rays too, SURVEY.md 8d, see config.rays_counted); the "4K frame time" half is
# ms_per_step / config.frame_ms of the same line, and the 1/2/4/8 curve is this line at --gpus 1, 2, 4, 8.
METRIC = 'Mrays/sec (primary+shadow) and 4K frame time at 1/2/4/8 B200 vs CPU cores'


def load_fixture(name):
    from tests import fixtures as fx
    name, _, var = name.partition(':')
    if name == 'soup10':
        # BASELINE config 5: generated here (no fixture can hold 1 M simplexes); scene construction (records + k-d
        # tree) runs in the native host-side builder and is NOT part of any timed region
        from ntracer_b200 import bulk
        sc = bulk.simplex_scene(bulk.soup(10, int(var)), max_depth=int(os.environ.get('NTR_BENCH_SOUP_DEPTH', '17')))
        sc['cam_origin'] = np.array([0, 0, -3] + [0] * 7, np.float32)
        return sc, {}
    sc, g = fx.load(name)
    if var:
        sc = fx.variant(sc, g, var)
    return sc, g


def flops_per_frame(dim, cnt, n_lights):
    """ALGORITHMIC flops of one frame (SURVEY.md section 8(d), DESIGN.md section 6) from the reference
    algorithm's counters (counting CPU restatement = the oracle)."""
    D = dim
    rays = cnt['primary_rays'] + cnt['reflection_rays']
    return (cnt['primary_rays'] * (7 * D + 2) + rays * 2 * D * D + cnt['node_steps'] * 4 +
            cnt['simplex_tests'] * (2 * D * D + 5 * D) + cnt['solid_tests'] * 8 * D * D +
            cnt['shaded_hits'] * max(n_lights, 1) * (20 * D + 60))


def bytes_per_frame(dim, cnt, frame_bytes):
    """ALGORITHMIC bytes: 16 B per node step + one simplex record per simplex test + the frame."""
    D = dim
    return cnt['node_steps'] * 16 + cnt['simplex_tests'] * 4 * ((D + 1) * D + 1) + frame_bytes


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def reference_arm(args, sc, g, w, h, rays_per_frame):
    """Times the reference's own CPU renderer (oracle/_ref: unmodified Rouslan/NTracer built by
    oracle/build_ref.sh) on this box's host cores.  Falls back to the C port (oracle/ntr_oracle.c, OpenMP)."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    cores = os.cpu_count() or 1
    import ref_bridge as rb
    times = []
    stream_ref = None
    if int(sc['simplex'].shape[0]) > 50000 if int(sc['kind']) == 1 else False:
        return {'value': None, 'unit': 'Mrays/s', 'cores': cores, 'kind': 'reference',
                'sample': 'not run: the reference cannot hold %d primitives (one Python object each, O(N^2) batch grouping); '
                          'see config c5s for the same generator at 16,000 simplexes timed on both sides' % int(sc['simplex'].shape[0])}
    if rb.have_reference():
        nt, scene, prims = rb.import_scene(sc)
        rb.make_immortal(prims.values())     # see ref_bridge.make_immortal: the reference races on primitive refcounts
        ntr = rb.load_reference()
        def rfmt(ww, hh):
            return ntr.ImageFormat(ww, hh, [ntr.Channel(8, 1, 0, 0), ntr.Channel(8, 0, 1, 0), ntr.Channel(8, 0, 0, 1)])
        r = ntr.BlockingRenderer()          # threads=-1: hardware_concurrency() workers (render.cpp:829-838)
        # The reference's workers check `busy_threads` WITHOUT the lock when they start (render.cpp:773-777): a worker
        # caught between that check and its first wait when render() posts a job is counted in busy_threads but sleeps
        # through the job, and render() then waits forever (seen as a hang of the first frame on a busy box).  Give
        # the workers time to reach their wait before the first job; every later job is posted under the lock.
        time.sleep(1.0)
        # probe at 1/8 resolution (also the warm-up: late-starting workers, SURVEY 8a-Q10), then pick the largest
        # frame of the same view (full, 1/2, 1/4 ... linear size) whose estimated cost fits ~6 s per frame
        pw, ph = max(w // 8, 32), max(h // 8, 32)
        pbuf = bytearray(pw * ph * 3)
        r.render(pbuf, rfmt(pw, ph), scene)
        t = time.perf_counter()
        r.render(pbuf, rfmt(pw, ph), scene)
        probe = (time.perf_counter() - t) / (pw * ph)
        div = 1
        while probe * (w // div) * (h // div) > 6.0 and div < 16:
            div *= 2
        sw, sh = w // div, h // div
        fmt = rfmt(sw, sh)
        buf = bytearray(sw * sh * 3)
        budget = time.perf_counter() + 25.0
        for _ in range(max(1, min(args.steps, 5))):
            t = time.perf_counter()
            r.render(buf, fmt, scene)
            times.append((time.perf_counter() - t) * (w * h) / (sw * sh))    # scaled to the full frame's pixel count
            if time.perf_counter() > budget:
                break
        if args.stream_frames >= 2 and div == 1 and min(times) < 0.5:
            # the rotating-camera loop of polytope.py --benchmark on the same camera path as the GPU's stream leg:
            # a bounded sample of its frames (every n-th camera), one BlockingRenderer.render per frame
            from ntracer_b200 import stream as nts
            cams = nts.rotation_cameras(sc['cam_origin'], sc['cam_axes'], args.stream_frames)
            pick = cams[::max(1, len(cams) // 8)][:8]
            st_times = []
            for o, a in pick:
                cam = nt.Camera()
                cam.origin = nt.Vector(*[float(x) for x in o])
                for i in range(int(sc['dim'])):
                    cam.axes[i] = nt.Vector(*[float(x) for x in a[i]])
                scene.set_camera(cam)
                t = time.perf_counter()
                r.render(buf, fmt, scene)
                st_times.append(time.perf_counter() - t)
            stream_ref = {'frames_sampled': len(pick), 'of': len(cams), 'ms_per_frame': 1e3 * sum(st_times) / len(st_times),
                          'frames_per_s': len(st_times) / sum(st_times)}
        kind = 'reference'
        sample = ('%d frame(s) of the same view at %dx%d (1/%d linear size; times scaled by pixel count to %dx%d), BlockingRenderer '
                  'all cores, SSE4.2 build (the AVX paths of the reference do not compile)' % (len(times), sw, sh, div, w, h))
    else:
        from tests import oracle_lib as ol
        from ntracer_b200 import _capi
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        ol.render_packed(sc, _capi.make_image_format(64, 36, _capi.RGB8))
        for _ in range(2):
            t = time.perf_counter()
            ol.render_packed(sc, fmt)
            times.append(time.perf_counter() - t)
        kind = 'port'
        sample = '%d full %dx%d frames, oracle C port with OpenMP' % (len(times), w, h)
    best = min(times)
    out = {'value': rays_per_frame / best / 1e6, 'unit': 'Mrays/s', 'cores': cores, 'kind': kind, 'sample': sample,
           'sec_per_frame': best, 'median_sec_per_frame': statistics.median(times), 'Mpix_per_s': w * h / best / 1e6}
    if stream_ref:
        out['stream'] = stream_ref
    return out


TAIL_TIMEOUT_S = int(os.environ.get('NTR_BENCH_TAIL_TIMEOUT', '480'))
REFERENCE_TIMEOUT_S = int(os.environ.get('NTR_BENCH_REFERENCE_TIMEOUT', '300'))


def reference_arm_subprocess(args):
    """cpu_baseline of the GPU arm: the reference arm in a process of its own (`bench.py --impl reference`), so that a
    crash or hang of the reference's renderer (see ref_bridge.make_immortal) cannot take the measurement with it."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--config', args.config, '--steps', str(args.steps),
           '--warmup', str(args.warmup), '--stream-frames', str(args.stream_frames)]
    env = dict(os.environ, RANK='0', WORLD_SIZE='1', LOCAL_RANK='0')
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=REFERENCE_TIMEOUT_S, env=env)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith('{'):
                return json.loads(ln)['cpu_baseline']
        why = 'no result (exit code %d): %s' % (out.returncode, out.stderr.strip()[-300:])
    except subprocess.TimeoutExpired:
        why = 'did not finish within %d s' % REFERENCE_TIMEOUT_S
    return {'value': None, 'unit': 'Mrays/s', 'cores': os.cpu_count() or 1, 'kind': 'reference', 'sample': 'reference arm failed: ' + why}


def kernel_name(sc, dim):
    """The kernel that dominates a frame of this scene (one render_pass_kernel instantiation per dimension and variant)."""
    fixed = 3 <= dim <= 10 and not int(os.environ.get('NTR_FORCE_GENERIC', '0') or 0)
    general = int(sc['kind']) == 1 and (bool(np.any(np.asarray(sc['materials'])[:, 6] < 1)) or len(sc['solids']) > 0)
    name = 'render_pass_kernel<%d,%d>' % (dim if fixed else 0, 1 if general else 0)
    if int(sc['kind']) == 1 and len(sc['nodes']):
        nodes = np.asarray(sc['nodes']).reshape(-1, 4)
        leaves = (nodes[:, 0] & 0x80000000) != 0
        if leaves.any() and int(nodes[leaves, 2].max()) >= 256:
            # scenes with big leaves: the bounce passes run the warp-synchronous instantiation (flag bit 2, capi.cu)
            name += ' (primary pass) + render_pass_kernel<%d,%d> (bounce passes)' % (dim if fixed else 0, (1 if general else 0) | 4)
    return name


def measured_traffic(config, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    capture of this workload (profiles/r02_traffic.json, written by tools/ncu_traffic.py); None when there is none."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))[config]
        if t['kernel'].split(',')[0] == kernel.split(',')[0]:           # same kernel family (dimension)
            return t
    except Exception:
        pass
    return None


class Workload:
    """One bench config on this rank's GPU: scene upload, the frame in the memory of rank 0's GPU, timed steps."""
    def __init__(self, name, rank, local_rank, world):
        import torch
        from ntracer_b200 import _capi
        from ntracer_b200 import dist as ntd
        from ntracer_b200.backend import DeviceScene
        self.name, self.rank, self.world = name, rank, world
        fixture, self.w, self.h, self.desc = CONFIGS[name]
        self.sc, self.g = load_fixture(fixture)
        self.dim = int(self.sc['dim'])
        self.ds = DeviceScene(self.sc, local_rank)
        self.fmt = _capi.make_image_format(self.w, self.h, _capi.RGB8)
        self.frame_bytes = self.w * self.h * 3
        self.gather = os.environ.get('NTR_BENCH_GATHER', 'peer')
        if world > 1 and self.gather == 'nccl':
            self.dr = ntd.DistributedRenderer(self.ds, self.fmt)
        else:
            self.dr = ntd.PeerFrameRenderer(self.ds, self.fmt)
        self.host_frame = torch.zeros(self.fmt.pitch * self.h, dtype=torch.uint8).pin_memory()
        self.cam_o = np.ascontiguousarray(self.sc['cam_origin'], np.float32)
        self.cam_a = np.ascontiguousarray(self.sc['cam_axes'], np.float32)
        self.ev0, self.ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # ray counts of the frame (device counters of a synchronous render of the whole frame)
        self.ds.render_float(self.w, self.h)
        self.cnt = self.ds.counters()
        self.rays = self.cnt['primary_rays'] + self.cnt['shadow_rays'] + self.cnt['reflection_rays']

    def step_device(self):
        """one frame, inputs resident, output stays on the device (the whole frame ends up in rank 0's GPU memory);
        returns device ms between CUDA events on the launching stream"""
        dr = self.dr
        self.ev0.record(dr.stream)
        if self.gather == 'nccl' and self.world > 1:
            dr.render_strip(); dr.gather(); dr.frame_on_device()
        else:
            dr.render(); dr.fence()
        self.ev1.record(dr.stream)
        self.ev1.synchronize()
        return self.ev0.elapsed_time(self.ev1)

    def step_e2e(self):
        """the same frame through the host-buffer path: camera upload + render (+ completion fence) + D2H"""
        self.ds.set_camera(self.cam_o, self.cam_a)
        if self.world == 1:
            self.ds.render(self.fmt, self.host_frame.numpy())       # ntr_render: what BlockingRenderer.render calls
        else:
            self.dr.render_to_host()

    def step_e2e_pageable(self):
        """the same call with the destination the API's real caller passes: a plain (pageable) bytearray"""
        if not hasattr(self, 'pageable'):
            self.pageable = bytearray(self.fmt.pitch * self.h)
        self.ds.set_camera(self.cam_o, self.cam_a)
        self.ds.render(self.fmt, self.pageable)

    def _pixels(self, packed):
        return np.asarray(packed, np.uint8).reshape(self.h, self.fmt.pitch)[:, :self.w * 3].reshape(self.h, self.w, 3).copy()

    def device_frame(self):
        """rank 0: the frame step_device left in GPU memory, as (height, width, 3) uint8; None on the other ranks"""
        from ntracer_b200.dist import PeerFrameRenderer
        if self.rank != 0:
            return None
        if isinstance(self.dr, PeerFrameRenderer):
            buf = np.zeros(self.fmt.pitch * self.h, np.uint8)
            self.dr.frame.download(self.fmt, buf, self.dr.stream.cuda_stream)
            self.dr.stream.synchronize()
            return self._pixels(buf)
        frame = self.dr.frame_on_device()
        self.dr.stream.synchronize()
        return self._pixels(frame.cpu().numpy())

    def e2e_frame(self):
        """rank 0: the frame step_e2e copied into host memory; None on the other ranks"""
        if self.rank != 0:
            return None
        return self._pixels(self.host_frame.numpy() if self.world == 1 else self.dr.host.numpy())

    def close(self):
        if hasattr(self.dr, 'close'):
            self.dr.close()
        self.ds.close()


# --dump-outputs: frames with more pixels than this are written as a fixed, seeded sample of their pixels (every run picks
# the same pixels), so that the dump of a 4K headline frame and its secondaries stays far below 64 MB
DUMP_SAMPLE_PIXELS = 1 << 19
DUMP_SEED = 20240601


def dump_outputs(directory, frames):
    """frames: {name: (height, width, 3) uint8} -> directory/<name>.npy in float32, 0..255: the whole frame
    (height, width, 3), or [DUMP_SAMPLE_PIXELS, 3] pixels at the seeded sample of flat pixel indices, in increasing order."""
    os.makedirs(directory, exist_ok=True)
    for name, px in frames.items():
        h, w, _ = px.shape
        if h * w > DUMP_SAMPLE_PIXELS:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, DUMP_SAMPLE_PIXELS, replace=False))
            px = px.reshape(h * w, 3)[idx]
        np.save(os.path.join(directory, name + '.npy'), px.astype(np.float32))


def timed(wl, steps, warmup, flush, barrier, keep=False):
    """-> (device ms per step, e2e ms per step, launches), each the MAX over ranks of the per-rank totals.
    keep: also store the frames of the last device step and the last e2e step in wl.kept (rank 0; outside the timing)"""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        wl.step_device()
        wl.step_e2e()
    barrier()
    launches0 = wl.ds.launch_count()
    dev_ms = []
    for _ in range(steps):
        flush.zero_()                   # L2 flush between timed iterations
        barrier()
        dev_ms.append(wl.step_device())
    barrier()
    if keep:
        wl.kept = {'frame': wl.device_frame()}
    e2e_s = []
    for _ in range(steps):
        flush.zero_()
        barrier()
        t = time.perf_counter()
        wl.step_e2e()
        e2e_s.append(time.perf_counter() - t)
    barrier()
    if keep:
        wl.kept['frame_e2e'] = wl.e2e_frame()
    launches = wl.ds.launch_count() - launches0
    wl.pageable_ms = None
    if wl.world == 1:                   # BlockingRenderer.render is handed a bytearray: the same frames into pageable memory
        wl.step_e2e_pageable()
        pg = []
        for _ in range(steps):
            flush.zero_()
            barrier()
            t = time.perf_counter()
            wl.step_e2e_pageable()
            pg.append(time.perf_counter() - t)
        wl.pageable_ms = 1e3 * sum(pg) / steps
    tot = torch.tensor([sum(dev_ms), sum(e2e_s) * 1e3, float(launches)], dtype=torch.float64, device='cuda')
    if wl.world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    d, e, l = [float(v) for v in tot.tolist()]
    return d / steps, e / steps, int(l), dev_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--config', default='c4', choices=sorted(CONFIGS))
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help='skip the secondary workloads (c4b, c2) reported beside the headline one')
    ap.add_argument('--stream-frames', type=int, default=160,
                    help='frames of the rotating-camera loop (polytope.py --benchmark); 0 = skip that leg')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the frames of the last device step and the last e2e step of every timed '
                         'workload to DIR/<config>_frame.npy and DIR/<config>_frame_e2e.npy (float32; frames over %d pixels as '
                         'a fixed seeded sample of their pixels)' % DUMP_SAMPLE_PIXELS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the frames of --impl ours')
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    fixture, w, h, desc = CONFIGS[args.config]

    if args.impl == 'reference':
        if rank != 0:
            return 0
        sc, g = load_fixture(fixture)

        def ref_watchdog():
            print(json.dumps({'impl': 'reference', 'unavailable': 'the reference renderer did not finish within %d s '
                              '(its worker threads race on Python refcounts, see oracle/ref_bridge.py)' % (2 * REFERENCE_TIMEOUT_S)}), flush=True)
            os._exit(0)
        rwd = threading.Timer(2 * REFERENCE_TIMEOUT_S, ref_watchdog)
        rwd.daemon = True
        rwd.start()
        if int(sc['kind']) == 1 and int(sc['simplex'].shape[0]) > 50000:
            # (config 5 proper) nothing to time: reference_arm says why; no ray counting on a scene the restatement needs
            # half an hour for either
            base = reference_arm(args, sc, g, w, h, 0)
            rwd.cancel()
            print(json.dumps({'impl': 'reference', 'unavailable': base['sample'], 'metric': METRIC, 'unit': 'Mrays/s',
                              'n_gpus': args.gpus, 'config': {'workload': desc, 'width': w, 'height': h}, 'cpu_baseline': base}), flush=True)
            return 0
        # ray counts of the frame from the counting CPU restatement (the reference does not count rays); counted on a
        # frame of 1/4 the linear size and scaled when the full frame would take the restatement minutes (the counts per
        # pixel of the same view agree to 0.1 % between the two sizes)
        from tests import oracle_lib as ol
        div = 4 if w * h > 4000000 else 1
        _, cnt = ol.render_float(sc, w // div, h // div, with_counters=True)
        rays = (cnt['primary_rays'] + cnt['shadow_rays'] + cnt['reflection_rays']) * div * div
        base = reference_arm(args, sc, g, w, h, rays)
        line = {'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'Mrays/s', 'n_gpus': args.gpus,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': base['sec_per_frame'] * 1e3,
                'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': desc, 'width': w, 'height': h, 'rays_per_frame': rays,
                           'frame_ms': base['sec_per_frame'] * 1e3, 'frames_per_s': 1.0 / base['sec_per_frame']},
                'cpu_baseline': base,
                'e2e': {'value': base['value'], 'unit': 'Mrays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        rwd.cancel()
        print(json.dumps(line), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    from ntracer_b200.backend import measure_fp32_peak

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = Workload(args.config, rank, local_rank, world)
    sc, g, dim, frame_bytes = wl.sc, wl.g, wl.dim, wl.frame_bytes
    n_lights = (len(sc.get('point_lights', [])) + len(sc.get('global_lights', []))) if int(sc['kind']) == 1 else 0
    cnt_gpu, rays = wl.cnt, wl.rays

    if os.environ.get('NTR_BENCH_BREAKDOWN'):
        os.environ['NTR_PASS_TIMING'] = '1'
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    keep = bool(args.dump_outputs)
    ms_per_step, e2e_ms, launches, dev_ms = timed(wl, args.steps, args.warmup, flush, barrier, keep)
    clocks = sampler.stop() if sampler else None
    outputs = {'%s_%s' % (args.config, k): v for k, v in wl.kept.items()} if keep else {}

    # the secondary workloads, measured the same way: BASELINE.json spells config 4's symbol {5/2,5,3}
    # (c4b) while naming the {5/2,3,3} polytope (c4, the headline); c2 is the round-1 headline
    secondary = {}
    if not args.no_secondary and args.config == 'c4':
        for name in ('c4b', 'c2'):
            w2 = Workload(name, rank, local_rank, world)
            d2, e2, l2, _ = timed(w2, args.steps, 3, flush, barrier, keep)
            if keep:
                outputs.update(('%s_%s' % (name, kk), v) for kk, v in w2.kept.items())
            secondary[name] = {'workload': w2.desc, 'width': w2.w, 'height': w2.h, 'rays_per_frame': w2.rays, 'steps': args.steps,
                               'ms_per_step': d2, 'value': w2.rays / (d2 * 1e-3) / 1e6, 'unit': 'Mrays/s',
                               'e2e_ms_per_step': e2, 'e2e_value': w2.rays / (e2 * 1e-3) / 1e6, 'frames_per_s': 1e3 / d2,
                               'gpu_launches': l2}
            w2.close()
    if keep and rank == 0:
        dump_outputs(args.dump_outputs, outputs)

    ds = wl.ds

    def stream_leg():
        """the interactive loop (SURVEY 8(f)-3): rotating camera, one frame per camera, two frames in flight, every frame
        copied into a pinned host buffer (ntr_render_begin / ntr_render_end); wall clock around the whole loop"""
        from ntracer_b200 import stream as nts
        n_frames = int(max(8, min(args.stream_frames, 4000.0 / max(statistics.median(dev_ms), 1e-3))))
        cams = nts.rotation_cameras(wl.cam_o, wl.cam_a, args.stream_frames)[:n_frames]
        bufs = [wl.host_frame.numpy(), torch.zeros(wl.fmt.pitch * h, dtype=torch.uint8).pin_memory().numpy()]
        nts.render_sequence(ds, wl.fmt, cams[:4], bufs)                    # warm-up
        torch.cuda.synchronize()
        launches_s0 = ds.launch_count()
        t = time.perf_counter()
        nts.render_sequence(ds, wl.fmt, cams, bufs)
        torch.cuda.synchronize()
        el = time.perf_counter() - t
        ds.set_camera(wl.cam_o, wl.cam_a)
        return {'frames': n_frames, 'camera_path': 'polytope.py RotatingCamera, %d steps per turn' % args.stream_frames,
                'in_flight': 2, 'ms_per_frame': 1e3 * el / n_frames, 'frames_per_s': n_frames / el,
                'Mpix_per_s': w * h * n_frames / el / 1e6, 'd2h_bytes_per_frame': int(frame_bytes),
                'gpu_launches': int(ds.launch_count() - launches_s0)}

    if rank == 0:
        value = rays / (ms_per_step * 1e-3) / 1e6
        line = {
            'metric': METRIC, 'value': value, 'unit': 'Mrays/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': desc, 'width': w, 'height': h, 'dim': dim, 'rays_per_frame': rays,
                       'ray_counts': {k: cnt_gpu[k] for k in ('primary_rays', 'shadow_rays', 'reflection_rays')},
                       'rays_counted': 'primary + shadow + reflection/transparency rays of the frame (device counters)',
                       'frame_ms': ms_per_step, 'frame_ms_e2e': e2e_ms,
                       'l2_flush_between_iterations': True, 'tree': 'reference k-d tree (exported, tests/golden)',
                       'partition': 'interleaved 32-px tile rows over %d GPU(s); every GPU stores its rows into one frame on GPU 0 over NVLink (peer stores, no gather)' % world
                                    if wl.gather != 'nccl' else 'interleaved 32-px tile rows over %d GPU(s), NCCL all-gather' % world,
                       'frames_per_s': 1e3 / ms_per_step, 'Mpix_per_s': w * h / (ms_per_step * 1e-3) / 1e6},
            'e2e': {'value': rays / (e2e_ms * 1e-3) / 1e6, 'unit': 'Mrays/s', 'ms_per_step': e2e_ms,
                    'h2d_bytes_per_step': int(4 * (dim + dim * dim)), 'd2h_bytes_per_step': int(frame_bytes),
                    'destination': 'pinned host buffer',
                    # the same call into a plain bytearray (pageable): pinned staging ring inside ntr_render
                    'pageable_ms_per_step': wl.pageable_ms,
                    'pageable_value': rays / (wl.pageable_ms * 1e-3) / 1e6 if wl.pageable_ms else None},
            'gpu_launches': int(launches),
            'clocks': clocks,
        }
        if secondary:
            line['secondary'] = secondary
        # The headline numbers are complete here.  The legs below (roofline counts, CPU baseline, interactive loop) run
        # under a watchdog: if one of them hangs -- the reference's renderer has a refcount race that can corrupt its
        # heap (oracle/ref_bridge.make_immortal) -- the line is printed without it instead of never.
        emitted = threading.Lock()

        def emit(note=None):
            if not emitted.acquire(blocking=False):
                return
            if note:
                line['incomplete'] = note
            print(json.dumps(line), flush=True)

        def watchdog():
            emit('a post-measurement leg did not finish within %d s; keys present are valid' % TAIL_TIMEOUT_S)
            os._exit(0)

        wd = threading.Timer(TAIL_TIMEOUT_S, watchdog)
        wd.daemon = True
        wd.start()
        if world == 1:
            # ---- roofline of the dominant kernel (render_pass_kernel: >= 99 % of the step, profiles/*_launches*) ----
            from tests import oracle_lib as ol
            counts_from = 'counting CPU restatement of the reference algorithm (oracle) on the same tree, same frame'
            kernel_counts = None
            if int(sc['kind']) == 1 and int(sc['simplex'].shape[0]) > 20000:
                # The scalar restatement is far too slow for a whole frame at this size: it traces a SAMPLE of the frame -- the
                # same view at 1/32 linear size, i.e. every 32nd pixel in x and y -- and its counts are scaled by the pixel
                # ratio.  (The reference algorithm with its exact mailbox; the kernels' own counts, from the instrumented
                # build, are reported beside it: their tag mailbox is lossy, so they test more.)
                sw, sh = max(w // 32, 16), max(h // 32, 9)
                _, cnt_s = ol.render_float(sc, sw, sh, with_counters=True)
                scale = (w * h) / float(sw * sh)
                cnt_ref = {k: (int(round(v * scale)) if k != 'primary_rays' else w * h) for k, v in cnt_s.items()}
                counts_from = ('counting CPU restatement of the reference algorithm (oracle) on the same tree, on a sample of the '
                               'frame: the same view at %dx%d (every 32nd pixel in x and y), counts scaled by %.1f' % (sw, sh, scale))
                ds.set_instrumented(True)
                ds.render_float(w, h)
                kernel_counts = ds.counters()
                ds.set_instrumented(False)
            else:
                _, mask, cnt_ref = ol.render_float(sc, w, h, with_mask=True, with_counters=True)     # reference-algorithm counts
                # share of the pixels on which the reference itself is defined (its mailbox / hit lists stay inside
                # their preallocation, tracer.hpp:670-680) and not decided by rounding noise (Q12): where parity is claimed
                line['config']['defined_pixel_fraction'] = float(np.mean(mask == 0))
            flops = flops_per_frame(dim, cnt_ref, n_lights)
            fp32_peak = measure_fp32_peak(local_rank)
            achieved = flops / (ms_per_step * 1e-3) / 1e12
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
            except Exception:
                pass
            hbm_peak = peaks.get('hbm_gbs', 6650.0)
            abytes = bytes_per_frame(dim, cnt_ref, frame_bytes)
            kern = kernel_name(sc, dim)
            traffic = measured_traffic(args.config, kern)
            line['roofline'] = {
                'bound': 'fp32', 'achieved': achieved, 'peak': fp32_peak, 'unit': 'TFLOP/s', 'frac': achieved / fp32_peak,
                'traffic': traffic['bytes_per_launch'] if traffic else None,
                'traffic_source': traffic['source'] if traffic else None,
                'peak_source': 'FP32 FMA micro-benchmark measured live in this run (ntr_measure_fp32_peak); MEASURED_PEAKS.json has HBM/BF16 only',
                'algorithmic_flops_per_launch': flops, 'kernel': kern, 'kernel_ms': ms_per_step,
                'launches_per_step': launches / (2.0 * args.steps),
                'reference_algorithm_counts': cnt_ref, 'counts_from': counts_from,
                **({'kernel_counts': kernel_counts} if kernel_counts else {}),
                'hbm': {'achieved': abytes / (ms_per_step * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                        'frac': abytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak,
                        'peak_source': 'MEASURED_PEAKS.json' if peaks else 'fallback',
                        'algorithmic_bytes_per_launch': abytes,
                        'note': 'working set (nodes+refs+simplexes, a few MB) is L2/L1-resident; DRAM traffic is the frame, the accumulators and the ray queues'},
            }
            if not args.no_cpu_baseline:
                line['cpu_baseline'] = reference_arm_subprocess(args)
            # single-pass scenes only: frames with wavefront passes are traced synchronously inside ntr_render_begin, so
            # the loop adds nothing over `e2e` there
            if args.stream_frames >= 2 and cnt_gpu['reflection_rays'] == 0:
                line['stream'] = stream_leg()
        wd.cancel()
        emit()
    wl.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
