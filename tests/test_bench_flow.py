"""bench.py's control flow on a box without a GPU: the CUDA library, torch.cuda and the renderers are replaced by
stubs with the same interface (no pixels are produced, timings are fake), everything else runs for real -- argument
handling, the JSON contract of the line, the roofline bookkeeping with the oracle's counters, the reference arm in a
process of its own, the rotating-camera leg and the watchdog that prints the line when a late leg hangs."""
import io
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
            'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline']

STUB = r'''
import sys, types, time, json
import numpy as np
sys.path.insert(0, %(root)r)
import torch

class _Ev:
    def __init__(self, enable_timing=False): self.t = 0.0
    def record(self, stream=None): self.t = time.perf_counter()
    def synchronize(self): pass
    def elapsed_time(self, other): return max((other.t - self.t) * 1e3, 1e-3)
class _Stream:
    cuda_stream = 1
    def __init__(self, device=None): pass
    def synchronize(self): pass
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda *a: None
torch.cuda.Event = _Ev
torch.cuda.Stream = _Stream
torch.cuda.current_device = lambda: 0
_real_empty, _real_tensor = torch.empty, torch.tensor
torch.empty = lambda *a, **k: _real_empty(*a, **{kk: vv for kk, vv in k.items() if kk != 'device'})
torch.tensor = lambda *a, **k: _real_tensor(*a, **{kk: vv for kk, vv in k.items() if kk != 'device'})
torch.Tensor.pin_memory = lambda self: self

from ntracer_b200 import backend, dist as ntd
def _fill(buf):                                      # a fixed pattern of bytes stands in for the frame
    b = np.frombuffer(buf, np.uint8)
    b[:] = np.arange(b.size) %% 251
class FakeScene:
    def __init__(self, sc, device=-1): self.sc, self.n, self.open = sc, 0, {}
    def render_float(self, w, h): self.w, self.h = w, h; return np.zeros((h, w, 3), np.float32)
    def counters(self):
        return {'primary_rays': self.w * self.h, 'reflection_rays': %(refl)d, 'shadow_rays': 1000, 'node_steps': 5,
                'simplex_tests': 7, 'solid_tests': 0, 'shaded_hits': 3, 'queue_overflows': 0}
    def set_camera(self, o, a): pass
    def set_instrumented(self, on): pass
    def render(self, fmt, dest=None): self.n += 1; _fill(dest); return dest
    def render_device(self, *a, **k): self.n += 1
    def render_begin(self, fmt, dest):
        self.n += 1
        if %(hang)d: time.sleep(3600)
        self.open[self.n] = 1; return self.n
    def render_end(self, t): del self.open[t]
    def launch_count(self): return self.n
    def close(self): pass
backend.DeviceScene = FakeScene
backend.measure_fp32_peak = lambda dev=0: 64.5
class FakeDR:
    def __init__(self, ds, fmt, group=None):
        self.ds, self.stream = ds, _Stream()
        self.frame = types.SimpleNamespace(download=lambda fmt, buf, stream=0: _fill(buf))
    def render_strip(self): self.ds.render_device()
    def render(self): self.ds.render_device()
    def gather(self): pass
    def fence(self): pass
    def frame_on_device(self): pass
    def render_to_host(self): self.ds.render_device()
    def close(self): pass
ntd.DistributedRenderer = FakeDR
ntd.PeerFrameRenderer = FakeDR
import torch.distributed as _dist
_real_init = _dist.init_process_group
_dist.init_process_group = lambda backend=None, **k: _real_init('gloo')      # NCCL needs GPUs; the flow is the same
import bench
sys.argv = ['bench.py'] + %(argv)r
sys.exit(bench.main())
'''


def run_stubbed(argv, refl=0, hang=0, env=None, timeout=300):
    code = STUB % {'root': ROOT, 'refl': refl, 'hang': hang, 'argv': argv}
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=timeout, env=e, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, (out.stdout[-2000:], out.stderr[-2000:])
    return json.loads(lines[0]), out


def test_bench_line_has_every_contract_key_and_the_optional_legs():
    line, out = run_stubbed(['--config', 'c1', '--steps', '3', '--warmup', '1', '--stream-frames', '12'])
    for k in REQUIRED:
        assert k in line, k
    assert line['warmup'] >= 3 and line['steps'] == 3 and line['n_gpus'] == 1
    baseline = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    assert line['metric'] == baseline['metric'] and line['unit'] == 'Mrays/s'                # BASELINE.json's metric, verbatim
    assert line['config']['frame_ms'] == line['ms_per_step'] and line['config']['frame_ms_e2e'] > 0
    assert line['roofline']['traffic'] is None or line['roofline']['traffic_source']       # measured (ncu) or null, never a literal
    assert line['e2e']['d2h_bytes_per_step'] == 640 * 480 * 3 and line['e2e']['value'] > 0
    assert line['roofline']['bound'] == 'fp32' and line['roofline']['peak'] == 64.5
    assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['cores'] >= 1
    if line['cpu_baseline']['value'] is not None:
        assert line['cpu_baseline']['value'] > 0
    assert line['stream']['frames'] == 12 and line['stream']['in_flight'] == 2
    assert 'incomplete' not in line
    assert line['gpu_launches'] == 2 * 3


def test_default_workload_is_the_4k_frame_with_the_secondary_workloads_beside_it():
    """No --config: the frame BASELINE.json's metric is quoted on (configs[3], 3840x2160), {5/2,5,3} and config 2 beside it."""
    line, out = run_stubbed(['--steps', '2', '--warmup', '1', '--no-cpu-baseline', '--stream-frames', '0'], refl=500, timeout=900)
    assert line['config']['width'] == 3840 and line['config']['height'] == 2160 and '{5/2,3,3}' in line['config']['workload']
    assert set(line['secondary']) == {'c4b', 'c2'}
    assert '{5/2,5,3}' in line['secondary']['c4b']['workload'] and line['secondary']['c2']['width'] == 1920
    for v in line['secondary'].values():
        assert v['value'] > 0 and v['e2e_value'] > 0 and v['ms_per_step'] > 0
    assert 0.3 < line['config']['defined_pixel_fraction'] < 0.7          # {5/2,3,3}: about half the frame (DESIGN.md section 5)
    assert line['roofline']['kernel'].startswith('render_pass_kernel<4,1> (primary pass) + render_pass_kernel<4,5>')


def test_stream_leg_is_skipped_for_scenes_with_wavefront_passes():
    line, out = run_stubbed(['--config', 'c1', '--steps', '3', '--no-cpu-baseline'], refl=500)
    assert 'stream' not in line and 'cpu_baseline' not in line and 'roofline' in line


def test_watchdog_prints_the_line_when_a_late_leg_hangs():
    line, out = run_stubbed(['--config', 'c1', '--steps', '3', '--no-cpu-baseline'], hang=1,
                            env={'NTR_BENCH_TAIL_TIMEOUT': '5'}, timeout=120)
    assert 'incomplete' in line and 'stream' not in line
    for k in ('value', 'e2e', 'roofline', 'clocks', 'gpu_launches'):
        assert k in line
    assert out.returncode == 0


def test_dump_outputs_writes_the_frames_of_the_last_timed_steps(tmp_path):
    line, out = run_stubbed(['--config', 'c1', '--steps', '2', '--no-cpu-baseline', '--stream-frames', '0',
                             '--dump-outputs', str(tmp_path / 'out')])
    assert line['steps'] == 2 and line['gpu_launches'] == 2 * 2
    w, h = 640, 480
    want = (np.arange(h * w * 3) % 251).reshape(h, w, 3).astype(np.float32)
    assert sorted(os.listdir(tmp_path / 'out')) == ['c1_frame.npy', 'c1_frame_e2e.npy']
    for name in ('c1_frame', 'c1_frame_e2e'):
        got = np.load(tmp_path / 'out' / (name + '.npy'))
        assert got.dtype == np.float32 and np.array_equal(got, want), name


def test_dump_outputs_samples_big_frames_the_same_pixels_every_time(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    big = np.random.default_rng(0).integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path / 'a'), {'big': big, 'small': big[:90, :160]})
    bench.dump_outputs(str(tmp_path / 'b'), {'big': big})
    a = np.load(tmp_path / 'a' / 'big.npy')
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLE_PIXELS, 3)
    assert np.array_equal(a, np.load(tmp_path / 'b' / 'big.npy'))
    assert np.array_equal(np.load(tmp_path / 'a' / 'small.npy'), big[:90, :160].astype(np.float32))
    # the default workload dumps six 4K-sized frames (c4, c4b, c2; device and e2e path each)
    assert 6 * os.path.getsize(tmp_path / 'a' / 'big.npy') <= 64e6


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--config', 'c1', '--steps', '3'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['impl'] == 'reference' and line['value'] > 0 and line['e2e']['value'] == line['value']
    assert line['cpu_baseline']['kind'] in ('reference', 'port')
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0


def test_two_rank_flow_prints_one_line_from_rank_0(tmp_path):
    """The launcher the driver uses for N > 1 (torch.distributed.run, one process per GPU), with gloo standing in for
    NCCL: both ranks run the timed regions, the maxima are reduced, rank 0 alone prints the line, nobody hangs."""
    script = tmp_path / 'stub_bench.py'
    script.write_text(STUB % {'root': ROOT, 'refl': 0, 'hang': 0,
                              'argv': ['--gpus', '2', '--config', 'c1', '--steps', '3', '--warmup', '1']})
    import socket
    with socket.socket() as sock:                      # a free rendezvous port
        sock.bind(('127.0.0.1', 0))
        port = sock.getsockname()[1]
    env = dict(os.environ, MASTER_ADDR='127.0.0.1')
    out = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                          '--master-addr', '127.0.0.1', '--master-port', str(port), str(script)],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert out.returncode == 0 and len(lines) == 1, (out.stdout[-1500:], out.stderr[-1500:])
    line = json.loads(lines[0])
    assert line['n_gpus'] == 2 and line['scaling'] == 'strong' and line['value'] > 0 and line['e2e']['value'] > 0
    assert 'roofline' not in line and 'cpu_baseline' not in line and 'stream' not in line     # N = 1 only
