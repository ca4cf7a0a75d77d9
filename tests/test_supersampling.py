"""Supersampled anti-aliasing (ntr_scene_set_supersampling / Scene.set_supersampling): output pixel (x, y) of a frame with
factor s is the box-filtered mean of pixels (s*x + i, s*y + j) of the s-times-larger view, summed j-major, i-minor.

CPU tier: the host-emulated device code (tests/emul_ss_lib.py: the frame driver runs trace_core.cuh's ss_pixel_color,
the code the NTR_F_SS kernels inline) against the oracle's big view, box-filtered here; and the Python surface on a test
double of the device.  GPU tier (`-m gpu`): the CUDA library, every render path, against its own 1-spp big view and the
oracle."""
import ctypes as C
import pickle
import threading

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_lib as el
from tests import emul_ss_lib as ess
from tests import fixtures as fx
from tests import oracle_lib as ol

FACTORS_CPU = (2, 3)


def box_sum(big, s):
    """float32 sequential sum of every s x s block, j-major, i-minor, times 1/s^2: the contract's reference."""
    h, w = big.shape[0] // s, big.shape[1] // s
    acc = np.zeros((h, w) + big.shape[2:], np.float32)
    for j in range(s):
        for i in range(s):
            acc = acc + big[j::s, i::s][:h, :w]
    return acc * np.float32(1.0 / (s * s))


def block_or(mask, s):
    """oracle mask of an output pixel: the OR over its s x s block of the big view"""
    h, w = mask.shape[0] // s, mask.shape[1] // s
    out = np.zeros((h, w), mask.dtype)
    for j in range(s):
        for i in range(s):
            out |= mask[j::s, i::s][:h, :w]
    return out


def oracle_ss(sc, w, h, s, with_counters=False):
    """the oracle's s-times-larger view, box-filtered, its mask OR-ed over the blocks"""
    big, mask, cnt = ol.render_float(sc, s * w, s * h, with_mask=True, with_counters=True)
    out = (box_sum(big, s), block_or(mask, s))
    return out + (cnt,) if with_counters else out


def scene_cases():
    cases = [('box4', None), ('solids6', None), ('mixed3', None)]
    _, g = fx.load('cell120')
    cases += [('cell120', str(v)) for v in g['variants']]
    return cases


def load_case(name, v):
    sc, g = fx.load(name)
    return fx.variant(sc, g, v) if v else sc


def pass_free(sc):
    """the scene without its reflections: no wavefront passes"""
    p = np.array(sc['params'], np.float64)
    p[3] = 0
    return dict(sc, params=p)


# ---------------------------------------------------------------- CPU tier: emulated device code ------------------
@pytest.mark.parametrize('name,v', scene_cases())
def test_emulated_frame_matches_the_box_filtered_oracle(name, v):
    sc = load_case(name, v)
    w, h = 64, 36
    col = fx.center_column_mask(w, h)
    for s in FACTORS_CPU:
        img, cnt = ess.render_ss(sc, w, h, s)
        ref, mask, ocnt = oracle_ss(sc, w, h, s, with_counters=True)
        bad, _ = fx.lsb_stats(img, ref, exclude=col | (mask != 0))
        assert bad <= 0.001, (name, v, s, bad)
        assert cnt['primary_rays'] == s * s * w * h
        for k in ('reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert cnt[k] == ocnt[k], (name, v, s, k)


@pytest.mark.parametrize('name,v', [('box4', None), ('box9', None), ('cell120', 'shadows'), ('cell120', 'transp'),
                                    ('solids6', None), ('soup9', None)])
def test_emulated_pass_free_frames_are_the_exact_box_sum(name, v):
    """Scaling by a power of two is exact: without wavefront passes the supersampled frame IS the box sum of the big view."""
    sc = pass_free(load_case(name, v)) if fx.load(name)[0]['kind'] == 1 else load_case(name, v)
    w, h = 48, 30
    for s in (2, 4):
        img, cnt = ess.render_ss(sc, w, h, s)
        big, bcnt = el.render(sc, s * w, s * h)
        assert bcnt['reflection_rays'] == 0
        assert np.array_equal(img, box_sum(big, s)), (name, v, s)
        assert cnt['shadow_rays'] == bcnt['shadow_rays'] and cnt['primary_rays'] == bcnt['primary_rays']
    img, _ = ess.render_ss(sc, w, h, 3)
    np.testing.assert_allclose(img, box_sum(el.render(sc, 3 * w, 3 * h)[0], 3), rtol=1e-6, atol=1e-7)


def test_emulated_factor_is_range_checked_and_generic_family_agrees():
    sc, _ = fx.load('cell120')
    for bad in (0, 9):
        with pytest.raises(ValueError):
            ess.render_ss(sc, 8, 4, bad)
    a, _ = ess.render_ss(sc, 32, 18, 2)
    b, _ = ess.render_ss(sc, 32, 18, 2, generic=True)
    assert np.abs(a - b).max() <= 2e-6


# ---------------------------------------------------------------- CPU tier: the Python surface -------------------
class _SSLibrary:
    def __init__(self, dev):
        self.dev = dev

    def ntr_render(self, handle, fmt_ref, ptr, size):
        fmt = fmt_ref._obj
        rgb = self.dev.render_float(fmt.width, fmt.height)
        packed = ol.pack(fmt, rgb)
        addr = ptr.value if hasattr(ptr, 'value') else ptr
        row_bytes = fmt.width * fmt.bytes_per_pixel
        for y in range(fmt.height):
            C.memmove(addr + y * fmt.pitch, packed[y * fmt.pitch:].ctypes.data, row_bytes)
        return 0


def _emulated_device_class():
    from tests.test_facade_emulated import _EmulatedFullDevice

    class _EmulatedSSDevice(_EmulatedFullDevice):
        """the test double of tests/test_facade_emulated.py plus the supersampling factor"""
        def __init__(self, sc, device=-1):
            super().__init__(sc, device)
            self._lib = _SSLibrary(self)
            self.supersampling = 1
            self.calls = []

        def set_supersampling(self, factor):
            self.calls.append(factor)
            self.supersampling = factor

        def render_float(self, w, h):
            return ess.render_ss(self.sc, w, h, self.supersampling)[0]

        def calculate_color(self, x, y, w, h):
            return self.render_float(w, h)[y, x]

    return _EmulatedSSDevice


@pytest.fixture
def emulated(monkeypatch):
    from ntracer_b200 import tracern
    cls = _emulated_device_class()
    monkeypatch.setattr(tracern, 'DeviceScene', cls)
    return cls


def _box_scene():
    from ntracer_b200 import NTracer
    nt = NTracer(4)
    scene = nt.BoxScene()
    cam = nt.Camera()
    cam.translate(nt.Vector.axis(2, -5))
    scene.set_camera(cam)
    return nt, scene


def test_set_supersampling_validates_and_respects_the_lock():
    from ntracer_b200.render import LockedError
    nt, scene = _box_scene()
    assert scene.supersampling == 1
    for bad in (0, 9, -1):
        with pytest.raises(ValueError):
            scene.set_supersampling(bad)
    for bad in (2.5, 2.0, '2', None, True):
        with pytest.raises(TypeError):
            scene.set_supersampling(bad)
    scene.set_supersampling(np.int64(3))
    assert scene.supersampling == 3 and type(scene.supersampling) is int
    scene.locked += 1
    with pytest.raises(LockedError):
        scene.set_supersampling(2)
    scene.locked -= 1
    assert scene.supersampling == 3
    for f in range(1, 9):
        scene.set_supersampling(f)


def test_supersampling_pickles_and_old_pickles_load_with_factor_one():
    from ntracer_b200 import Material, NTracer
    nt, scene = _box_scene()
    scene.set_supersampling(4)
    back = pickle.loads(pickle.dumps(scene))
    assert back.supersampling == 4
    comp = nt.build_composite_scene([nt.TrianglePrototype([nt.Vector(1, 0, 0, 0), nt.Vector(0, 1, 0, 0), nt.Vector(0, 0, 1, 0),
                                                           nt.Vector(0, 0, 0, 1)], Material((1, 1, 1)))])
    comp.set_supersampling(2)
    assert pickle.loads(pickle.dumps(comp)).supersampling == 2
    # a scene pickled before the attribute existed: its state has no 'supersampling'
    del scene.__dict__['supersampling']
    state = pickle.dumps(scene)
    old = pickle.loads(state)
    assert 'supersampling' not in old.__dict__ and old.supersampling == 1
    assert isinstance(NTracer(4).BoxScene().supersampling, int)


def test_renderers_pass_the_factor_through(emulated):
    from ntracer_b200 import BlockingRenderer, CallbackRenderer, Channel, ImageFormat
    nt, scene = _box_scene()
    w, h = 48, 32
    fmt = ImageFormat(w, h, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)])
    flat = dict(scene._flat(), cam_origin=scene._cam._origin, cam_axes=scene._cam._axes)
    native = _capi.make_image_format(w, h, _capi.RGB8)
    plain = bytearray(w * h * 3)
    assert BlockingRenderer().render(plain, fmt, scene) is True
    assert bytes(plain) == bytes(ol.pack(native, el.render(flat, w, h)[0]))
    scene.set_supersampling(2)
    want = ol.pack(native, box_sum(el.render(flat, 2 * w, 2 * h)[0], 2))
    buf = bytearray(w * h * 3)
    assert BlockingRenderer().render(buf, fmt, scene) is True
    assert bytes(buf) == bytes(want) and bytes(buf) != bytes(plain)
    assert scene._dev.calls == [2] and scene.locked == 0
    buf2 = bytearray(w * h * 3)
    done = threading.Event()
    r = CallbackRenderer()
    r.begin_render(buf2, fmt, scene, lambda rr: done.set())
    assert done.wait(60)
    r.abort_render()
    assert bytes(buf2) == bytes(want)
    assert scene._dev.calls == [2]                      # applied once: the device keeps it until it changes
    assert list(scene.calculate_color(5, 7, w, h)) == pytest.approx(list(box_sum(el.render(flat, 2 * w, 2 * h)[0], 2)[7, 5]),
                                                                     abs=0)
    scene.set_supersampling(1)
    assert BlockingRenderer().render(buf, fmt, scene) is True
    assert bytes(buf) == bytes(plain) and scene._dev.calls == [2, 1]


# ---------------------------------------------------------------- GPU tier -----------------------------------------
def _dev(sc, s=1):
    from ntracer_b200.backend import DeviceScene
    ds = DeviceScene(sc)
    ds.set_supersampling(s)
    return ds


@pytest.mark.gpu
def test_device_rejects_bad_factors():
    from ntracer_b200.backend import DeviceScene
    sc, _ = fx.load('box4')
    with DeviceScene(sc) as ds:
        for bad in (0, 9, -3):
            with pytest.raises(ValueError):
                ds.set_supersampling(bad)
        ds.set_supersampling(8)
        assert ds.render_float(4, 3).shape == (3, 4, 3) and ds.counters()['primary_rays'] == 64 * 12


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', [('cell120', None), ('ggs120', 'refl_transp')])
def test_factor_one_changes_nothing(name, v):
    sc = load_case(name, v)
    _, g = fx.load(name)
    w, h = [int(x) for x in g['size']]
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    pts = [(0, 0), (w // 3, h // 2), (w - 1, h - 1)]
    out = []
    for touched in (False, True):
        with _dev(sc) as ds:
            if touched:
                ds.set_supersampling(2)
                ds.set_supersampling(1)
            n0 = ds.launch_count()
            img = ds.render(fmt)
            fl = ds.render_float(w, h)
            cc = [ds.calculate_color(x, y, w, h) for x, y in pts]
            out.append((img, fl, cc, ds.counters(), ds.launch_count() - n0))
    (a, fa, ca, na, la), (b, fb, cb, nb, lb) = out
    assert la == lb and na == nb                                    # the same kernels, the same rays
    if not v:
        assert np.array_equal(a, b) and np.array_equal(fa, fb)
        assert all(np.array_equal(x, y) for x, y in zip(ca, cb))
    else:
        # the bounce passes add into the frame with float atomics in no fixed order: two frames of the SAME scene may
        # differ in the last bit, so the reflective scene is held to what repeated renders guarantee
        assert np.abs(a.astype(np.int32) - b.astype(np.int32)).max() <= 1
        assert np.abs(fa - fb).max() <= 1e-6
        assert all(np.abs(x - y).max() <= 1e-6 for x, y in zip(ca, cb))


def _exact_cases():
    return [('box4', False), ('box9', False), ('cell120', False), ('soup9', False), ('soup9', True)]


@pytest.mark.gpu
@pytest.mark.parametrize('name,generic', _exact_cases())
def test_pass_free_frames_are_the_exact_box_sum(name, generic, monkeypatch):
    if generic:
        monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    sc, g = fx.load(name)
    if name == 'cell120':
        sc = fx.variant(sc, g, 'shadows')
    if int(sc['kind']) == 1:
        sc = pass_free(sc)
    w, h = 160, 96
    with _dev(sc) as plain, _dev(sc) as ss:
        for s in (2, 4, 3):
            big = plain.render_float(s * w, s * h)
            assert plain.counters()['reflection_rays'] == 0
            ss.set_supersampling(s)
            fl = ss.render_float(w, h)
            ref = box_sum(big, s)
            if s == 3:
                np.testing.assert_allclose(fl, ref, rtol=1e-6, atol=1e-7)
                continue
            assert np.array_equal(fl, ref), (name, generic, s, float(np.abs(fl - ref).max()))
            fmt = _capi.make_image_format(w, h, _capi.RGB8)
            assert np.array_equal(ss.render(fmt), ol.pack(fmt, ref)), (name, generic, s)


def _parity_cases():
    cases = []
    for name in ('cell120', 'ggs120', 'ssc120'):
        _, g = fx.load(name)
        cases += [(name, str(v)) for v in g['variants']]
    return cases + [('solids6', None), ('mixed3', None), ('soup9', None)]


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', _parity_cases())
def test_parity_with_the_box_filtered_oracle(name, v):
    """The bounds of tests/test_gpu_parity.py, on the oracle's 2x view box-filtered."""
    sc = load_case(name, v)
    _, g = fx.load(name)
    w, h = [int(x) for x in g['size']]
    s = 2
    col = fx.center_column_mask(w, h)
    with _dev(sc, s) as ds:
        img = ds.render_float(w, h)
        cnt = ds.counters()
    ref, mask, ocnt = oracle_ss(sc, w, h, s, with_counters=True)
    if name == 'mixed3':
        assert fx.lsb_stats(img, ref, exclude=mask != 0)[0] <= 0.001
        assert fx.lsb_stats(img, ref)[0] <= 0.015
    elif v is None:
        assert fx.lsb_stats(img, ref)[0] <= 0.001, name
    else:
        undefined, noise = (mask & 3) != 0, (mask & 4) != 0
        assert fx.lsb_stats(img, ref, exclude=col | noise)[0] <= 0.002, (name, v)
        assert fx.lsb_stats(img, ref, exclude=col | undefined | noise)[0] <= 0.001, (name, v)
        assert fx.lsb_stats(img, ref, exclude=col)[0] <= 0.03, (name, v)
    assert cnt['primary_rays'] == s * s * w * h
    for k in ('reflection_rays', 'shadow_rays', 'shaded_hits'):
        assert abs(cnt[k] - ocnt[k]) <= 0.01 * max(ocnt[k], 100), (name, v, k, cnt[k], ocnt[k])


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', [('cell120', 'shadows'), ('cell120', 'refl_transp'), ('ggs120', 'refl'),
                                    ('mixed3', None), ('stacked', None)])
def test_counters_are_those_of_the_big_view(name, v):
    sc = fx.stacked_layers(20) if name == 'stacked' else load_case(name, v)
    w, h = 96, 54
    with _dev(sc) as plain, _dev(sc) as ss:
        for s in (2, 3):
            plain.render_float(s * w, s * h)
            want = plain.counters()
            ss.set_supersampling(s)
            ss.render_float(w, h)
            got = ss.counters()
            assert got['primary_rays'] == s * s * w * h == want['primary_rays']
            for k in ('reflection_rays', 'shadow_rays', 'shaded_hits', 'truncated_hit_lists'):
                assert got[k] == want[k], (name, v, s, k)
    if name == 'stacked':
        assert want['truncated_hit_lists'] > 0


def _strips(ds, fmt, world, import_torch):
    torch = import_torch
    h = fmt.height
    out = np.zeros((h, fmt.pitch), np.uint8)
    for rank in range(world):
        rows = [ty for ty in range((h + 31) // 32) if ty % world == rank]
        strip = torch.zeros(len(rows) * 32 * fmt.pitch, dtype=torch.uint8, device='cuda')
        ds.render_device(fmt, strip.data_ptr(), strip.numel(), 0, rank, world, True)
        torch.cuda.synchronize()
        st = strip.cpu().numpy().reshape(len(rows) * 32, fmt.pitch)
        for k, ty in enumerate(rows):
            n = min(32, h - ty * 32)
            out[ty * 32:ty * 32 + n] = st[k * 32:k * 32 + n]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('v', ['shadows', 'refl'])
def test_every_render_path_gives_the_same_frame(v, monkeypatch):
    import torch
    from ntracer_b200.backend import DeviceGroup
    sc, g = fx.load('cell120')
    sc = fx.variant(sc, g, v)
    w, h = 320, 288                     # 9 tile rows: the slab path runs (2 slabs) and the interleaves are ragged
    s = 2
    tol = 0 if v == 'shadows' else 1    # bounce passes: float atomics in no fixed order
    fmt = _capi.make_image_format(w, h, _capi.RGB8)

    def same(a, what):
        d = np.abs(np.asarray(a, np.int32).reshape(h, fmt.pitch) - want.astype(np.int32).reshape(h, fmt.pitch)).max()
        assert d <= tol, (v, what, d)

    with _dev(sc, s) as ds:
        fl = ds.render_float(w, h)
        want = ol.pack(fmt, fl)
        same(ds.render(fmt), 'ntr_render, slabs + staging')
        pinned = torch.zeros(fmt.pitch * h, dtype=torch.uint8).pin_memory()
        same(ds.render(fmt, pinned.numpy()), 'ntr_render, pinned destination')
        dev = torch.zeros(fmt.pitch * h, dtype=torch.uint8, device='cuda')
        ds.render_device(fmt, dev.data_ptr(), dev.numel())
        torch.cuda.synchronize()
        same(dev.cpu().numpy(), 'ntr_render_device')
        for world in (2, 3):
            same(_strips(ds, fmt, world, torch), 'interleaved tile rows, compact, %d ranks' % world)
        # begin / end with the camera moved between the frames: each frame is the blocking render at its camera
        cam0 = (np.array(sc['cam_origin'], np.float32), np.array(sc['cam_axes'], np.float32))
        cam1 = (cam0[0] + np.float32(0.07), cam0[1])
        bufs = [bytearray(fmt.pitch * h) for _ in range(2)]
        t0 = ds.render_begin(fmt, bufs[0])
        ds.set_camera(*cam1)
        t1 = ds.render_begin(fmt, bufs[1])
        ds.render_end(t0)
        ds.render_end(t1)
        same(np.frombuffer(bufs[0], np.uint8), 'render_begin/end, first camera')
        moved = ds.render(fmt)
        d = np.abs(np.frombuffer(bufs[1], np.uint8).astype(np.int32) - moved.astype(np.int32)).max()
        assert d <= tol and not np.array_equal(moved, want)
        ds.set_camera(*cam0)
    for env in ('NTR_NO_SLABS', 'NTR_NO_STAGING'):
        monkeypatch.setenv(env, '1')
        with _dev(sc, s) as ds:
            same(ds.render(fmt), env)
        monkeypatch.delenv(env)
    # a group listing the same device twice (the ABI allows it): two ranks of interleaved tile rows on one GPU
    with DeviceGroup(sc, devices=[0, 0]) as grp:
        grp.set_supersampling(s)
        same(grp.render(fmt), 'ntr_group_render')
        c = grp.counters()
        assert c['primary_rays'] == s * s * w * h


@pytest.mark.gpu
def test_stream_renderer_frames_match_blocking_renders():
    from ntracer_b200 import BlockingRenderer, Channel, ImageFormat, StreamRenderer
    nt, scene = _box_scene()
    scene.set_supersampling(2)
    w, h = 200, 120
    fmt = ImageFormat(w, h, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)])
    cams = []
    for k in range(3):
        cam = nt.Camera()
        cam.translate(nt.Vector.axis(2, -5 + 0.3 * k))
        cams.append(cam)
    r = StreamRenderer()
    bufs = [bytearray(w * h * 3) for _ in cams]
    tickets = []
    for cam, buf in zip(cams, bufs):
        scene.set_camera(cam)
        tickets.append(r.submit(buf, fmt, scene))
        if len(tickets) == 2:
            assert r.wait(tickets[0])
    assert r.wait(tickets[1]) and r.wait(tickets[2])
    for cam, buf in zip(cams, bufs):
        scene.set_camera(cam)
        ref = bytearray(w * h * 3)
        assert BlockingRenderer().render(ref, fmt, scene)
        assert bytes(ref) == bytes(buf)
    assert len(set(bytes(b) for b in bufs)) == 3


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', [('cell120', 'shadows'), ('ggs120', 'refl')])
def test_calculate_color_and_hit_ids(name, v):
    sc = load_case(name, v)
    w, h = 128, 72
    tol = 0 if v == 'shadows' else 1e-6
    with _dev(sc) as plain:
        ids0, d0 = plain.primary_hit_ids(w, h)
    with _dev(sc, 2) as ds:
        fl = ds.render_float(w, h)
        rng = np.random.RandomState(5)
        for _ in range(8):
            x, y = int(rng.randint(w)), int(rng.randint(h))
            assert np.abs(ds.calculate_color(x, y, w, h) - fl[y, x]).max() <= tol, (x, y)
        ids, d = ds.primary_hit_ids(w, h)
        assert np.array_equal(ids, ids0) and np.array_equal(d, d0)
        assert ds.counters()['primary_rays'] == w * h


@pytest.mark.gpu
def test_abort_of_a_supersampled_frame(monkeypatch):
    """Following tests/test_gpu_parity.py's abort test: a 960x540 frame at factor 4 traces the rays of a 4K frame."""
    import time
    from ntracer_b200 import bulk
    monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    pts = bulk.soup(10, 60000)
    sc = bulk.simplex_scene(pts, max_depth=14)
    sc['cam_origin'] = np.array([0, 0, -3] + [0] * 7, np.float32)
    with _dev(sc, 4) as ds:
        fmt = _capi.make_image_format(960, 540, _capi.RGB8)
        t0 = time.perf_counter()
        ds.render(fmt)
        full = time.perf_counter() - t0
        result = {}

        def run():
            try:
                ds.render(fmt)
                result['rc'] = 'finished'
            except RuntimeError as e:
                result['rc'] = str(e)

        th = threading.Thread(target=run)
        t0 = time.perf_counter()
        th.start()
        time.sleep(min(0.05, full / 10))
        ds.abort()
        th.join()
        aborted = time.perf_counter() - t0
        if full > 0.3:
            assert result['rc'] == 'render aborted'
            assert aborted < 0.8 * full
        assert ds.render(fmt).size == fmt.pitch * 540


@pytest.mark.gpu
def test_forced_queue_regrow_of_a_supersampled_frame(monkeypatch):
    sc, g = fx.load('cell120')
    sc = fx.variant(sc, g, 'refl_transp')
    w, h = 160, 90
    with _dev(sc, 2) as ds:
        ref = ds.render_float(w, h)
        assert ds.counters()['queue_overflows'] == 0
    monkeypatch.setenv('NTR_QUEUE_INIT', '512')
    with _dev(sc, 2) as ds:
        img = ds.render_float(w, h)
        assert ds.counters()['queue_overflows'] >= 1
        assert np.abs(img - ref).max() <= 1e-5
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        assert np.abs(ds.render(fmt).astype(np.int32) - ol.pack(fmt, ref).astype(np.int32)).max() <= 1
