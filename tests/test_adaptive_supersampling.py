"""Adaptive supersampling (ntr_scene_set_supersampling_threshold / Scene.set_supersampling(s, threshold)): with a factor
s > 1 and a threshold t, pixel (x, y) is refined -- gets the s x s samples of full supersampling -- iff, in some channel,
the plain 1-spp colours of {(x, y), (x+1, y), (x, y+1), (x+1, y+1)} intersected with the view span more than t; every
other pixel keeps its plain colour.

CPU tier: the host build of the device's refine rule and accumulator-slot layout (tests/emul_aa_lib.py) against the numpy
statement below, and the Python surface on a test double.  GPU tier (`-m gpu`): the CUDA library on every render path,
against its own plain and fully supersampled frames."""
import math
import pickle
import threading

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_aa_lib as eaa
from tests import emul_lib as el
from tests import emul_ss_lib as ess
from tests import fixtures as fx
from tests import oracle_lib as ol

THRESHOLDS = (0.0, 1 / 255, 4 / 255, 16 / 255)


def rule(rgb, t):
    """The contract's mask over a whole plain frame (h, w, 3): corner sets clipped to the view, float32 max - min > t."""
    rgb = np.asarray(rgb, np.float32)
    h, w = rgb.shape[:2]
    lo, hi = rgb.copy(), rgb.copy()
    for dy, dx in ((0, 1), (1, 0), (1, 1)):
        nb = rgb[dy:, dx:]
        lo[:h - dy, :w - dx] = np.minimum(lo[:h - dy, :w - dx], nb)
        hi[:h - dy, :w - dx] = np.maximum(hi[:h - dy, :w - dx], nb)
    return ((hi - lo) > np.float32(t)).any(axis=2).astype(np.uint8)


def compose(plain, full, mask):
    return np.where(mask[..., None] != 0, full, plain)


def owned_rows(h, trf, trs):
    return np.array([(y // 32) % trs == trf for y in range(h)])


def load_case(name, v=None):
    sc, g = fx.load(name)
    return fx.variant(sc, g, v) if v else sc


def pass_free(sc):
    p = np.array(sc['params'], np.float64)
    p[3] = 0
    return dict(sc, params=p)


# ---------------------------------------------------------------- CPU tier: the host build of the rule ----------------
def _frames():
    out = []
    for name, v in (('cell120', 'shadows'), ('ggs120', 'refl_transp'), ('box4', None)):
        sc = load_case(name, v)
        out.append((name, ol.render_float(sc, 72, 70)))
    rng = np.random.RandomState(3)
    out.append(('quantised noise', (rng.randint(0, 6, (70, 72, 3)) / np.float32(255)).astype(np.float32)))
    return out


@pytest.fixture(scope='module')
def frames():
    return _frames()


def test_host_rule_on_whole_frames_matches_numpy(frames):
    for name, rgb in frames:
        for t in THRESHOLDS:
            mask, halo = eaa.refine_mask(rgb, t)
            assert halo == 0
            assert np.array_equal(mask, rule(rgb, t)), (name, t)
        # 1 x N, N x 1 and 1 x 1 views
        for view in (rgb[:1], rgb[:, :1], rgb[:1, :1], rgb[:2, :1]):
            view = np.ascontiguousarray(view)
            for t in THRESHOLDS:
                assert np.array_equal(eaa.refine_mask(view, t)[0], rule(view, t)), (name, view.shape, t)


def test_host_rule_on_interleaved_and_compact_launches(frames):
    for name, rgb in frames:
        h, w = rgb.shape[:2]
        for t in THRESHOLDS:
            want = rule(rgb, t)
            for trs in (2, 3):
                for trf in range(trs):
                    own = owned_rows(h, trf, trs)
                    for compact in (False, True):
                        mask, halo = eaa.refine_mask(rgb, t, trf=trf, trs=trs, compact=compact)
                        assert np.array_equal(mask[own], want[own]), (name, t, trf, trs, compact)
                        assert not mask[~own].any()
                        # the row below every owned tile row that ends inside the view
                        assert halo == w * sum(1 for ty in range(trf, (h + 31) // 32, trs) if (ty + 1) * 32 < h)


def test_host_rule_on_windows_inside_and_at_the_view_border(frames):
    for name, rgb in frames:
        h, w = rgb.shape[:2]
        for t in THRESHOLDS:
            want = rule(rgb, t)
            # the 1 x 1 windows of calculate_color: interior, right edge, bottom edge, the corner, the origin
            for x, y in ((30, 20), (w - 1, 20), (30, h - 1), (w - 1, h - 1), (0, 0)):
                mask, halo = eaa.refine_mask(rgb, t, window=(x, y, 1, 1))
                assert mask[0, 0] == want[y, x], (name, t, x, y)
                assert halo == (x + 1 < w) + (y + 1 < h) + (x + 1 < w and y + 1 < h)
            for win in ((5, 7, 40, 33), (32, 36, w - 32, h - 36), (0, 0, w - 1, h), (3, 0, 1, h), (0, 4, w, 1)):
                x0, y0, ww, wh = win
                for trf, trs, compact in ((0, 1, False), (1, 2, False), (0, 2, True)):
                    mask, _ = eaa.refine_mask(rgb, t, window=win, trf=trf, trs=trs, compact=compact)
                    own = owned_rows(wh, trf, trs)
                    assert np.array_equal(mask[own], want[y0:y0 + wh, x0:x0 + ww][own]), (name, t, win, trf, trs, compact)


# ---------------------------------------------------------------- CPU tier: the Python surface -------------------
def _box_scene():
    from ntracer_b200 import NTracer
    nt = NTracer(4)
    scene = nt.BoxScene()
    cam = nt.Camera()
    cam.translate(nt.Vector.axis(2, -5))
    scene.set_camera(cam)
    return nt, scene


def test_set_supersampling_threshold_validates_and_respects_the_lock():
    from ntracer_b200.render import LockedError
    nt, scene = _box_scene()
    assert scene.supersampling_threshold is None
    for bad in ('0.1', True, [0.1], 1j):
        with pytest.raises(TypeError):
            scene.set_supersampling(2, bad)
    for bad in (-0.001, -1, math.nan, math.inf, -math.inf):
        with pytest.raises(ValueError):
            scene.set_supersampling(2, bad)
    assert scene.supersampling == 1 and scene.supersampling_threshold is None       # a rejected call changes nothing
    scene.set_supersampling(4, np.float32(0.25))
    assert scene.supersampling == 4 and scene.supersampling_threshold == 0.25 and type(scene.supersampling_threshold) is float
    scene.set_supersampling(2, 0)
    assert scene.supersampling_threshold == 0.0
    scene.locked += 1
    with pytest.raises(LockedError):
        scene.set_supersampling(2, 0.5)
    scene.locked -= 1
    assert scene.supersampling_threshold == 0.0
    scene.set_supersampling(2)
    assert scene.supersampling_threshold is None


def test_threshold_pickles_and_scenes_without_one_pickle_as_before():
    nt, scene = _box_scene()
    scene.set_supersampling(3)
    before = pickle.dumps(scene)
    assert b'supersampling_threshold' not in before
    scene.set_supersampling(3, 4 / 255)
    back = pickle.loads(pickle.dumps(scene))
    assert back.supersampling == 3 and back.supersampling_threshold == 4 / 255
    scene.set_supersampling(3)
    assert pickle.dumps(scene) == before
    # a scene pickled before the attribute existed loads with the threshold off
    old = pickle.loads(before)
    assert 'supersampling_threshold' not in old.__dict__ and old.supersampling_threshold is None


def _adaptive_device_class():
    from tests.test_supersampling import _emulated_device_class
    base = _emulated_device_class()

    class _EmulatedAdaptiveDevice(base):
        """the supersampling test double plus the threshold: the frame is composed from the emulated plain and full frames"""
        def __init__(self, sc, device=-1):
            super().__init__(sc, device)
            self.supersampling_threshold = None
            self.threshold_calls = []

        def set_supersampling_threshold(self, t):
            self.threshold_calls.append(t)
            self.supersampling_threshold = t

        def render_float(self, w, h):
            full = super().render_float(w, h)
            if self.supersampling_threshold is None or self.supersampling == 1:
                return full
            plain = el.render(self.sc, w, h)[0]
            return compose(plain, full, rule(plain, self.supersampling_threshold))

    return _EmulatedAdaptiveDevice


def test_renderers_pass_the_threshold_through(monkeypatch):
    from ntracer_b200 import BlockingRenderer, CallbackRenderer, Channel, ImageFormat, tracern
    cls = _adaptive_device_class()
    monkeypatch.setattr(tracern, 'DeviceScene', cls)
    nt, scene = _box_scene()
    w, h = 48, 32
    fmt = ImageFormat(w, h, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)])
    flat = dict(scene._flat(), cam_origin=scene._cam._origin, cam_axes=scene._cam._axes)
    native = _capi.make_image_format(w, h, _capi.RGB8)
    plain = el.render(flat, w, h)[0]
    full = ess.render_ss(flat, w, h, 2)[0]
    t = 4 / 255
    m = rule(plain, t)
    assert 0 < m.sum() < m.size
    want = ol.pack(native, compose(plain, full, m))
    scene.set_supersampling(2, t)
    buf = bytearray(w * h * 3)
    assert BlockingRenderer().render(buf, fmt, scene) is True
    assert bytes(buf) == bytes(want) and bytes(buf) != bytes(ol.pack(native, full))
    assert scene._dev.threshold_calls == [t] and scene.locked == 0
    buf2 = bytearray(w * h * 3)
    done = threading.Event()
    r = CallbackRenderer()
    r.begin_render(buf2, fmt, scene, lambda rr: done.set())
    assert done.wait(60)
    r.abort_render()
    assert bytes(buf2) == bytes(want)
    assert scene._dev.threshold_calls == [t]            # applied once: the device keeps it until it changes
    scene.set_supersampling(2)
    assert BlockingRenderer().render(buf, fmt, scene) is True
    assert bytes(buf) == bytes(ol.pack(native, full)) and scene._dev.threshold_calls == [t, None]


# ---------------------------------------------------------------- GPU tier -----------------------------------------
def _dev(sc, s=1, t=None):
    from ntracer_b200.backend import DeviceScene
    ds = DeviceScene(sc)
    ds.set_supersampling(s)
    ds.set_supersampling_threshold(t)
    return ds


def _reference(sc, w, h, s, generic=False):
    """(plain, full) float frames of the device at factors 1 and s"""
    with _dev(sc) as ds:
        plain = ds.render_float(w, h)
        ds.set_supersampling(s)
        full = ds.render_float(w, h)
    return plain, full


@pytest.mark.gpu
def test_device_rejects_bad_thresholds():
    sc = load_case('box4')
    with _dev(sc, 2) as ds:
        for bad in (math.nan, math.inf):
            with pytest.raises(ValueError):
                ds.set_supersampling_threshold(bad)
        for off in (-1.0, -math.inf, None):
            ds.set_supersampling_threshold(off)
        ds.render_float(8, 4)
        mask, n = ds.refine_mask()
        assert mask.shape == (4, 8) and not mask.any() and n == 0


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', [('cell120', 'shadows'), ('ggs120', 'refl_transp')])
def test_off_and_factor_one_change_nothing(name, v):
    sc = load_case(name, v)
    w, h = 160, 96
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    tol = 0 if v == 'shadows' else 1
    for s in (1, 2):
        out = []
        for t in (None, 'set-then-off' if s > 1 else 4 / 255):
            with _dev(sc, s) as ds:
                if t == 'set-then-off':
                    ds.set_supersampling_threshold(4 / 255)
                    ds.set_supersampling_threshold(None)
                elif t is not None:
                    ds.set_supersampling_threshold(t)
                n0 = ds.launch_count()
                img = ds.render(fmt)
                fl = ds.render_float(w, h)
                cc = ds.calculate_color(w // 3, h // 2, w, h)
                out.append((img, fl, cc, ds.counters(), ds.launch_count() - n0))
        (a, fa, ca, na, la), (b, fb, cb, nb, lb) = out
        assert la == lb and na == nb, (name, s)
        assert np.abs(a.astype(np.int32) - b.astype(np.int32)).max() <= tol
        if tol == 0:
            assert np.array_equal(fa, fb) and np.array_equal(ca, cb)


@pytest.mark.gpu
@pytest.mark.parametrize('name,generic', [('box4', False), ('box9', False), ('cell120', False), ('soup9', False),
                                          ('soup9', True)])
def test_pass_free_frames_are_exact(name, generic, monkeypatch):
    if generic:
        monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    sc = load_case(name, 'shadows' if name == 'cell120' else None)
    if int(sc['kind']) == 1:
        sc = pass_free(sc)
    w, h = 160, 96
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    for s in (2, 3, 4):
        plain, full = _reference(sc, w, h, s)
        for t in (0.0, 4 / 255, 16 / 255):
            m = rule(plain, t)
            with _dev(sc, s, t) as ds:
                fl = ds.render_float(w, h)
                mask, n = ds.refine_mask()
                assert np.array_equal(mask, m), (name, s, t, int(np.sum(mask != m)))
                assert n == int(m.sum())
                assert np.array_equal(fl, compose(plain, full, m)), (name, generic, s, t)
                assert ds.counters()['primary_rays'] == w * h + n * s * s
                assert np.array_equal(ds.render(fmt), ol.pack(fmt, compose(plain, full, m)))
                assert np.array_equal(ds.refine_mask()[0], m)
                # the hit-id hook ignores the setting and leaves the last frame's mask alone
                ds.primary_hit_ids(w, h)
                assert ds.counters()['primary_rays'] == w * h
                assert np.array_equal(ds.refine_mask()[0], m)
        if name == 'cell120':
            assert 0 < int(m.sum()) < w * h


@pytest.mark.gpu
def test_huge_threshold_gives_the_plain_frame():
    sc = load_case('ggs120', 'refl')
    w, h = 128, 72
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    with _dev(sc) as ds:
        want = ds.render(fmt)
    with _dev(sc, 4, 1e30) as ds:
        got = ds.render(fmt)
        mask, n = ds.refine_mask()
        assert n == 0 and not mask.any()
        assert ds.counters()['primary_rays'] == w * h
    assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1
    with _dev(load_case('cell120', 'shadows'), 4, 1e30) as ds:
        with _dev(load_case('cell120', 'shadows')) as plain:
            assert np.array_equal(ds.render(fmt), plain.render(fmt))


def _contrast(rgb):
    """max over channels of the corner-set span (the quantity the rule compares with t)"""
    h, w = rgb.shape[:2]
    lo, hi = rgb.copy(), rgb.copy()
    for dy, dx in ((0, 1), (1, 0), (1, 1)):
        nb = rgb[dy:, dx:]
        lo[:h - dy, :w - dx] = np.minimum(lo[:h - dy, :w - dx], nb)
        hi[:h - dy, :w - dx] = np.maximum(hi[:h - dy, :w - dx], nb)
    return (hi - lo).max(axis=2)


@pytest.mark.gpu
@pytest.mark.parametrize('name,v', [('cell120', 'refl_transp'), ('ggs120', 'refl'), ('ssc120', 'refl_transp')])
def test_reflective_frames_match_the_composition(name, v):
    sc = load_case(name, v)
    w, h = 160, 90
    s, t = 2, 4 / 255
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    plain, full = _reference(sc, w, h, s)
    m = rule(plain, t)
    with _dev(sc, s, t) as ds:
        img = ds.render(fmt)
        mask, n = ds.refine_mask()
        cnt = ds.counters()
    differ = mask != m
    # the bounce passes add with float atomics in no fixed order: only pixels whose contrast is that close to t may flip
    assert np.all(np.abs(_contrast(plain)[differ] - t) <= 1e-5), (name, v, int(differ.sum()))
    want = ol.pack(fmt, compose(plain, full, mask))
    assert np.abs(img.astype(np.int32) - want.astype(np.int32)).max() <= 1, (name, v)
    assert n == int(mask.sum()) and cnt['primary_rays'] == w * h + n * s * s
    assert cnt['reflection_rays'] > 0


def _strips(ds, fmt, world, compact, torch):
    h = fmt.height
    out = np.zeros((h, fmt.pitch), np.uint8)
    mask = np.zeros((h, fmt.width), np.uint8)
    prim = 0
    for rank in range(world):
        rows = [ty for ty in range((h + 31) // 32) if ty % world == rank]
        n = (len(rows) * 32 if compact else h) * fmt.pitch
        strip = torch.zeros(n, dtype=torch.uint8, device='cuda')
        ds.render_device(fmt, strip.data_ptr(), strip.numel(), 0, rank, world, compact)
        torch.cuda.synchronize()
        st = strip.cpu().numpy().reshape(-1, fmt.pitch)
        for k, ty in enumerate(rows):
            r = min(32, h - ty * 32)
            out[ty * 32:ty * 32 + r] = st[(k * 32 if compact else ty * 32):][:r]
        rm, _ = ds.refine_mask()
        own = owned_rows(h, rank, world)
        assert not rm[~own].any()
        mask[own] = rm[own]
        prim += ds.counters()['primary_rays']
    return out, mask, prim


@pytest.mark.gpu
@pytest.mark.parametrize('v', ['shadows', 'refl'])
def test_every_render_path_gives_the_same_frame(v, monkeypatch):
    import torch
    from ntracer_b200.backend import DeviceGroup
    sc = load_case('cell120', v)
    w, h = 320, 288                     # 9 tile rows: ragged interleaves
    s, t = 2, 4 / 255
    tol = 0 if v == 'shadows' else 1
    fmt = _capi.make_image_format(w, h, _capi.RGB8)

    def same(a, what):
        d = np.abs(np.asarray(a, np.int32).reshape(h, fmt.pitch) - want.astype(np.int32).reshape(h, fmt.pitch)).max()
        assert d <= tol, (v, what, d)

    def same_mask(m, what):
        if tol == 0:
            assert np.array_equal(m, want_mask), (v, what)
        else:
            assert np.mean(m != want_mask) <= 0.001, (v, what)

    with _dev(sc, s, t) as ds:
        fl = ds.render_float(w, h)
        want_mask, want_n = ds.refine_mask()
        assert 0 < want_n < w * h
        want = ol.pack(fmt, fl)
        same(ds.render(fmt), 'ntr_render, staged')
        same_mask(ds.refine_mask()[0], 'ntr_render')
        pinned = torch.zeros(fmt.pitch * h, dtype=torch.uint8).pin_memory()
        same(ds.render(fmt, pinned.numpy()), 'ntr_render, pinned destination')
        dev = torch.zeros(fmt.pitch * h, dtype=torch.uint8, device='cuda')
        ds.render_device(fmt, dev.data_ptr(), dev.numel())
        torch.cuda.synchronize()
        same(dev.cpu().numpy(), 'ntr_render_device')
        whole = ds.counters()['primary_rays']
        for world in (2, 3):
            for compact in (True, False):
                img, m, prim = _strips(ds, fmt, world, compact, torch)
                what = 'interleaved tile rows, %s, %d ranks' % ('compact' if compact else 'at frame positions', world)
                same(img, what)
                same_mask(m, what)
                if tol == 0:
                    # every rank traces its own pixels, its halo rows and its refined pixels
                    halo = w * sum(1 for ty in range((h + 31) // 32) if (ty + 1) * 32 < h)
                    assert prim == whole + halo, what
        # calculate_color at interior, edge and view-border pixels
        for x, y in ((100, 100), (w - 1, 50), (60, h - 1), (w - 1, h - 1), (0, 0), (31, 31), (32, 32)):
            c = ds.calculate_color(x, y, w, h)
            assert np.abs(c - fl[y, x]).max() <= (0 if tol == 0 else 1e-5), (v, x, y)
            assert ds.refine_mask()[0].shape == (1, 1)
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
        with _dev(sc, s, t) as ds:
            same(ds.render(fmt), env)
        monkeypatch.delenv(env)
    # a group listing the same device twice: two ranks of interleaved tile rows on one GPU
    with DeviceGroup(sc, devices=[0, 0]) as grp:
        grp.set_supersampling(s)
        grp.set_supersampling_threshold(t)
        same(grp.render(fmt), 'ntr_group_render')
        m, n = grp.refine_mask()
        same_mask(m, 'ntr_group_render')
        assert n == int(m.sum())
        halo = w * sum(1 for ty in range((h + 31) // 32) if (ty + 1) * 32 < h)
        assert grp.counters()['primary_rays'] == w * h + halo + n * s * s


@pytest.mark.gpu
def test_stream_renderer_frames_match_blocking_renders():
    from ntracer_b200 import BlockingRenderer, Channel, ImageFormat, StreamRenderer
    nt, scene = _box_scene()
    scene.set_supersampling(3, 4 / 255)
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
    assert scene._dev.refine_mask()[1] > 0


@pytest.mark.gpu
def test_abort_of_an_adaptive_frame():
    """A 960x540 frame at factor 4 with threshold 0 refines most of its pixels: the rays of a 4K frame."""
    import time
    from ntracer_b200 import bulk
    pts = bulk.soup(10, 60000)
    sc = bulk.simplex_scene(pts, max_depth=14)
    sc['cam_origin'] = np.array([0, 0, -3] + [0] * 7, np.float32)
    with _dev(sc, 4, 0.0) as ds:
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
def test_forced_queue_regrow_in_the_refine_round(monkeypatch):
    sc = load_case('cell120', 'refl_transp')
    w, h = 160, 90
    s, t = 3, 0.0                       # threshold 0: the refine round holds most of the bounces
    monkeypatch.setenv('NTR_QUEUE_INIT', str(w * h * 2 * s * s * 4))
    with _dev(sc, s, t) as ds:
        ref = ds.render_float(w, h)
        m0 = ds.refine_mask()[0]
        assert ds.counters()['queue_overflows'] == 0
    # the plain frame's passes fit, the refine round's (up to s*s times as many) do not
    monkeypatch.setenv('NTR_QUEUE_INIT', str(w * h * 2))
    with _dev(sc, s, t) as ds:
        img = ds.render_float(w, h)
        assert ds.counters()['queue_overflows'] >= 1
        agree = ds.refine_mask()[0] == m0
        assert np.mean(~agree) <= 0.001
        assert np.abs(img - ref)[agree].max() <= 1e-5
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        assert np.abs(ds.render(fmt).astype(np.int32) - ol.pack(fmt, ref).astype(np.int32)).max() <= 1
