"""Batches of camera views in one call (ntr_render_views, ntr_render_views_device, ntr_group_render_views,
BlockingRenderer.render_views): frame k is what ntr_render gives after ntr_scene_set_camera(origins[k], axes[k]) --
byte-identical for frames without reflection passes, within 1 LSB with them -- and the counters are the per-view sums.

CPU tier: the host emulation of the device code shows that the NTR_F_VIEWS primary pass (ss_pixel_color at factor 1, as
those kernels run it) is the plain primary pass bit for bit, and the Python surface runs on a test double of the library.
GPU tier (`-m gpu`): the CUDA library against per-view renders on the kernel matrix's scenes, every route of a views call,
and NTR_LAUNCH_LOG=1 coverage of the 36 NTR_F_VIEWS builds (4 per dimension family)."""
import ctypes as C
import re
import threading

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_lib as el
from tests import emul_views_lib as ev
from tests import fixtures as fx
from tests import oracle_lib as ol
from tests.test_facade_emulated import _FakeLibrary
from tests.test_kernel_matrix import CASE_IDS, CASES, giant_leaf_soup, pass_free

W, H = 64, 36
F_GENERAL, F_COUNT, F_VIEWS = 1, 2, 64
FAMILIES = (3, 4, 5, 6, 7, 8, 9, 10, 0)
VIEWS_BUILDS = {(fam, F_VIEWS | k) for fam in FAMILIES for k in range(4)}
GOLDEN_SCENES = ('box3', 'box4', 'box6', 'box9', 'cell120', 'ggs120', 'mixed3', 'solids6', 'soup9', 'ssc120')


def cameras(sc, n=5, steps=40):
    """n views of the rotation of `polytope.py --benchmark` (stream.rotation_cameras), a few degrees apart"""
    from ntracer_b200.stream import rotation_cameras
    return rotation_cameras(sc['cam_origin'], sc['cam_axes'], steps)[:n]


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------

def _same_bits(r, what):
    a, b = r['plain'].view(np.uint32), r['views'].view(np.uint32)
    assert np.array_equal(a, b), (what, int((a != b).sum()))
    assert r['same_records'] and r['plain_records'] == r['views_records'], what
    assert r['plain_counters'] == r['views_counters'], what


@pytest.mark.parametrize('name', GOLDEN_SCENES)
def test_emulated_views_pass_at_factor_one_is_the_plain_pass(name):
    """Colour bits (signed zeros included), emitted bounce records and counters, on every golden scene and its variants."""
    sc, g = fx.load(name)
    scenes = [sc] + [fx.variant(sc, g, str(v)) for v in g.get('variants', [])]
    for s in scenes:
        for cam in cameras(s, 2):
            _same_bits(ev.factor1(s, W, H, cam=cam), name)


@pytest.mark.parametrize('dim', [3, 4, 9, 16])
def test_emulated_views_pass_on_the_giant_leaf_soup(dim):
    for transparent in (False, True):
        sc = giant_leaf_soup(dim, transparent=transparent)
        for generic in ((False, True) if dim <= 10 else (True,)):
            _same_bits(ev.factor1(sc, W, H, generic=generic), (dim, transparent, generic))


def test_emulated_views_pass_on_the_fuzz_corpus():
    """>= 200 random mixed scenes: solids, transparent and reflective materials, random shadows / lights / depths."""
    for seed in range(200):
        sc = fx.fuzz_scene(3 + seed % 5, seed)
        _same_bits(ev.factor1(sc, 32, 18), seed)


def test_the_views_pass_keeps_negative_zeros_where_the_supersampled_pass_does_not():
    """Why the NTR_F_VIEWS builds call ss_pixel_color with EXACT1: the BoxScene background stores -0 where the direction's
    gradient axis is +0 (the centre column of an axis-aligned camera, where the rays miss the box), and the supersampled
    pass's 0.0f + c makes it +0.  With EXACT1 the factor-1 pixel keeps the plain path's bits."""
    sc, _ = fx.load('box4')
    cam = (np.array([0, 0, -5, 0], np.float32), np.eye(4, dtype=np.float32))
    exact = ev.factor1(sc, 64, 96, cam=cam, exact=True)
    plain = exact['plain']
    negz = (plain == 0) & np.signbit(plain)
    assert negz.sum() > 0
    _same_bits(exact, 'exact')
    default = ev.factor1(sc, 64, 96, cam=cam, exact=False)
    assert not np.signbit(default['views'][negz]).any()


# ---- the Python surface on a test double ------------------------------------------------------------------------------

class _FakeViewsLibrary(_FakeLibrary):
    """+ ntr_render_views answered by the host emulation, view by view; records the cameras it was handed."""
    def __init__(self, dev):
        super().__init__(dev)
        self.calls, self.during = [], None

    def ntr_render_views(self, handle, n, optr, aptr, fmt_ref, ptr, size):
        fmt, D = fmt_ref._obj, self.dev.dim
        addr = lambda p: p.value if hasattr(p, 'value') else p
        o = np.frombuffer((C.c_float * (n * D)).from_address(addr(optr)), np.float32).reshape(n, D).copy()
        a = np.frombuffer((C.c_float * (n * D * D)).from_address(addr(aptr)), np.float32).reshape(n, D, D).copy()
        self.calls.append((o, a))
        if self.during:
            self.during()
        fb, row_bytes = fmt.pitch * fmt.height, fmt.width * fmt.bytes_per_pixel
        for k in range(n):
            packed = ol.pack(fmt, el.render(self.dev.sc, fmt.width, fmt.height, cam=(o[k], a[k]))[0])
            for y in range(fmt.height):
                C.memmove(addr(ptr) + k * fb + y * fmt.pitch, packed[y * fmt.pitch:].ctypes.data, row_bytes)
        return 0


@pytest.fixture
def emulated(monkeypatch):
    from ntracer_b200 import tracern
    from tests.test_mirror_vs_reference import _EmulatedRenderDevice

    class Dev(_EmulatedRenderDevice):
        last = None

        def __init__(self, sc, device=-1):
            super().__init__(sc, device)
            self.dim = int(sc['dim'])
            self._lib, self._h = _FakeViewsLibrary(self), C.c_void_p(1)
            Dev.last = self

        def abort(self):
            pass

    monkeypatch.setattr(tracern, 'DeviceScene', Dev)
    return Dev


def _box_scene(dim=4):
    from ntracer_b200 import NTracer
    nt = NTracer(dim)
    scene = nt.BoxScene()
    cam = nt.Camera()
    cam.translate(nt.Vector.axis(2, -5))
    scene.set_camera(cam)
    return nt, scene


def _fmt(w=24, h=16, pitch=0):
    from ntracer_b200.render import Channel, ImageFormat
    return ImageFormat(w, h, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)], pitch)


def test_render_views_on_the_emulated_device(emulated):
    from ntracer_b200.render import BlockingRenderer
    nt, scene = _box_scene()
    fmt = _fmt()
    cams = []
    for k in range(3):
        c = nt.Camera()
        c.translate(nt.Vector.axis(2, -5 - k))
        cams.append(c)
    r = BlockingRenderer()
    buf = bytearray(3 * fmt.pitch * fmt.height)
    assert r.render_views(buf, fmt, scene, cams) is True
    frames = np.frombuffer(buf, np.uint8).reshape(3, -1)
    for k, c in enumerate(cams):             # frame k is render() with camera k
        scene.set_camera(c)
        one = bytearray(fmt.pitch * fmt.height)
        assert r.render(one, fmt, scene)
        assert bytes(frames[k]) == bytes(one)
    assert scene.locked == 0
    # Camera objects and (origin, axes) pairs give the same call
    lib = emulated.last._lib
    r.render_views(bytearray(len(buf)), fmt, scene, [(c._origin, c._axes) for c in cams])
    r.render_views(bytearray(len(buf)), fmt, scene, [cams[0], (cams[1]._origin, cams[1]._axes), cams[2]])
    for o, a in lib.calls[-2:]:
        assert np.array_equal(o, lib.calls[0][0]) and np.array_equal(a, lib.calls[0][1])


def test_render_views_argument_errors(emulated):
    from ntracer_b200 import NTracer
    from ntracer_b200.render import BlockingRenderer
    nt, scene = _box_scene()
    fmt = _fmt()
    r = BlockingRenderer()
    cam = nt.Camera()
    buf = bytearray(2 * fmt.pitch * fmt.height)
    with pytest.raises(TypeError):
        r.render_views(buf, 'not a format', scene, [cam])
    with pytest.raises(TypeError):
        r.render_views(buf, fmt, object(), [cam])
    with pytest.raises(TypeError):
        r.render_views(buf, fmt, scene, [cam, 'not a camera'])
    with pytest.raises(TypeError):
        r.render_views(buf, fmt, scene, 5)
    with pytest.raises(ValueError):                 # dimension mismatch
        r.render_views(buf, fmt, scene, [NTracer(5).Camera()])
    with pytest.raises(ValueError):
        r.render_views(buf, fmt, scene, [(np.zeros(3), np.eye(3))])
    with pytest.raises(ValueError):                 # short buffer
        r.render_views(bytearray(2 * fmt.pitch * fmt.height - 1), fmt, scene, [cam, cam])
    with pytest.raises(ValueError):
        r.render_views(buf, fmt, scene, [])
    with pytest.raises(BufferError):
        r.render_views(bytes(len(buf)), fmt, scene, [cam])
    assert scene.locked == 0


def test_render_views_locks_the_scene_and_the_renderer(emulated):
    from ntracer_b200.render import BlockingRenderer, LockedError
    nt, scene = _box_scene()
    fmt = _fmt()
    r = BlockingRenderer()
    cam = nt.Camera()
    scene._prepare()
    seen = {}

    def during():
        seen['locked'] = scene.locked
        with pytest.raises(LockedError):
            scene.set_camera(nt.Camera())
        with pytest.raises(RuntimeError):               # the renderer is already running
            r.render_views(bytearray(fmt.pitch * fmt.height), fmt, scene, [cam])

    emulated.last._lib.during = during
    assert r.render_views(bytearray(fmt.pitch * fmt.height), fmt, scene, [cam])
    assert seen['locked'] == 1 and scene.locked == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------

_SEEN_VIEWS = set()         # (family, flags) of the NTR_F_VIEWS launches of this module
_RAN = set()


def _launches(text):
    return [(int(a), int(b)) for a, b in re.findall(r'ntr launch family=(\d+) flags=(\d+) grid=\d+', text)]


@pytest.fixture
def log(monkeypatch, capfd):
    """log(views_call) -> the launches since the last call; a views call's are recorded, any other call may launch none
    of the NTR_F_VIEWS builds"""
    monkeypatch.setenv('NTR_LAUNCH_LOG', '1')
    capfd.readouterr()

    def read(views_call):
        got = _launches(capfd.readouterr().err)
        views = {x for x in got if x[1] & F_VIEWS}
        if views_call:
            assert views, 'a views call launched no NTR_F_VIEWS build'
            _SEEN_VIEWS.update(views)
        else:
            assert not views, views
        return got
    return read


@pytest.fixture
def env(monkeypatch):
    from tests.test_kernel_matrix import SWITCHES

    def set_(**kw):
        for k in SWITCHES + ('NTR_VIEWS_PER_LAUNCH',):
            monkeypatch.delenv(k, raising=False)
        for k, v in kw.items():
            monkeypatch.setenv(k, str(v))
    set_()
    return set_


def _per_view(ds, fmt, cams):
    """per-view ntr_render frames and counters summed over the views"""
    frames, total = [], {}
    for o, a in cams:
        ds.set_camera(o, a)
        frames.append(ds.render(fmt))
        for k, v in ds.counters().items():
            total[k] = total.get(k, 0) + v
    return np.stack(frames), total


def _check(views, ref, exact, what):
    if exact:
        assert np.array_equal(views, ref), (what, int((views != ref).sum()))
    else:
        assert np.abs(views.astype(np.int32) - ref.astype(np.int32)).max() <= 1, what


def _check_counters(cnt, ref, n, w, h, ss, instrumented, what):
    assert cnt['primary_rays'] == n * w * h * ss * ss, what
    keys = ('reflection_rays', 'shadow_rays', 'shaded_hits') + (('node_steps', 'simplex_tests', 'solid_tests') if instrumented else ())
    for k in keys:
        assert cnt[k] == ref[k], (what, k, cnt[k], ref[k])


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
@pytest.mark.parametrize('kind', ['giant_opaque', 'giant_general', 'soup', 'soup_refl'])
def test_views_equal_per_view_renders(dim, generic, kind, env, log):
    from ntracer_b200.backend import DeviceScene
    env(**({'NTR_FORCE_GENERIC': 1} if generic else {}))
    if kind.startswith('giant'):
        sc = giant_leaf_soup(dim, transparent=kind == 'giant_general')
    else:
        sc = fx.batched_soup(dim, 40)
        sc = sc if kind == 'soup_refl' else pass_free(sc)
    exact = kind in ('giant_opaque', 'soup')
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    cams = cameras(sc)
    with DeviceScene(sc) as ds:
        for instrumented in (False, True):
            ds.set_instrumented(instrumented)
            ref, total = _per_view(ds, fmt, cams)
            log(False)
            got = ds.render_views(fmt, cams)
            log(True)
            _check(got, ref.reshape(len(cams), -1), exact, (dim, generic, kind, instrumented))
            _check_counters(ds.counters(), total, len(cams), W, H, 1, instrumented, (dim, generic, kind, instrumented))
    _RAN.add('matrix')


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['box3', 'box4', 'box6', 'box9'])
def test_box_scene_views(name, env, log):
    from ntracer_b200.backend import DeviceScene
    sc, _ = fx.load(name)
    fmt = _capi.make_image_format(W, 96, _capi.RGB8)
    d = int(sc['dim'])
    cams = [(np.array([0, 0, -5 - 0.5 * k] + [0] * (d - 3), np.float32), np.eye(d, dtype=np.float32)) for k in range(3)]
    cams += cameras(dict(sc, cam_origin=cams[0][0], cam_axes=cams[0][1]), 3, 12)[1:]
    with DeviceScene(sc) as ds:
        for ss in (1, 2):
            ds.set_supersampling(ss)
            ref, _ = _per_view(ds, fmt, cams)
            log(False)
            _check(ds.render_views(fmt, cams), ref.reshape(len(cams), -1), True, (name, ss))
            log(True)


def _ggs(v):
    sc, g = fx.load('ggs120')
    return fx.variant(sc, g, v) if v else sc


@pytest.mark.gpu
@pytest.mark.parametrize('reflective', [False, True], ids=['single_pass', 'passes'])
def test_supersampled_and_adaptive_views(reflective, env, log):
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('refl_transp') if reflective else pass_free(_ggs(None))
    fmt = _capi.make_image_format(80, 48, _capi.RGB8)
    cams = cameras(sc)
    with DeviceScene(sc) as ds:
        for ss in (2, 3):
            ds.set_supersampling(ss)
            ref, total = _per_view(ds, fmt, cams)
            log(False)
            _check(ds.render_views(fmt, cams), ref.reshape(len(cams), -1), not reflective, ss)
            log(True)
            _check_counters(ds.counters(), total, len(cams), 80, 48, ss, False, ss)
        ds.set_supersampling(3)
        ds.set_supersampling_threshold(4 / 255)
        ref, total = _per_view(ds, fmt, cams)
        mask_last = ds.refine_mask()
        got = ds.render_views(fmt, cams)
        log(False)                      # adaptive: view after view through the single-view route
        _check(got, ref.reshape(len(cams), -1), not reflective, 'adaptive')
        assert ds.counters()['primary_rays'] == total['primary_rays']
        m, c = ds.refine_mask()         # describes the last view
        assert np.array_equal(m, mask_last[0]) and c == mask_last[1]


@pytest.mark.gpu
def test_launch_size_and_queue_regrowth(env, log):
    from ntracer_b200.backend import DeviceScene
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    for name, sc, exact in (('single_pass', pass_free(_ggs(None)), True), ('passes', _ggs('refl_transp'), False)):
        cams = cameras(sc)
        with DeviceScene(sc) as ds:
            ref, _ = _per_view(ds, fmt, cams)
            one = ds.render_views(fmt, cams)
        log(True)
        env(NTR_VIEWS_PER_LAUNCH=2)
        with DeviceScene(sc) as ds:
            _check(ds.render_views(fmt, cams), ref.reshape(len(cams), -1), exact, name)
            assert np.array_equal(ds.render_views(fmt, cams), one) or not exact
        got = log(True)
        assert sum(1 for x in got if x[1] & F_VIEWS) == 2 * 3, name        # 5 views in launches of 2, twice
        env()
        if not exact:
            env(NTR_QUEUE_INIT=512)
            with DeviceScene(sc) as ds:
                _check(ds.render_views(fmt, cams), ref.reshape(len(cams), -1), False, 'regrow')
                assert ds.counters()['queue_overflows'] > 0
            log(True)
            env()


@pytest.mark.gpu
@pytest.mark.parametrize('reflective', [False, True], ids=['single_pass', 'passes'])
def test_device_and_pinned_destinations_and_pitch_padding(reflective, env, log):
    import torch
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('refl_transp') if reflective else pass_free(_ggs(None))
    w, h, pitch = 70, 40, 256
    fmt = _capi.make_image_format(w, h, _capi.RGB8, pitch)
    cams = cameras(sc, 4)
    n, fb = len(cams), pitch * h
    with DeviceScene(sc) as ds:
        ref, _ = _per_view(ds, fmt, cams)
        log(False)
        host = np.full(n * fb, 0xAB, np.uint8)
        ds.render_views(fmt, cams, host)
        pinned = torch.full((n * fb,), 0xAB, dtype=torch.uint8).pin_memory()
        ds.render_views(fmt, cams, pinned.numpy())
        dev = torch.full((n, h, pitch), 0xAB, dtype=torch.uint8, device='cuda')
        stream = torch.cuda.Stream()
        ds.render_views_device(fmt, cams, dev.data_ptr(), dev.numel(), stream.cuda_stream)
        stream.synchronize()
        log(True)
        frames = host.reshape(n, h, pitch)
        pixels = (slice(None), slice(None), slice(0, w * 3))
        ref = ref.reshape(n, h, pitch)
        _check(frames[pixels], ref[pixels], not reflective, 'host')
        assert np.array_equal(pinned.numpy(), host) or reflective
        _check(dev.cpu().numpy()[pixels], frames[pixels], not reflective, 'device')
        for out in (frames, pinned.numpy().reshape(n, h, pitch), dev.cpu().numpy()):
            assert (out[:, :, w * 3:] == 0xAB).all()            # pitch padding left alone
        # the scene's own camera is still the last one set (by _per_view)
        _check(ds.render(fmt), ref[-1].reshape(-1), not reflective, 'camera')
        with pytest.raises(ValueError):
            ds.render_views(fmt, cams, np.zeros(n * fb - 1, np.uint8))
        with pytest.raises(ValueError):
            ds.render_views_device(fmt, cams, dev.data_ptr(), n * fb - 1)


@pytest.mark.gpu
def test_scene_state_is_untouched_by_a_views_call(env, log):
    """A frame after a views call makes the same sort and tile-order decisions (equal launch counts) and gives the same
    bytes as without the call in between."""
    from ntracer_b200.backend import DeviceScene
    sc = giant_leaf_soup(4)
    fmt = _capi.make_image_format(320, 180, _capi.RGB8)
    cams = cameras(sc, 6)
    runs = []
    for with_views in (False, True):
        with DeviceScene(sc) as ds:
            out = []
            for k in (0, 1):
                if k == 1 and with_views:
                    ds.render_views(fmt, cams[2:])
                ds.set_camera(*cams[k])
                l0 = ds.launch_count()
                img = ds.render(fmt)
                out.append((img, ds.launch_count() - l0))
                ds.set_camera(*cams[k])
                l0 = ds.launch_count()
                out.append((ds.render(fmt), ds.launch_count() - l0))        # a second frame of the view: sorted passes
            runs.append(out)
    log(True)
    for (a, la), (b, lb) in zip(*runs):
        assert la == lb
        _check(a, b, False, 'state')


@pytest.mark.gpu
def test_abort_of_a_views_call(monkeypatch):
    """Following tests/test_supersampling.py's abort test: three 960x540 views at factor 4."""
    import time
    from ntracer_b200 import bulk
    from ntracer_b200.backend import DeviceScene
    from ntracer_b200.render import BlockingRenderer, ImageFormat, Channel, Scene
    monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    pts = bulk.soup(10, 60000)
    sc = bulk.simplex_scene(pts, max_depth=14)
    sc['cam_origin'] = np.array([0, 0, -3] + [0] * 7, np.float32)
    ds = DeviceScene(sc)
    ds.set_supersampling(4)

    class Big(Scene):
        locked, dimension = 0, 10

        def _prepare(self, gpus=1):
            return ds

    scene = Big()
    fmt = ImageFormat(960, 540, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)])
    cams = cameras(sc, 3)
    buf = bytearray(3 * fmt.pitch * 540)
    r = BlockingRenderer()
    t0 = time.perf_counter()
    assert r.render_views(buf, fmt, scene, cams) is True
    full = time.perf_counter() - t0
    result = {}
    th = threading.Thread(target=lambda: result.setdefault('rc', r.render_views(buf, fmt, scene, cams)))
    t0 = time.perf_counter()
    th.start()
    time.sleep(min(0.05, full / 10))
    r.signal_abort()
    th.join()
    aborted = time.perf_counter() - t0
    if full > 0.3:
        assert result['rc'] is False
        assert aborted < 0.8 * full
    assert r.render_views(buf, fmt, scene, cams) is True
    ds.close()


@pytest.mark.gpu
def test_group_deals_whole_views(env, log):
    """A group (one device listed twice on a one-GPU box: two entries, two chains) equals single-device render_views, with
    the counters summed and every entry tracing its run."""
    from ntracer_b200.backend import DeviceGroup, DeviceScene, device_count
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    devices = [0, 1] if device_count() >= 2 else [0, 0]
    for sc, exact in ((pass_free(_ggs(None)), True), (_ggs('refl_transp'), False)):
        cams = cameras(sc)
        with DeviceScene(sc) as ds:
            ref = ds.render_views(fmt, cams)
            cnt = ds.counters()
        log(True)
        with DeviceGroup(sc, devices=devices) as g:
            got = g.render_views(fmt, cams)
            gcnt = g.counters()
            assert g.last_kernel_ms() > 0
        launches = [x for x in log(True) if x[1] & F_VIEWS]
        assert len(launches) == len(devices)            # runs of 2 and 3 views: one launch per entry
        _check(got, ref, exact, 'group')
        for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert gcnt[k] == cnt[k], k
        with DeviceGroup(sc, devices=devices) as g:       # more entries than views: the idle entry is skipped
            _check(g.render_views(fmt, cams[:1]), ref[:1], exact, 'one view')
        log(True)


@pytest.mark.gpu
def test_every_views_build_ran():
    """All 36 NTR_F_VIEWS builds (4 per dimension family) appear among this module's views calls; no other call launched
    one (the log fixture checks every call)."""
    if 'matrix' not in _RAN:
        pytest.skip('the views matrix did not run in this session')
    assert VIEWS_BUILDS <= _SEEN_VIEWS, sorted(VIEWS_BUILDS - _SEEN_VIEWS)
    assert len(VIEWS_BUILDS) == 36
