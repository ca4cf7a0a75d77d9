"""Orthographic and equirectangular projections (ntr_scene_set_projection, Scene.set_projection) and the camera's own rays
(ntr_camera_rays, DeviceScene.camera_rays).

CPU tier: the host emulation of projected frames (tests/emul_proj_lib.py: the product's ray generator and the primary pass of
the NTR_F_PROJ builds) against the oracle's colour of each emulated camera ray, against the ray-fed pass of the same rays
(colour bits, bounce records, counters) and against a float64 statement of the two formulas; sample (0, 0) at powers of two;
the Python surface on a test double.  GPU tier: every route against render_rays of the device's own camera rays, the kernel
matrix against the oracle, AOVs, abort, queue regrowth and launch-log coverage of the 108 builds."""
import ctypes as C
import math
import pickle
import re

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_proj_lib as ep
from tests import emul_rays_lib as er
from tests import fixtures as fx
from tests import oracle_lib as ol
from tests import oracle_rays_lib as orl
from tests.test_kernel_matrix import CASE_IDS, CASES, giant_leaf_soup, pass_free
from tests.test_supersampling import box_sum
from tests.test_views import GOLDEN_SCENES, _ggs, cameras

EMUL_TOL = 2e-6                 # the host emulation against the oracle (tests/test_render_rays.py)
FAMILIES = (3, 4, 5, 6, 7, 8, 9, 10, 0)
VIEWS, AOV, LIST, PROJ = 64, 128, 32, 256
PROJ_BUILDS = {(fam, k | extra) for fam in FAMILIES for k in range(4) for extra in (VIEWS | PROJ, VIEWS | AOV | PROJ, LIST | PROJ)}


def scene_box(sc):
    D = int(sc['dim'])
    if int(sc['kind']) == 0:
        return np.full(D, -1.0), np.full(D, 1.0)
    lo, hi = np.asarray(sc['boundary'], np.float64)
    return lo, hi


def projections(sc):
    """an orthographic view as wide as the scene box and a full-sphere panorama"""
    lo, hi = scene_box(sc)
    return [('orthographic', float(np.max(hi - lo)) * 0.6), ('equirectangular', 2 * math.pi)]


def ortho_camera(sc, cam):
    """cam moved back along its forward axis so that the orthographic image plane lies outside the scene box"""
    lo, hi = scene_box(sc)
    o, a = np.asarray(cam[0], np.float64), np.asarray(cam[1], np.float64)
    centre, r = (lo + hi) / 2, np.linalg.norm(hi - lo)
    return (centre - a[2] * r).astype(np.float32), a.astype(np.float32)


def cams_for(sc, kind, n=1):
    cs = cameras(sc, n) if n > 1 else [(np.asarray(sc['cam_origin'], np.float32), np.asarray(sc['cam_axes'], np.float32))]
    return [ortho_camera(sc, c) for c in cs] if kind == 'orthographic' else cs


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def formula_rays(cam, w, h, kind, param):
    """the contract's two formulas in float64 (k and a as the host computes them, in float)"""
    o, ax = np.asarray(cam[0], np.float64), np.asarray(cam[1], np.float64)
    right, up, fwd = ax[0], ax[1], ax[2]
    hw, hh = np.float32(w / 2), np.float32(h / 2)
    y, x = np.mgrid[0:h, 0:w]
    x, y = x.ravel().astype(np.float64), y.ravel().astype(np.float64)
    if kind == 'orthographic':
        k = float(np.float32(param) / hw)
        fx_, fy_ = k * (x - hw), k * (y - hh)
        org = o + fx_[:, None] * right - fy_[:, None] * up
        d = np.tile(fwd, (len(x), 1))
    else:
        a = float(np.float32(param) / (np.float32(2) * hw))
        th, ph = a * (x - hw), a * (y - hh)
        org = np.tile(o, (len(x), 1))
        d = np.cos(ph)[:, None] * (np.sin(th)[:, None] * right + np.cos(th)[:, None] * fwd) - np.sin(ph)[:, None] * up
    return org, d / np.linalg.norm(d, axis=1, keepdims=True)


def oracle_frame(sc, w, h, kind, param, s, cam):
    """the oracle's colours of the emulated camera rays of the sW x sH view, box-averaged as the contract states"""
    o, d = ep.camera_rays(sc, s * w, s * h, kind, param, cam=cam)
    ref = orl.ray_colors(sc, o, d)
    rgb = ref['rgb'].reshape(s * h, s * w, 3)
    und = ref['undefined'].reshape(s * h, s * w).astype(bool)
    und = np.logical_or.reduce([und[j::s, i::s] for j in range(s) for i in range(s)])
    return (box_sum(rgb, s) if s > 1 else rgb), und


def check_oracle(sc, w, h, kind, param, what, cam=None, factors=(1, 2, 3), threshold=4 / 255, generic=False):
    cam = cam if cam is not None else cams_for(sc, kind)[0]
    refs = {}
    for s in factors:
        got = ep.render(sc, w, h, kind, param, ss=s, cam=cam, generic=generic)
        ref, und = refs[s] = oracle_frame(sc, w, h, kind, param, s, cam)
        diff = np.where((got['rgb'] == ref) | (np.isnan(got['rgb']) & np.isnan(ref)), 0, np.abs(got['rgb'] - ref))
        # relative beyond 1: rays that graze a point light give colours up to 1e23, where factors that are not powers of two
        # round the weighted sum differently from the box mean
        assert (diff / np.maximum(1, np.abs(ref)))[~und].max(initial=0) <= EMUL_TOL * s * s, (what, kind, s)
        assert got['primary_rays'] == w * h * s * s
    # adaptive at factor 2: refined pixels are the full-SS oracle frame, the others the plain one
    if threshold is not None and 1 in refs and 2 in refs:
        got = ep.render(sc, w, h, kind, param, ss=2, threshold=threshold, cam=cam, generic=generic)
        m = got['mask'].astype(bool)
        ref = np.where(m[..., None], refs[2][0], refs[1][0])
        und = np.where(m, refs[2][1], refs[1][1])
        diff = np.where(got['rgb'] == ref, 0, np.abs(got['rgb'] - ref))
        assert (diff / np.maximum(1, np.abs(ref)))[~und].max(initial=0) <= 4 * EMUL_TOL, (what, kind, 'adaptive')
        assert got['primary_rays'] == w * h + 4 * int(m.sum())


def check_vs_rays(sc, w, h, kind, param, what, cam=None, generic=False):
    r = ep.vs_rays(sc, w, h, kind, param, cam=cam, generic=generic)
    assert same_bits(r['frame'], r['rays']), (what, kind, int((r['frame'] != r['rays']).sum()))
    assert r['same_records'] and r['frame_records'] == r['rays_records'], (what, kind)
    assert r['frame_counters'] == r['rays_counters'], (what, kind)
    # and the whole ray-fed call (emul_rays) gives the frame's colours after the bounces too
    assert same_bits(ep.render(sc, w, h, kind, param, cam=cam, generic=generic)['rgb'].reshape(-1, 3),
                     er.render_rays(sc, r['origins'], r['dirs'], generic=generic)['rgb']), (what, kind)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('name', GOLDEN_SCENES)
def test_emulated_projected_frames_match_the_oracle_on_the_golden_scenes(name):
    sc, g = fx.load(name)
    for i, s in enumerate([sc] + [fx.variant(sc, g, str(v)) for v in g.get('variants', [])][:2]):
        for kind, param in projections(s):
            check_oracle(s, 20, 12, kind, param, (name, i))
            check_vs_rays(s, 20, 12, kind, param, (name, i))


@pytest.mark.parametrize('dim', [3, 4, 9, 16])
def test_emulated_projected_frames_on_the_giant_leaf_soup(dim):
    for transparent in (False, True):
        sc = giant_leaf_soup(dim, transparent=transparent)
        for kind, param in projections(sc):
            check_oracle(sc, 12, 8, kind, param, (dim, transparent), factors=(1, 2), generic=dim > 10)
            check_vs_rays(sc, 12, 8, kind, param, (dim, transparent), generic=dim > 10)


def test_emulated_projected_frames_on_the_fuzz_corpus():
    for seed in range(200):
        sc = fx.fuzz_scene(3 + seed % 5, seed)
        kind, param = projections(sc)[seed % 2]
        check_oracle(sc, 8, 6, kind, param, seed, factors=(1, 2) if seed % 4 < 2 else (1, 3),
                     threshold=1 / 255 if seed % 4 < 2 else None)
        check_vs_rays(sc, 8, 6, kind, param, seed)


@pytest.mark.parametrize('w,h', [(17, 9), (16, 10)])
def test_camera_rays_follow_the_formulas(w, h):
    sc, _ = fx.load('solids6')
    cam = (np.asarray(sc['cam_origin'], np.float32), np.asarray(sc['cam_axes'], np.float32))
    for kind, param in (('orthographic', 1.7), ('equirectangular', 2 * math.pi), ('equirectangular', 1.3)):
        o, d = ep.camera_rays(sc, w, h, kind, param)
        ro, rd = formula_rays(cam, w, h, kind, param)
        assert np.abs(d - rd).max() <= 1e-6, kind
        assert np.abs(o - ro).max() <= 1e-5 * max(1.0, np.abs(ro).max()), kind
        assert np.allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1, atol=1e-6)
        go, gd = ep.camera_rays(sc, w, h, kind, param, generic=True)
        assert same_bits(go, o) and same_bits(gd, d)


def test_full_sphere_panorama_covers_every_direction():
    """a W x W/2 frame at 2 pi: theta in [-pi, pi), phi in [-pi/2, pi/2)"""
    sc, _ = fx.load('box4')
    w, h = 64, 32
    _, d = ep.camera_rays(sc, w, h, 'equirectangular', 2 * math.pi)
    ax = np.asarray(sc['cam_axes'], np.float64)
    c = d.astype(np.float64) @ ax.T                     # components along right, up, fwd, ...
    th = np.arctan2(c[:, 0], c[:, 2]).reshape(h, w)
    ph = -np.arcsin(np.clip(c[:, 1], -1, 1)).reshape(h, w)
    assert abs(th[h // 2 + 1, 0] + math.pi) < 1e-5 or abs(th[h // 2 + 1, 0] - math.pi) < 1e-5
    assert abs(ph[0, 1] + math.pi / 2) < 1e-5 and np.all(np.diff(ph[1:, 1]) > 0)
    assert np.all(np.abs(c[:, 3:]) < 1e-6)             # the camera's 3-flat


@pytest.mark.parametrize('ss', [2, 4, 8])
@pytest.mark.parametrize('w,h', [(13, 7), (12, 8)])
def test_sample_zero_is_the_plain_ray_at_powers_of_two(ss, w, h):
    sc, _ = fx.load('mixed3')
    for kind, param in (('orthographic', 2.5), ('equirectangular', 2 * math.pi), ('equirectangular', 0.9)):
        o1, d1 = ep.camera_rays(sc, w, h, kind, param)
        os_, ds_ = ep.camera_rays(sc, ss * w, ss * h, kind, param)
        D = o1.shape[1]
        os_ = os_.reshape(ss * h, ss * w, D)[::ss, ::ss].reshape(-1, D)
        ds_ = ds_.reshape(ss * h, ss * w, D)[::ss, ::ss].reshape(-1, D)
        assert same_bits(o1, os_) and same_bits(d1, ds_), (kind, ss, w, h)


def test_perspective_camera_rays_are_the_plain_rays():
    sc, _ = fx.load('cell120')
    r = er.vs_plain(sc, 24, 14)
    o, d = ep.camera_rays(sc, 24, 14, 'perspective', None)
    assert same_bits(o, r['origins']) and same_bits(d, r['dirs'])


# ---- the Python surface on a test double ------------------------------------------------------------------------------

def _box_scene():
    from ntracer_b200 import NTracer
    nt = NTracer(4)
    scene = nt.BoxScene()
    cam = nt.Camera()
    cam.translate(nt.Vector.axis(2, -5))
    scene.set_camera(cam)
    return nt, scene


def test_set_projection_validates_and_respects_the_lock():
    from ntracer_b200.render import LockedError
    nt, scene = _box_scene()
    assert scene.projection == ('perspective', None)
    for bad in ('fisheye', 'Orthographic'):
        with pytest.raises(ValueError):
            scene.set_projection(bad, 1.0)
    for bad in (0, None, 1.0, b'orthographic'):
        with pytest.raises(TypeError):
            scene.set_projection(bad)
    for bad in ('1', True, [1.0]):
        with pytest.raises(TypeError):
            scene.set_projection('orthographic', bad)
    with pytest.raises(ValueError):
        scene.set_projection('orthographic')                 # the half width is required
    for bad in (0.0, -1.0, math.inf, math.nan, 1e39):
        with pytest.raises(ValueError):
            scene.set_projection('orthographic', bad)
    for bad in (0.0, -0.5, 6.3, math.inf, math.nan):
        with pytest.raises(ValueError):
            scene.set_projection('equirectangular', bad)
    assert scene.projection == ('perspective', None)
    scene.set_projection('equirectangular')
    assert scene.projection == ('equirectangular', 2 * math.pi)
    scene.set_projection('orthographic', np.float32(2.5))
    assert scene.projection == ('orthographic', 2.5) and type(scene.projection[1]) is float
    scene.locked += 1
    with pytest.raises(LockedError):
        scene.set_projection('perspective')
    scene.locked -= 1
    assert scene.projection == ('orthographic', 2.5)
    scene.set_projection('perspective', 3.0)                 # the parameter is ignored
    assert scene.projection == ('perspective', None) and 'projection' not in scene.__dict__


def test_projection_pickles_only_when_set_and_old_pickles_load_as_perspective():
    from ntracer_b200 import Material
    nt, scene = _box_scene()
    assert 'projection' not in scene.__getstate__()         # never set: pickles as before
    scene.set_projection('orthographic', 3.0)
    assert pickle.loads(pickle.dumps(scene)).projection == ('orthographic', 3.0)
    comp = nt.build_composite_scene([nt.TrianglePrototype([nt.Vector(1, 0, 0, 0), nt.Vector(0, 1, 0, 0), nt.Vector(0, 0, 1, 0),
                                                           nt.Vector(0, 0, 0, 1)], Material((1, 1, 1)))])
    comp.set_projection('equirectangular', 1.5)
    assert pickle.loads(pickle.dumps(comp)).projection == ('equirectangular', 1.5)
    comp.set_projection('perspective')
    assert 'projection' not in comp.__getstate__()
    del scene.__dict__['projection']                        # a scene pickled before the attribute existed
    old = pickle.loads(pickle.dumps(scene))
    assert 'projection' not in old.__dict__ and old.projection == ('perspective', None)


class _ProjLibrary:
    """ntr_scene_set_projection / ntr_group_set_projection / ntr_camera_rays answered by the host emulation"""
    def __init__(self, sc):
        self.sc, self.calls, self.cam = sc, [], (sc['cam_origin'], sc['cam_axes'])

    def ntr_scene_set_projection(self, h, kind, param):
        self.calls.append((kind, param))
        return 0

    ntr_group_set_projection = ntr_scene_set_projection

    def ntr_scene_set_camera(self, h, o, a):
        return 0

    ntr_group_set_camera = ntr_scene_set_camera

    def ntr_camera_rays(self, h, w, ht, op, dp):
        from ntracer_b200.backend import PROJECTIONS
        kind, param = self.calls[-1] if self.calls else (0, 0.0)
        o, d = ep.camera_rays(self.sc, w, ht, PROJECTIONS[kind], param)
        C.memmove(op, o.ctypes.data, o.nbytes)
        C.memmove(dp, d.ctypes.data, d.nbytes)
        return 0

    def ntr_scene_destroy(self, h):
        pass

    ntr_group_destroy = ntr_scene_destroy


def _fake(sc):
    from ntracer_b200.backend import DeviceGroup, DeviceScene
    ds, g = DeviceScene.__new__(DeviceScene), DeviceGroup.__new__(DeviceGroup)
    for x in (ds, g):
        x._lib, x._h, x.dim, x.device = _ProjLibrary(sc), C.c_void_p(1), int(sc['dim']), 0
        x.projection = ('perspective', None)
    return ds, g


def test_device_scene_and_group_forward_the_projection():
    sc, _ = fx.load('box4')
    ds, g = _fake(sc)
    for x in (ds, g):
        x.set_projection('orthographic', 2.0)
        x.set_projection('equirectangular')
        x.set_projection('perspective')
        assert x._lib.calls == [(1, 2.0), (2, pytest.approx(2 * math.pi)), (0, 0.0)]
        assert x.projection == ('perspective', None)
        with pytest.raises(ValueError):
            x.set_projection('orthographic', -1.0)
        assert len(x._lib.calls) == 3                        # refused before the library is called
    ds.set_projection('orthographic', 2.0)
    o, d = ds.camera_rays(9, 5)
    ro, rd = ep.camera_rays(sc, 9, 5, 'orthographic', 2.0)
    assert o.shape == (45, 4) and same_bits(o, ro) and same_bits(d, rd)
    torch = pytest.importorskip('torch')
    with pytest.raises(TypeError):
        ds.camera_rays_device(9, 5, o, d)                    # numpy, not tensors
    with pytest.raises(TypeError):
        ds.camera_rays_device(9, 5, torch.zeros((45, 4)), torch.zeros((45, 4)))     # CPU tensors


def test_scene_prepare_sends_the_projection(monkeypatch):
    """_prepare hands the projection to the device copy once, and again only when it changes"""
    from ntracer_b200 import tracern
    nt, scene = _box_scene()
    sent = []

    class _Dev:
        supersampling, supersampling_threshold, projection = 1, None, ('perspective', None)

        def __init__(self, *a):
            pass

        def set_camera(self, o, a):
            pass

        def set_projection(self, kind, param=None):
            sent.append((kind, param))
            self.projection = (kind, param)

    monkeypatch.setattr(tracern, 'DeviceScene', _Dev)
    scene._prepare()
    assert sent == []
    scene.set_projection('orthographic', 2.0)
    scene._prepare()
    scene._prepare()
    assert sent == [('orthographic', 2.0)]
    scene.set_projection('perspective')
    scene._prepare()
    assert sent == [('orthographic', 2.0), ('perspective', None)]


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------

_SEEN = set()
_CAM = set()
_RAN = set()


@pytest.fixture
def log(monkeypatch, capfd):
    """log() -> the render-pass launches since the last call (recorded for the coverage test)"""
    monkeypatch.setenv('NTR_LAUNCH_LOG', '1')
    capfd.readouterr()

    def read():
        text = capfd.readouterr().err
        got = [(int(a), int(b)) for a, b in re.findall(r'ntr launch family=(\d+) flags=(\d+) grid=\d+', text)]
        _SEEN.update(got)
        _CAM.update(int(a) for a in re.findall(r'ntr camrays-launch family=(\d+) grid=\d+', text))
        return got
    return read


@pytest.fixture
def env(monkeypatch):
    from tests.test_kernel_matrix import SWITCHES

    def set_(**kw):
        for k in SWITCHES + ('NTR_QUEUE_INIT', 'NTR_VIEWS_PER_LAUNCH', 'NTR_NO_SLABS', 'NTR_NO_STAGING'):
            monkeypatch.delenv(k, raising=False)
        for k, v in kw.items():
            monkeypatch.setenv(k, str(v))
    set_()
    return set_


def _dev(sc, kind=None, param=None, s=1, t=None, cam=None):
    from ntracer_b200.backend import DeviceScene
    ds = DeviceScene(sc)
    if cam is not None:
        ds.set_camera(*cam)
    ds.set_supersampling(s)
    ds.set_supersampling_threshold(t)
    if kind:
        ds.set_projection(kind, param)
    return ds


def _rays_frame(ds, w, h, s=1):
    """render_rays of the device's own camera rays of the sW x sH view, box-averaged at factor s"""
    o, d = ds.camera_rays(s * w, s * h)
    rgb = ds.render_rays(o, d).reshape(s * h, s * w, 3)
    return box_sum(rgb, s) if s > 1 else rgb


def _ref_scenes():
    return [(pass_free(_ggs(None)), True), (_ggs('refl_transp'), False)]


@pytest.mark.gpu
def test_perspective_is_unchanged_and_camera_rays_are_the_plain_rays(env, log):
    """launches and frames of the perspective projection, set explicitly or restored, are those of a scene that never set one;
    render_rays of camera_rays is render_float"""
    w, h = 64, 36
    for sc, exact in _ref_scenes():
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        with _dev(sc) as ds:
            n0 = ds.launch_count()
            ref = ds.render(fmt)
            ref_n = ds.launch_count() - n0
            ref_log = log()
            fl = ds.render_float(w, h)
            rr = _rays_frame(ds, w, h)
        if exact:
            assert same_bits(rr, fl)
        else:
            assert np.abs(rr - fl).max() <= 1e-5
        with _dev(sc, 'orthographic', 1.0) as ds:
            ds.set_projection('perspective')
            log()
            n0 = ds.launch_count()
            img = ds.render(fmt)
            assert ds.launch_count() - n0 == ref_n and log() == ref_log
            assert np.array_equal(img, ref) if exact else np.abs(img.astype(int) - ref.astype(int)).max() <= 1


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['orthographic', 'equirectangular'])
def test_factors_and_adaptive_frames_are_those_of_the_camera_rays(kind, env, log):
    w, h = 48, 30
    for sc, exact in _ref_scenes():
        param = projections(sc)[0 if kind == 'orthographic' else 1][1]
        cam = cams_for(sc, kind)[0]
        with _dev(sc, kind, param, cam=cam) as ds:
            plain = ds.render_float(w, h)
            ref1 = _rays_frame(ds, w, h)
            assert ds.counters()['primary_rays'] == w * h
            if exact:
                assert same_bits(plain, ref1), (kind, 1)
            else:
                assert np.abs(plain - ref1).max() <= 1e-5
            full = {}
            for s in (2, 3, 4, 8):
                ds.set_supersampling(s)
                img = ds.render_float(w, h)
                assert ds.counters()['primary_rays'] == w * h * s * s
                ref = _rays_frame(ds, w, h, s)
                if exact and s != 3:
                    assert same_bits(img, ref), (kind, s)
                else:
                    assert np.abs(img - ref).max() <= 1e-5, (kind, s)
                full[s] = img
            ds.set_supersampling(2)
            ds.set_supersampling_threshold(4 / 255)
            img = ds.render_float(w, h)
            mask, count = ds.refine_mask()
            assert 0 < count < w * h
            want = np.where(mask[..., None] != 0, full[2], plain)
            if exact:
                assert same_bits(img, want)
            else:
                assert np.abs(img - want).max() <= 1e-5
        assert log()


def _strips(ds, fmt, world, torch):
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
@pytest.mark.parametrize('kind', ['orthographic', 'equirectangular'])
@pytest.mark.parametrize('s,t', [(1, None), (2, None), (2, 4 / 255)], ids=['f1', 'f2', 'adaptive'])
def test_every_route_gives_the_same_frame(kind, s, t, env, log):
    import torch
    from ntracer_b200.backend import DeviceGroup
    sc = _ggs('refl_transp')
    param = projections(sc)[0 if kind == 'orthographic' else 1][1]
    cam = cams_for(sc, kind)[0]
    w, h = 320, 288                     # 9 tile rows: the slab path runs and the interleaves are ragged
    fmt = _capi.make_image_format(w, h, _capi.RGB8)

    def same(a, what, tol=1):
        d = np.abs(np.asarray(a, np.int32).reshape(h, fmt.pitch) - want.astype(np.int32).reshape(h, fmt.pitch)).max()
        assert d <= tol, (kind, s, t, what, d)

    with _dev(sc, kind, param, s, t, cam) as ds:
        fl = ds.render_float(w, h)
        want = ol.pack(fmt, fl)
        same(ds.render(fmt), 'ntr_render, slabs + staging')
        pinned = torch.zeros(fmt.pitch * h, dtype=torch.uint8).pin_memory()
        same(ds.render(fmt, pinned.numpy()), 'ntr_render, pinned')
        dev = torch.zeros(fmt.pitch * h, dtype=torch.uint8, device='cuda')
        ds.render_device(fmt, dev.data_ptr(), dev.numel())
        torch.cuda.synchronize()
        same(dev.cpu().numpy(), 'ntr_render_device')
        for world in (2, 3):
            same(_strips(ds, fmt, world, torch), 'interleaved tile rows, compact, %d ranks' % world)
        buf = bytearray(fmt.pitch * h)
        tk = ds.render_begin(fmt, buf)
        ds.render_end(tk)
        same(np.frombuffer(buf, np.uint8), 'render_begin/end')
        for x, y in ((0, 0), (w - 1, h - 1), (17, 203), (160, 144)):
            assert np.abs(ds.calculate_color(x, y, w, h) - fl[y, x]).max() <= 1e-5, ('calculate_color', x, y)
        views = ds.render_views(fmt, [cam, cam])
        for v in range(2):
            same(views[v], 'views %d' % v)
    for e in ('NTR_NO_SLABS', 'NTR_NO_STAGING'):
        env(**{e: 1})
        with _dev(sc, kind, param, s, t, cam) as ds:
            same(ds.render(fmt), e)
    env()
    with DeviceGroup(sc, devices=[0, 0]) as grp:
        grp.set_camera(*cam)
        grp.set_supersampling(s)
        grp.set_supersampling_threshold(t)
        grp.set_projection(kind, param)
        same(grp.render(fmt), 'ntr_group_render')
    log()


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['orthographic', 'equirectangular'])
def test_views_and_aovs_under_a_projection(kind, env, log):
    """each view of a batch is its single frame; the AOV ids and depth are primary_hit_ids under the projection, and that hook
    is trace_rays of the camera rays from aabb_distance"""
    FLT_MAX = 3.4028234663852886e38
    for sc, exact in _ref_scenes():
        param = projections(sc)[0 if kind == 'orthographic' else 1][1]
        cams = cams_for(sc, kind, 3)
        w, h = 40, 24
        fmt = _capi.make_image_format(w, h, _capi.RGB8)
        for s in (1, 3):
            with _dev(sc, kind, param, s) as ds:
                frames, a = ds.render_views_aovs(fmt, cams)
                plain = ds.render_views(fmt, cams)
                for k, cam in enumerate(cams):
                    ds.set_camera(*cam)
                    one = ds.render(fmt)
                    d = np.abs(frames[k].astype(int) - one.astype(int)).max()
                    assert d <= (0 if exact else 1) and np.abs(plain[k].astype(int) - one.astype(int)).max() <= (0 if exact else 1)
                    ids, depth = ds.primary_hit_ids(w, h)
                    assert np.array_equal(a['ids'][k], ids) and same_bits(a['depth'][k], depth), (kind, s, k)
                    if s == 1:
                        o, dd = ds.camera_rays(w, h)
                        t0 = orl.ray_colors(sc, o, dd)['t0']
                        want = np.full(w * h, -1, np.int32)
                        wd = np.zeros(w * h, np.float32)
                        for t in np.unique(t0[t0 >= 0]):
                            sel = np.nonzero(t0 == t)[0]
                            i, dist, _ = ds.trace_rays(o[sel], dd[sel], t_near=float(t), t_far=FLT_MAX)
                            want[sel], wd[sel] = i, dist
                        assert np.array_equal(ids.ravel(), want), (kind, k)
                        assert same_bits(depth.ravel(), wd), (kind, k)
    log()


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
@pytest.mark.parametrize('kind', ['giant_opaque', 'giant_general', 'soup_refl'])
def test_projections_on_the_kernel_matrix(dim, generic, kind, env, log):
    """every family against the oracle's colours of the device's own camera rays, plain and instrumented, views AOVs too"""
    from ntracer_b200.backend import DeviceScene
    env(**({'NTR_FORCE_GENERIC': 1} if generic else {}))
    sc = giant_leaf_soup(dim, transparent=kind == 'giant_general') if kind.startswith('giant') else fx.batched_soup(dim, 40)
    w, h = 32, 18
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    with DeviceScene(sc) as ds:
        for proj, param in projections(sc):
            cam = cams_for(sc, proj)[0]
            ds.set_camera(*cam)
            ds.set_projection(proj, param)
            o, d = ds.camera_rays(w, h)
            ref = orl.ray_colors(sc, o, d)
            for instrumented in (False, True):
                ds.set_instrumented(instrumented)
                for s, t in ((1, None), (2, 4 / 255)):
                    ds.set_supersampling(s)
                    ds.set_supersampling_threshold(t)
                    img = ds.render_float(w, h)
                    if s == 1:
                        bad, _ = fx.lsb_stats(img, ref['rgb'].reshape(h, w, 3), exclude=ref['undefined'].reshape(h, w) != 0)
                        assert bad <= 0.001, (dim, generic, kind, proj, instrumented, bad)
                ds.set_supersampling(1)
                ds.set_supersampling_threshold(None)
                frames, a = ds.render_views_aovs(fmt, [cam])
                ids, depth = ds.primary_hit_ids(w, h)
                assert np.array_equal(a['ids'][0], ids) and same_bits(a['depth'][0], depth)
            assert log()
    _RAN.add('matrix')


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['box3', 'box4', 'box9'])
def test_box_scenes(name, env, log):
    sc, _ = fx.load(name)
    w, h = 40, 24
    for kind, param in (('orthographic', 1.5), ('equirectangular', 2 * math.pi)):
        cam = cams_for(sc, kind)[0]
        with _dev(sc, kind, param, cam=cam) as ds:
            img = ds.render_float(w, h)
            assert same_bits(img, _rays_frame(ds, w, h))
            o, d = ds.camera_rays(w, h)
            ref = orl.ray_colors(sc, o, d)
            bad, _ = fx.lsb_stats(img, ref['rgb'].reshape(h, w, 3))
            assert bad <= 0.001
            ds.set_supersampling(4)
            assert same_bits(ds.render_float(w, h), _rays_frame(ds, w, h, 4))
    log()


@pytest.mark.gpu
def test_camera_rays_device_and_errors(env, log):
    import torch
    sc = _ggs(None)
    with _dev(sc, 'equirectangular', 2 * math.pi) as ds:
        o, d = ds.camera_rays(33, 17)
        D = int(sc['dim'])
        to = torch.zeros((33 * 17, D), device='cuda')
        td = torch.zeros((33 * 17, D), device='cuda')
        stream = torch.cuda.Stream()
        ds.camera_rays_device(33, 17, to, td, stream.cuda_stream)
        stream.synchronize()
        assert same_bits(to.cpu().numpy(), o) and same_bits(td.cpu().numpy(), d)
        with pytest.raises(TypeError):
            ds.camera_rays_device(33, 17, to.double(), td)
        with pytest.raises(ValueError):
            ds.camera_rays_device(33, 16, to, td)
        for bad in ((0, 5), (5, 0), (65536, 32768)):
            with pytest.raises(ValueError):
                ds.camera_rays(*bad)
        for kind, param in ((3, 1.0), (1, 0.0), (1, float('nan')), (2, 7.0), (1, float('inf'))):
            with pytest.raises(ValueError):
                _capi.check(ds._lib.ntr_scene_set_projection(ds._h, kind, param))
    log()


@pytest.mark.gpu
def test_abort_of_a_projected_views_call(monkeypatch):
    import threading
    import time
    from ntracer_b200 import bulk
    from ntracer_b200.backend import DeviceScene
    monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    pts = bulk.soup(10, 60000)
    sc = bulk.simplex_scene(pts, max_depth=14)
    sc['cam_origin'] = np.array([0, 0, -3] + [0] * 7, np.float32)
    fmt = _capi.make_image_format(480, 270, _capi.RGB8)
    cams = [(sc['cam_origin'], np.asarray(sc['cam_axes'], np.float32))] * 8
    with DeviceScene(sc) as ds:
        ds.set_projection('equirectangular', 2.0)
        t0 = time.perf_counter()
        ref = ds.render_views(fmt, cams[:2])
        full = (time.perf_counter() - t0) * 4
        result = {}

        def run():
            try:
                ds.render_views(fmt, cams)
                result['rc'] = 'finished'
            except _capi.AbortedError:
                result['rc'] = 'aborted'
        th = threading.Thread(target=run)
        th.start()
        time.sleep(min(0.05, full / 10))
        ds.abort()
        th.join()
        if full > 0.3:
            assert result['rc'] == 'aborted'
        assert np.array_equal(ds.render_views(fmt, cams[:2]), ref)


@pytest.mark.gpu
def test_forced_queue_regrow_under_a_projection(env, log):
    sc = _ggs('refl_transp')
    w, h = 160, 90
    kind, param = projections(sc)[0]                    # the scene fills the view: its bounces outgrow 512 records
    cam = cams_for(sc, kind)[0]
    with _dev(sc, kind, param, 2, cam=cam) as ds:
        ref = ds.render_float(w, h)
    env(NTR_QUEUE_INIT=512)
    with _dev(sc, kind, param, 2, cam=cam) as ds:
        img = ds.render_float(w, h)
        assert ds.counters()['queue_overflows'] >= 1
        assert np.abs(img - ref).max() <= 1e-5
    log()


@pytest.mark.gpu
def test_projected_frames_leave_perspective_frames_alone(env, log):
    """perspective frames before and after projected ones take the same launches and give the same bytes as without them"""
    sc = _ggs('refl_transp')
    fmt = _capi.make_image_format(96, 54, _capi.RGB8)

    def frames(with_proj):
        out = []
        with _dev(sc, s=2, t=4 / 255) as ds:
            for k in range(3):
                if with_proj and k == 2:
                    ds.set_projection('orthographic', 1.0)
                    ds.render(fmt)
                    ds.render_float(200, 100)
                    ds.set_projection('perspective')
                n0 = ds.launch_count()
                img = ds.render(fmt)
                out.append((ds.launch_count() - n0, img.tobytes()))
        return out
    a, b = frames(False), frames(True)
    log()
    assert [x[0] for x in a] == [x[0] for x in b]
    assert all(np.abs(np.frombuffer(x[1], np.uint8).astype(int) - np.frombuffer(y[1], np.uint8).astype(int)).max() <= 1
               for x, y in zip(a, b))


@pytest.mark.gpu
def test_stream_renderer_under_a_projection():
    from ntracer_b200 import BlockingRenderer, Channel, ImageFormat, StreamRenderer
    nt, scene = _box_scene()
    scene.set_projection('equirectangular')
    scene.set_supersampling(2)
    w, h = 128, 64
    fmt = ImageFormat(w, h, [Channel(8, 1, 0, 0), Channel(8, 0, 1, 0), Channel(8, 0, 0, 1)])
    r = StreamRenderer()
    bufs = [bytearray(w * h * 3) for _ in range(2)]
    tickets = [r.submit(b, fmt, scene) for b in bufs]
    assert all(r.wait(t) for t in tickets)
    ref = bytearray(w * h * 3)
    assert BlockingRenderer().render(ref, fmt, scene)
    assert bytes(ref) == bytes(bufs[0]) == bytes(bufs[1])
    scene.set_projection('perspective')
    plain = bytearray(w * h * 3)
    assert BlockingRenderer().render(plain, fmt, scene)
    assert bytes(plain) != bytes(ref)


@pytest.mark.gpu
def test_every_projection_build_ran():
    """All 108 NTR_F_PROJ builds (12 per dimension family) and the 9 camera_rays builds appear among this module's launches"""
    if 'matrix' not in _RAN:
        pytest.skip('the projection matrix did not run in this session')
    assert len(PROJ_BUILDS) == 108
    assert PROJ_BUILDS <= _SEEN, sorted(PROJ_BUILDS - _SEEN)
    assert set(FAMILIES) <= _CAM, sorted(set(FAMILIES) - _CAM)
