"""Shading of caller-given primary rays (ntr_render_rays, DeviceScene.render_rays): the colour of arbitrary rays through the
full render pipeline.

CPU tier: the ray-fed primary pass (trace_core.cuh: given_ray_color, as render_rays_kernel runs it) on the host, fed the
camera's own rays, against the plain primary pass (colour bits, bounce records, counters), and whole emulated rays calls
against the oracle's ray_color on rays that exercise the reference's branch rules; the Python surface on a test double.
GPU tier: the kernel matrix against the oracle, camera rays against render_float, every route of a rays call, abort, a
group, the state a rays call must leave alone, and launch-log coverage of the 36 builds."""
import ctypes as C
import re

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_rays_lib as er
from tests import fixtures as fx
from tests import oracle_rays_lib as orl
from tests.test_kernel_matrix import CASE_IDS, CASES, giant_leaf_soup, pass_free
from tests.test_views import GOLDEN_SCENES, _ggs, cameras

FLT_MAX = 3.4028234663852886e38
FAMILIES = (3, 4, 5, 6, 7, 8, 9, 10, 0)
RAY_BUILDS = {(fam, k) for fam in FAMILIES for k in range(4)}
EMUL_TOL = 2e-6                 # the host emulation against the oracle (tests/test_host_emul.py)


def ray_set(sc, n, seed):
    """n rays that exercise the reference's branch rules: origins inside and outside the scene box and inside solids,
    directions with zero components and along the axes, rays aimed at vertices shared by several facets (quirk Q11 ties),
    and directions that are not unit vectors -> (origins, dirs) float32 (n, D)"""
    rng = np.random.default_rng(seed)
    D = int(sc['dim'])
    if int(sc['kind']) == 0:
        lo, hi = np.full(D, -1.0), np.full(D, 1.0)
    else:
        lo, hi = np.asarray(sc['boundary'], np.float64)
    c, e = (lo + hi) / 2, np.maximum((hi - lo) / 2, 1e-3)
    o = np.empty((n, D))
    d = rng.normal(size=(n, D))
    k = n // 6
    o[:k] = c + e * rng.uniform(-0.9, 0.9, (k, D))                    # inside the box
    o[k:] = c + e * rng.uniform(-3, 3, (n - k, D))                      # mostly outside
    solids = np.asarray(sc.get('solids', np.zeros((0, 1))))
    if len(solids):                                                     # at the centres of solids
        m = min(k, 3 * len(solids))
        o[k:k + m] = solids[rng.integers(0, len(solids), m), 1 + 2 * D * D:1 + 2 * D * D + D]
    simplex = np.asarray(sc.get('simplex', np.zeros((0, 1))))
    if len(simplex):                                                    # aimed at vertices (shared by several facets)
        sel = slice(2 * k, 3 * k)
        verts = simplex[rng.integers(0, len(simplex), k), D + 1:2 * D + 1]
        d[sel] = verts - o[sel]
    z = slice(3 * k, 4 * k)                                             # zero components
    d[z] *= rng.random((k, D)) < 0.5
    d[z][np.all(d[z] == 0, axis=1), 0] = 1
    a = slice(4 * k, 5 * k)                                             # along the axes
    d[a] = 0
    d[a, rng.integers(0, D, k)] = rng.choice([-1.0, 1.0], k)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[5 * k:] *= rng.uniform(0.25, 4, (n - 5 * k, 1))                   # not unit
    return o.astype(np.float32), d.astype(np.float32)


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------

def _same_as_plain(r, what):
    assert same_bits(r['plain'], r['rays']), (what, int((r['plain'] != r['rays']).sum()))
    assert r['same_records'] and r['plain_records'] == r['rays_records'], what
    assert r['plain_counters'] == r['rays_counters'], what


@pytest.mark.parametrize('name', GOLDEN_SCENES)
def test_emulated_rays_pass_is_the_plain_pass(name):
    sc, g = fx.load(name)
    for s in [sc] + [fx.variant(sc, g, str(v)) for v in g.get('variants', [])]:
        for cam in cameras(s, 2):
            _same_as_plain(er.vs_plain(s, 32, 18, cam=cam), name)


@pytest.mark.parametrize('dim', [3, 4, 9, 16])
def test_emulated_rays_pass_on_the_giant_leaf_soup(dim):
    for transparent in (False, True):
        sc = giant_leaf_soup(dim, transparent=transparent)
        for generic in ((False, True) if dim <= 10 else (True,)):
            _same_as_plain(er.vs_plain(sc, 24, 12, generic=generic), (dim, transparent, generic))


def _against_oracle(sc, o, d, what, generic=False):
    got = er.render_rays(sc, o, d, generic=generic)
    ref = orl.ray_colors(sc, o, d)
    ok = ref['undefined'] == 0
    a, b = got['rgb'], ref['rgb']
    # equal infinities and NaNs on both sides (rays that start at the centre of a sphere) are equal
    diff = np.where((a == b) | (np.isnan(a) & np.isnan(b)), 0, np.abs(a - b))
    assert diff[ok].max(initial=0) <= EMUL_TOL, what
    assert np.array_equal(got['ids'], ref['ids']), (what, int((got['ids'] != ref['ids']).sum()))
    assert same_bits(got['depth'], ref['dist']), what
    assert ref['counters']['primary_rays'] == len(o)
    # counters over the rays where the reference is defined (elsewhere it may trace other bounces, tracer.hpp quirk Q12)
    cg, cr = (got['counters'], ref['counters']) if ok.all() else \
        (er.render_rays(sc, o[ok], d[ok], generic=generic)['counters'], orl.ray_colors(sc, o[ok], d[ok])['counters'])
    for k in ('reflection_rays', 'shadow_rays', 'node_steps', 'shaded_hits'):
        assert cg[k] == cr[k], (what, k)
    assert not got['normals'][got['ids'] < 0].any(), what
    return got, ref


@pytest.mark.parametrize('name', GOLDEN_SCENES)
def test_emulated_rays_match_the_oracle_on_the_golden_scenes(name):
    sc, g = fx.load(name)
    for i, s in enumerate([sc] + [fx.variant(sc, g, str(v)) for v in g.get('variants', [])]):
        o, d = ray_set(s, 300, i)
        _against_oracle(s, o, d, (name, i))


@pytest.mark.parametrize('dim', [3, 4, 9, 16])
def test_emulated_rays_match_the_oracle_on_the_giant_leaf_soup(dim):
    for transparent in (False, True):
        sc = giant_leaf_soup(dim, transparent=transparent)
        o, d = ray_set(sc, 200, dim)
        _against_oracle(sc, o, d, (dim, transparent), generic=dim > 10)


def test_emulated_rays_match_the_oracle_on_the_fuzz_corpus():
    for seed in range(200):
        sc = fx.fuzz_scene(3 + seed % 5, seed)
        o, d = ray_set(sc, 60, seed)
        _against_oracle(sc, o, d, seed)


def test_the_rays_the_oracle_tests_reach_every_branch():
    """the ray set is what it claims: origins inside and outside the box, misses of the box, zero components"""
    sc, _ = fx.load('mixed3')
    o, d = ray_set(sc, 300, 0)
    ref = orl.ray_colors(sc, o, d)
    assert (ref['t0'] == 0).any() and (ref['t0'] > 0).any() and (ref['t0'] < 0).any()
    assert (ref['ids'] >= 0).any() and (ref['ids'] < 0).any()
    assert (d == 0).any() and not np.allclose(np.linalg.norm(d, axis=1), 1)


# ---- the Python surface on a test double ------------------------------------------------------------------------------

class _FakeRaysLibrary:
    """ntr_render_rays / ntr_group_render_rays answered by the host emulation"""
    def __init__(self, sc):
        self.sc, self.calls = sc, []

    def ntr_render_rays(self, h, n, op, dp, rgbp, aovs):
        D = int(self.sc['dim'])
        self.calls.append(n)
        if n == 0:
            return 0
        o = np.ctypeslib.as_array(C.cast(op, C.POINTER(C.c_float)), (n, D)).copy()
        d = np.ctypeslib.as_array(C.cast(dp, C.POINTER(C.c_float)), (n, D)).copy()
        r = er.render_rays(self.sc, o, d)
        C.memmove(rgbp, r['rgb'].ctypes.data, r['rgb'].nbytes)
        if aovs is not None:
            a = aovs._obj
            for name, src in (('ids', r['ids']), ('depth', r['depth']), ('normals', r['normals'])):
                p = getattr(a, name)
                if p is not None:
                    assert getattr(a, name + '_len') >= src.size
                    C.memmove(p, src.ctypes.data, src.nbytes)
        return 0

    ntr_group_render_rays = ntr_render_rays

    def ntr_scene_destroy(self, h):
        pass

    ntr_group_destroy = ntr_scene_destroy


def _fake_scene(sc):
    from ntracer_b200.backend import DeviceGroup, DeviceScene
    ds, g = DeviceScene.__new__(DeviceScene), DeviceGroup.__new__(DeviceGroup)
    for x in (ds, g):
        x._lib, x._h, x.dim, x.device = _FakeRaysLibrary(sc), C.c_void_p(1), int(sc['dim']), 0
    return ds, g


def test_render_rays_on_the_test_double():
    sc, _ = fx.load('mixed3')
    o, d = ray_set(sc, 50, 1)
    ref = er.render_rays(sc, o, d)
    for x in _fake_scene(sc):
        rgb = x.render_rays(o, d)
        assert rgb.shape == (50, 3) and rgb.dtype == np.float32 and same_bits(rgb, ref['rgb'])
        rgb, a = x.render_rays(o.astype(np.float64), d.tolist(), aovs=('normals', 'ids'))
        assert sorted(a) == ['ids', 'normals'] and same_bits(rgb, ref['rgb'])
        assert a['ids'].dtype == np.int32 and a['ids'].shape == (50,) and np.array_equal(a['ids'], ref['ids'])
        assert a['normals'].shape == (50, 3) and same_bits(a['normals'], ref['normals'])
        _, a = x.render_rays(o, d, aovs=('depth',))
        assert list(a) == ['depth'] and same_bits(a['depth'], ref['depth'])
        empty = x.render_rays(np.zeros((0, 3)), np.zeros((0, 3)))
        assert empty.shape == (0, 3) and x._lib.calls[-1] == 0


def test_render_rays_argument_errors():
    sc, _ = fx.load('mixed3')
    ds, g = _fake_scene(sc)
    o, d = ray_set(sc, 4, 2)
    for x in (ds, g):
        with pytest.raises(ValueError):
            x.render_rays(o[:, :2], d[:, :2])               # another dimension
        with pytest.raises(ValueError):
            x.render_rays(o, d[:3])                         # different counts
        with pytest.raises(ValueError):
            x.render_rays(o.ravel(), d.ravel())             # not n x D
        with pytest.raises(ValueError):
            x.render_rays(o, d, aovs=('colour',))
    assert not ds._lib.calls and not g._lib.calls
    torch = pytest.importorskip('torch')
    t = torch.zeros((4, 3))
    with pytest.raises(TypeError):                          # numpy, not a tensor
        ds.render_rays_device(o, d, t)
    with pytest.raises(TypeError):                          # a CPU tensor
        ds.render_rays_device(torch.from_numpy(o), torch.from_numpy(d), t)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------

_SEEN = set()
_RAN = set()


def _launches(text):
    return [(int(a), int(b)) for a, b in re.findall(r'ntr rays-launch family=(\d+) flags=(\d+) grid=\d+', text)]


@pytest.fixture
def log(monkeypatch, capfd):
    """log() -> the ray-fed launches since the last call (recorded for the coverage test)"""
    monkeypatch.setenv('NTR_LAUNCH_LOG', '1')
    capfd.readouterr()

    def read():
        got = _launches(capfd.readouterr().err)
        _SEEN.update(got)
        return got
    return read


@pytest.fixture
def env(monkeypatch):
    from tests.test_kernel_matrix import SWITCHES

    def set_(**kw):
        for k in SWITCHES + ('NTR_RAYS_PER_LAUNCH', 'NTR_QUEUE_INIT'):
            monkeypatch.delenv(k, raising=False)
        for k, v in kw.items():
            monkeypatch.setenv(k, str(v))
    set_()
    return set_


def _pinned_hits(ds, o, d, t0):
    """ids / depth of ntr_trace_rays(scene, 1, o_i, d_i, t0_i, FLT_MAX), -1 / 0 where t0_i < 0"""
    ids = np.full(len(o), -1, np.int32)
    depth = np.zeros(len(o), np.float32)
    for t in np.unique(t0[t0 >= 0]):
        sel = np.nonzero(t0 == t)[0]
        i, dist, _ = ds.trace_rays(o[sel], d[sel], t_near=float(t), t_far=FLT_MAX)
        ids[sel], depth[sel] = i, dist
    return ids, depth


# The tolerances of the GPU parity tests (tests/test_gpu_parity.py): at most 0.1 % of a camera's rays more than 1 LSB off, and
# at most 3 % where rays sit on the edges the reference's branch rules decide (ray_set: rays through shared vertices, along the
# axes, with zero components).  There the device's contracted arithmetic (FMA) and the oracle's twice-rounded one may take
# different sides of a grazing hit or of a tie, and a reflection then leaves in another direction; the host emulation, which
# runs the same code without contraction, matches the oracle on those rays (the CPU tier).
CAMERA_TOL, EDGE_TOL = 0.001, 0.03


def _check_colours(rgb, ref, what, ids=None, tol=CAMERA_TOL):
    """rays where the reference is undefined and exact-t ties between coincident facets (quirk Q11) aside"""
    skip = ref['undefined'] != 0
    if ids is not None:
        skip |= (ids != ref['ids']) & (ids >= 0) & (ref['ids'] >= 0)
    bad, _ = fx.lsb_stats(rgb[None], ref['rgb'][None], exclude=skip[None])
    assert bad <= tol, (what, bad)


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
@pytest.mark.parametrize('kind', ['giant_opaque', 'giant_general', 'soup_refl'])
def test_rays_on_the_kernel_matrix(dim, generic, kind, env, log):
    from ntracer_b200.backend import DeviceScene
    env(**({'NTR_FORCE_GENERIC': 1} if generic else {}))
    if kind.startswith('giant'):
        sc = giant_leaf_soup(dim, transparent=kind == 'giant_general')
    else:
        sc = fx.batched_soup(dim, 40)
    o, d = ray_set(sc, 700, dim)
    ref = orl.ray_colors(sc, o, d)
    cam = er.vs_plain(sc, 32, 18)               # the camera's rays
    co, cd = cam['origins'], cam['dirs']
    cref = orl.ray_colors(sc, co, cd)
    emu = er.render_rays(sc, co, cd, generic=generic or dim > 10)
    with DeviceScene(sc) as ds:
        pins = _pinned_hits(ds, o, d, ref['t0'])
        for instrumented in (False, True):
            ds.set_instrumented(instrumented)
            rgb, a = ds.render_rays(o, d, aovs=('ids', 'depth', 'normals'))
            assert log(), 'no ray-fed launch'
            what = (dim, generic, kind, instrumented)
            _check_colours(rgb, ref, what, a['ids'], tol=EDGE_TOL)
            assert np.array_equal(a['ids'], pins[0]), (what, int((a['ids'] != pins[0]).sum()))
            assert same_bits(a['depth'], pins[1]), what
            assert not a['normals'][a['ids'] < 0].any(), what
            assert ds.counters()['primary_rays'] == len(o)
            _check_colours(ds.render_rays(co, cd), cref, what)
            cnt = ds.counters()
            if instrumented and kind == 'giant_opaque':     # a single-pass scene: the work equals the host emulation's
                for k in ('node_steps', 'simplex_tests', 'solid_tests', 'shaded_hits', 'shadow_rays'):
                    assert cnt[k] == emu['counters'][k], (what, k, cnt[k], emu['counters'][k])
    _RAN.add('matrix')


@pytest.mark.gpu
@pytest.mark.parametrize('variant', [None, 'refl_transp'])
def test_camera_rays_equal_render_float(variant, env, log):
    """the camera's own primary rays give render_float's colours"""
    from ntracer_b200.backend import DeviceScene
    sc = _ggs(variant)
    if variant is None:
        sc = pass_free(sc)
    w, h = 64, 36
    r = er.vs_plain(sc, w, h)                  # the camera's rays, as the device computes them (primary_ray_of)
    with DeviceScene(sc) as ds:
        img = ds.render_float(w, h)
        rgb = ds.render_rays(r['origins'], r['dirs']).reshape(h, w, 3)
    assert log()
    # the device contracts the ray arithmetic into FMAs where the host rounds twice: the parity tolerance, not bits
    bad, _ = fx.lsb_stats(rgb, img, exclude=fx.center_column_mask(w, h))
    assert bad <= 0.001, bad


@pytest.mark.gpu
@pytest.mark.parametrize('reflective', [False, True], ids=['single_pass', 'passes'])
def test_every_route_of_a_rays_call(reflective, env, log):
    """launch splits, queue regrowth, odd counts, n = 0, the device route on a torch stream, short AOV buffers"""
    import torch
    from ntracer_b200.backend import DeviceScene, aov_struct
    sc = _ggs('refl_transp') if reflective else pass_free(_ggs(None))
    D = int(sc['dim'])
    o, d = ray_set(sc, 1001, 5)
    close = same_bits if not reflective else (lambda a, b: np.abs(np.asarray(a) - np.asarray(b)).max() <= 1e-5)
    with DeviceScene(sc) as ds:
        rgb, a = ds.render_rays(o, d, aovs=('ids', 'depth', 'normals'))
        assert len(log()) == 1
        assert close(ds.render_rays(o[:1], d[:1]), rgb[:1]) and close(ds.render_rays(o[:33], d[:33]), rgb[:33])
        assert len(log()) == 2
        assert ds.render_rays(o[:0], d[:0]).shape == (0, 3)
        assert not log()
        # device tensors on a stream
        t = {k: torch.from_numpy(v).cuda() for k, v in (('o', o), ('d', d))}
        out = torch.full((len(o), 3), 7.0, device='cuda')
        dev_aovs = {'ids': torch.full((len(o),), 7, dtype=torch.int32, device='cuda'),
                    'depth': torch.zeros(len(o), device='cuda'), 'normals': torch.zeros((len(o), D), device='cuda')}
        stream = torch.cuda.Stream()
        ds.render_rays_device(t['o'], t['d'], out, dev_aovs, stream.cuda_stream)
        stream.synchronize()
        assert close(out.cpu().numpy(), rgb)
        for k in a:
            assert np.array_equal(dev_aovs[k].cpu().numpy(), a[k]), k
        with pytest.raises(TypeError):
            ds.render_rays_device(t['o'].double(), t['d'], out)
        with pytest.raises(TypeError):
            ds.render_rays_device(t['o'].cpu(), t['d'], out)
        with pytest.raises(ValueError):
            ds.render_rays_device(t['o'][:, :2].contiguous(), t['d'], out)
        with pytest.raises(ValueError):
            ds.render_rays_device(t['o'], t['d'], out[:-1])
        with pytest.raises(ValueError):                 # a short AOV buffer is refused before any work
            short = aov_struct({'ids': (dev_aovs['ids'].data_ptr(), len(o) - 1)})
            _capi.check(ds._lib.ntr_render_rays_device(ds._h, len(o), t['o'].data_ptr(), t['d'].data_ptr(), out.data_ptr(),
                                                       C.byref(short), None))
        with pytest.raises(ValueError):
            _capi.check(ds._lib.ntr_render_rays(ds._h, len(o), None, d.ctypes.data, rgb.ctypes.data, None))
    log()
    env(NTR_RAYS_PER_LAUNCH=2)
    with DeviceScene(sc) as ds:
        r2, a2 = ds.render_rays(o[:41], d[:41], aovs=('ids', 'depth', 'normals'))
        assert ds.counters()['primary_rays'] == 41
    assert len(log()) == 21                            # 41 rays in launches of 2
    assert close(r2, rgb[:41])
    for k in a:
        assert np.array_equal(a2[k], a[k][:41]), ('split', k)
    if reflective:
        # the camera's rays: every one hits, so their bounces outgrow a queue of 512 records
        cam = er.vs_plain(sc, 64, 36)
        env()
        with DeviceScene(sc) as ds:
            r1, a1 = ds.render_rays(cam['origins'], cam['dirs'], aovs=('ids', 'depth', 'normals'))
            assert ds.counters()['queue_overflows'] == 0
        env(NTR_QUEUE_INIT=512)
        with DeviceScene(sc) as ds:
            r3, a3 = ds.render_rays(cam['origins'], cam['dirs'], aovs=('ids', 'depth', 'normals'))
            assert ds.counters()['queue_overflows'] > 0
        log()
        assert close(r3, r1)
        for k in a:
            assert np.array_equal(a3[k], a1[k]), ('regrow', k)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['box3', 'box4', 'box9'])
def test_box_scene_rays(name, env, log):
    from ntracer_b200.backend import DeviceScene
    sc, _ = fx.load(name)
    o, d = ray_set(sc, 333, 3)
    ref = orl.ray_colors(sc, o, d)
    with DeviceScene(sc) as ds:
        rgb, a = ds.render_rays(o, d, aovs=('ids', 'depth', 'normals'))
    assert log()
    _check_colours(rgb, ref, name)
    assert np.mean(a['ids'] == ref['ids']) >= 0.99
    n = a['normals'][a['ids'] >= 0]
    assert np.array_equal(np.abs(n).sum(-1), np.ones(len(n), np.float32))


@pytest.mark.gpu
def test_abort_of_a_rays_call(monkeypatch):
    import threading
    import time
    from ntracer_b200 import bulk
    from ntracer_b200.backend import DeviceScene
    monkeypatch.setenv('NTR_FORCE_GENERIC', '1')
    pts = bulk.soup(10, 60000)
    sc = bulk.simplex_scene(pts, max_depth=14)
    # 2 M rays from one point through the scene box: every one of them walks the soup
    rng = np.random.default_rng(9)
    lo, hi = np.asarray(sc['boundary'], np.float32)
    o = np.tile(np.array([0, 0, -3] + [0] * 7, np.float32), (2_000_000, 1))
    d = (lo + (hi - lo) * rng.random((2_000_000, 10), dtype=np.float32)) - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    with DeviceScene(sc) as ds:
        t0 = time.perf_counter()
        ref = ds.render_rays(o, d)
        full = time.perf_counter() - t0
        result = {}

        def run():
            try:
                result['rgb'] = ds.render_rays(o, d)
            except _capi.AbortedError:
                result['aborted'] = True
        th = threading.Thread(target=run)
        th.start()
        time.sleep(min(0.05, full / 10))
        ds.abort()
        th.join()
        if full > 0.3:
            assert result.get('aborted'), full
        assert same_bits(ds.render_rays(o[:1000], d[:1000]), ref[:1000])


@pytest.mark.gpu
def test_group_equals_one_device(env, log):
    """A group (one device listed twice on a one-GPU box) equals one device"""
    from ntracer_b200.backend import DeviceGroup, DeviceScene, device_count
    devices = [0, 1] if device_count() >= 2 else [0, 0]
    for sc, exact in ((pass_free(_ggs(None)), True), (_ggs('refl_transp'), False)):
        o, d = ray_set(sc, 999, 4)
        with DeviceScene(sc) as ds:
            ref, ref_a = ds.render_rays(o, d, aovs=('ids', 'depth', 'normals'))
            cnt = ds.counters()
        log()
        with DeviceGroup(sc, devices=devices) as g:
            got, a = g.render_rays(o, d, aovs=('ids', 'depth', 'normals'))
            gcnt = g.counters()
        assert len(log()) == len(devices)
        assert same_bits(got, ref) if exact else np.abs(got - ref).max() <= 1e-5
        for k in a:
            assert np.array_equal(a[k], ref_a[k]), k
        for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert gcnt[k] == cnt[k], k


@pytest.mark.gpu
def test_a_rays_call_leaves_the_frames_alone(env, log):
    """frames rendered before and after a rays call take the same launches and give the same bytes as without it (the rays
    call keeps its own sort sizes and pass cost), and the refine-mask record is left alone"""
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('refl_transp')
    fmt = _capi.make_image_format(96, 54, _capi.RGB8)
    o, d = ray_set(sc, 200000, 6)

    def frames(with_rays):
        out = []
        with DeviceScene(sc) as ds:
            ds.set_supersampling(2)
            ds.set_supersampling_threshold(4 / 255)
            for k in range(3):
                if with_rays and k == 2:
                    mask = ds.refine_mask()
                    ds.render_rays(o, d)
                    m2 = ds.refine_mask()
                    assert np.array_equal(mask[0], m2[0]) and mask[1] == m2[1]
                n0 = ds.launch_count()
                img = ds.render(fmt)
                out.append((ds.launch_count() - n0, img.tobytes()))
        return out
    a, b = frames(False), frames(True)
    log()
    assert [x[0] for x in a] == [x[0] for x in b]
    assert a[0][1] == b[0][1]
    assert all(np.abs(np.frombuffer(x[1], np.uint8).astype(int) - np.frombuffer(y[1], np.uint8).astype(int)).max() <= 1
               for x, y in zip(a, b))


@pytest.mark.gpu
def test_every_rays_build_ran():
    """All 36 builds of render_rays_kernel (4 per dimension family) appear among this module's launches"""
    if 'matrix' not in _RAN:
        pytest.skip('the rays matrix did not run in this session')
    assert RAY_BUILDS <= _SEEN, sorted(RAY_BUILDS - _SEEN)
    assert len(RAY_BUILDS) == 36
