"""Per-pixel AOVs of a views call (ntr_render_views_aovs, ntr_render_views_aovs_device, ntr_group_render_views_aovs,
DeviceScene.render_views_aovs, BlockingRenderer.render_views(..., ids=, depth=, normals=)): for view k and pixel (x, y) the
hit id, depth and shading normal of the pixel's plain (factor-1) primary ray, whatever the supersampling factor or threshold,
with the frames and counters of the same call without AOVs.

CPU tier: the host emulation of the AOV capture (ss_pixel_color with a PrimaryAov) against the oracle's KDNode.intersects
(oracle_lib.trace_ray_full) and primary_hit_ids, with colour bits, bounce records and counters unchanged by the capture; the
sample-(0, 0) shortcut at factors 2, 4 and 8; the Python surface on a test double.
GPU tier (`-m gpu`): ids and depth bit-identical to primary_hit_ids per view, normals against the oracle, frames and counters
equal to render_views, on the kernel matrix's scenes and every route of a views call, and NTR_LAUNCH_LOG=1 coverage of the 36
NTR_F_VIEWS | NTR_F_AOV builds."""
import ctypes as C
import re

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_aov_lib as ea
from tests import fixtures as fx
from tests import oracle_lib as ol
from tests.test_kernel_matrix import CASE_IDS, CASES, giant_leaf_soup, pass_free
from tests.test_views import GOLDEN_SCENES, _box_scene, _fmt, _ggs, cameras, emulated  # noqa: F401 (fixture)

W, H = 32, 18
F_VIEWS, F_AOV = 64, 128
FAMILIES = (3, 4, 5, 6, 7, 8, 9, 10, 0)
AOV_BUILDS = {(fam, F_VIEWS | F_AOV | k) for fam in FAMILIES for k in range(4)}
# Normals on the GPU against the oracle: the device code contracts products and sums into FMAs where the oracle rounds
# twice, so a unit normal's components may differ in their last bits; 1e-5 is a few hundred ulps of a unit vector's
# components and far below any difference between two faces.  The host emulation (no contraction) matches exactly.
GPU_NORMAL_TOL = 1e-5


def oracle_normals(sc, origin, dirs, ids, mask):
    """the oracle's RayIntersection.normal of the hit with id ids[p] of the ray (origin, dirs[p]) at every pixel of mask, and
    the pixels whose ray also passes transparent layers.  There the normal that shades the hit may be another one (reference
    quirk Q12, DESIGN section 4: a later transparent hit or cube test writes into o_hit.normal), and the AOV is that one."""
    out = np.zeros(dirs.shape, np.float32)
    layered = np.zeros(mask.shape, bool)
    for p in zip(*np.nonzero(mask)):
        hits = ol.trace_ray_full(sc, origin, dirs[p])
        mine = [h for h in hits if h[1] == ids[p]]
        assert mine, p
        out[p] = mine[-1][3]
        layered[p] = len(hits) > 1
    return out, layered


def check_against_oracle(sc, cam, r, tol=0.0, what=None):
    """ids / depth of an AOV result r against the oracle's primary_hit_ids, normals against trace_ray_full where ids agree"""
    h, w = r['ids'].shape
    oids, odist = ol.primary_hit_ids(sc, w, h, cam=cam)
    agree, _ = fx.id_agreement(r['ids'], oids, r['depth'], odist)
    assert agree >= 0.999, (what, agree)
    same = (r['ids'] == oids) & (oids >= 0)
    assert np.array_equal(r['depth'][r['ids'] < 0], np.zeros(int((r['ids'] < 0).sum()), np.float32)), what
    assert not r['normals'][r['ids'] < 0].any(), what             # a miss: zeros
    if int(sc['kind']) == 0:            # BoxScene: the axis vector of the face, against the ray
        n = r['normals'][r['ids'] >= 0]
        assert np.array_equal(np.abs(n).sum(-1), np.ones(len(n), np.float32)), what
        assert ((n * r['dirs'][r['ids'] >= 0]).sum(-1) < 0).all(), what
        return
    on, layered = oracle_normals(sc, np.asarray(cam[0], np.float32), r['dirs'], oids, same)
    clean = same & ~layered
    diff = np.abs(on[clean] - r['normals'][clean]).max(initial=0.0)
    assert diff <= tol, (what, diff)
    # simplex normals face the ray (flat ids below the scene's simplex count)
    simplex = same & (oids < len(sc.get('simplex', ())))
    if simplex.any():
        assert ((r['normals'][simplex] * r['dirs'][simplex]).sum(-1) <= 0).all(), what


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------

def _unchanged(r, what):
    """the capture leaves colour bits, bounce records and counters alone (test_views.py: _same_bits)"""
    a, b = r['plain'].view(np.uint32), r['aov'].view(np.uint32)
    assert np.array_equal(a, b), (what, int((a != b).sum()))
    assert r['same_records'] and r['plain_records'] == r['aov_records'], what
    assert r['plain_counters'] == r['aov_counters'], what


@pytest.mark.parametrize('name', GOLDEN_SCENES)
def test_emulated_aovs_on_the_golden_scenes(name):
    sc, g = fx.load(name)
    for s in [sc] + [fx.variant(sc, g, str(v)) for v in g.get('variants', [])]:
        for cam in cameras(s, 2):
            r = ea.aov_pass(s, W, H, cam=cam)
            _unchanged(r, name)
            check_against_oracle(s, cam, r, what=name)


@pytest.mark.parametrize('dim', [3, 4, 9, 16])
def test_emulated_aovs_on_the_giant_leaf_soup(dim):
    for transparent in (False, True):
        sc = giant_leaf_soup(dim, transparent=transparent)
        cam = (sc['cam_origin'], sc['cam_axes'])
        for generic in ((False, True) if dim <= 10 else (True,)):
            r = ea.aov_pass(sc, W, H, generic=generic)
            _unchanged(r, (dim, transparent, generic))
            check_against_oracle(sc, cam, r, what=(dim, transparent, generic))


def test_emulated_aovs_on_the_fuzz_corpus():
    for seed in range(200):
        sc = fx.fuzz_scene(3 + seed % 5, seed)
        r = ea.aov_pass(sc, 16, 9)
        _unchanged(r, seed)
        check_against_oracle(sc, (sc['cam_origin'], sc['cam_axes']), r, what=seed)


def test_simplex_normals_face_the_ray():
    """a simplex's normal is unit(face_normal) turned against the ray: dot(n, dir) <= 0 at every simplex hit"""
    for name in ('cell120', 'ggs120', 'ssc120', 'soup9'):
        sc, _ = fx.load(name)
        r = ea.aov_pass(sc, W, H)
        hit = (r['ids'] >= 0) & (r['ids'] < len(sc['simplex']))
        assert hit.any()
        assert ((r['normals'][hit] * r['dirs'][hit]).sum(-1) <= 0).all(), name
        assert np.allclose(np.linalg.norm(r['normals'][hit], axis=-1), 1, atol=1e-6), name


@pytest.mark.parametrize('ss', [2, 3, 4])
def test_supersampled_aovs_are_the_plain_rays(ss):
    """At any factor the AOVs are those of factor 1, bit for bit (sample (0, 0) at 2 and 4, a traversal of their own at 3),
    and the capture leaves the supersampled colours alone."""
    for name in ('box4', 'cell120', 'mixed3', 'solids6'):
        sc, _ = fx.load(name)
        cam = cameras(sc, 1)[0]
        one = ea.aov_pass(sc, 21, 14, cam=cam)
        r = ea.aov_pass(sc, 21, 14, ss=ss, cam=cam)
        _unchanged(r, (name, ss))
        for k in ('ids', 'depth', 'normals'):
            assert np.array_equal(r[k].view(np.uint32), one[k].view(np.uint32)), (name, ss, k)


@pytest.mark.parametrize('ss', [2, 4, 8])
@pytest.mark.parametrize('w,h', [(64, 36), (63, 35), (17, 40), (40, 17), (1, 1), (1919, 3)])
def test_sample_zero_is_the_plain_ray_at_powers_of_two(ss, w, h):
    """What ss_pixel_color's shortcut rests on: fovI / ss and ss * x - ss * half_w scale exactly, so sample (0, 0) of the
    ss-times-larger view is the plain primary ray bit for bit, for odd and even sizes"""
    rng = np.random.default_rng(ss * 1000 + w + h)
    for dim in (3, 4, 7, 16):
        for _ in range(3):
            axes = np.linalg.qr(rng.normal(size=(dim, dim)))[0].astype(np.float32)
            origin = rng.normal(size=dim).astype(np.float32) * 5
            for fov in (0.8, 1.3, np.pi / 2):
                assert ea.sample0_mismatches(dim, (origin, axes), fov, w, h, ss) == 0, (dim, fov)
    # a factor that is not a power of two does not have that property (hence the separate traversal)
    axes = np.linalg.qr(rng.normal(size=(4, 4)))[0].astype(np.float32)
    assert ea.sample0_mismatches(4, (np.zeros(4, np.float32), axes), 0.8, 64, 36, 3) > 0


# ---- the Python surface on a test double ------------------------------------------------------------------------------

def _install_aovs(lib):
    """+ ntr_render_views_aovs answered by the host emulation: frames as ntr_render_views, AOVs from emul_aov_lib"""
    dev = lib.dev
    lib.aov_calls = []

    def ntr_render_views_aovs(handle, n, optr, aptr, fmt_ref, ptr, size, aovs_ref):
        rc = lib.ntr_render_views(handle, n, optr, aptr, fmt_ref, ptr, size)
        o, a = lib.calls[-1]
        fmt, a_s, D = fmt_ref._obj, aovs_ref._obj, dev.dim
        lib.aov_calls.append({k: getattr(a_s, k) is not None for k in ('ids', 'depth', 'normals')})
        npix = fmt.width * fmt.height
        for k in range(n):
            r = ea.aov_pass(dev.sc, fmt.width, fmt.height, cam=(o[k], a[k]))
            for name, per in (('ids', 1), ('depth', 1), ('normals', D)):
                p = getattr(a_s, name)
                if p is not None:
                    assert getattr(a_s, name + '_len') >= n * npix * per
                    src = np.ascontiguousarray(r[name])
                    C.memmove(p + k * npix * per * 4, src.ctypes.data, src.nbytes)
        return rc
    lib.ntr_render_views_aovs = ntr_render_views_aovs


def test_render_views_with_aovs_on_the_emulated_device(emulated):
    from ntracer_b200.render import BlockingRenderer
    nt, scene = _box_scene()
    fmt = _fmt()
    cams = []
    for k in range(3):
        c = nt.Camera()
        c.translate(nt.Vector.axis(2, -5 - 0.5 * k))
        cams.append(c)
    r = BlockingRenderer()
    plain = bytearray(3 * fmt.pitch * fmt.height)
    assert r.render_views(plain, fmt, scene, cams) is True
    lib = emulated.last._lib
    _install_aovs(lib)
    assert not lib.aov_calls                        # without keywords: ntr_render_views, as before
    n, w, h = 3, fmt.width, fmt.height
    buf = bytearray(len(plain))
    ids = np.full((n, h, w), 7, np.int32)
    depth = np.full((n, h, w), 7, np.float32)
    normals = np.full((n, h, w, 4), 7, np.float32)
    assert r.render_views(buf, fmt, scene, cams, ids=ids, depth=depth, normals=normals) is True
    assert bytes(buf) == bytes(plain)
    assert lib.aov_calls[-1] == {'ids': True, 'depth': True, 'normals': True}
    for k, c in enumerate(cams):
        ref = ea.aov_pass(emulated.last.sc, w, h, cam=(c._origin, c._axes))
        assert np.array_equal(ids[k], ref['ids']) and np.array_equal(depth[k], ref['depth'])
        assert np.array_equal(normals[k], ref['normals'])
    assert (ids >= 0).any() and (ids == -1).any()
    # subsets, and any writable buffer of the right size
    d2 = bytearray(4 * n * h * w)
    assert r.render_views(bytearray(len(plain)), fmt, scene, cams, depth=d2)
    assert lib.aov_calls[-1] == {'ids': False, 'depth': True, 'normals': False}
    assert np.array_equal(np.frombuffer(d2, np.float32).reshape(n, h, w), depth)
    assert scene.locked == 0


def test_render_views_aov_argument_errors(emulated):
    from ntracer_b200.render import BlockingRenderer
    nt, scene = _box_scene()
    fmt = _fmt()
    r = BlockingRenderer()
    cams = [nt.Camera(), nt.Camera()]
    n, w, h = 2, fmt.width, fmt.height
    buf = bytearray(n * fmt.pitch * h)
    with pytest.raises(ValueError):                 # short buffers
        r.render_views(buf, fmt, scene, cams, ids=np.zeros((n, h, w - 1), np.int32))
    with pytest.raises(ValueError):
        r.render_views(buf, fmt, scene, cams, normals=np.zeros((n, h, w, 3), np.float32))
    with pytest.raises(TypeError):                  # wrong dtypes
        r.render_views(buf, fmt, scene, cams, ids=np.zeros((n, h, w), np.float32))
    with pytest.raises(TypeError):
        r.render_views(buf, fmt, scene, cams, depth=np.zeros((n, h, w), np.float64))
    with pytest.raises(TypeError):                  # not a buffer
        r.render_views(buf, fmt, scene, cams, depth=5)
    with pytest.raises(BufferError):                # read-only
        r.render_views(buf, fmt, scene, cams, depth=bytes(4 * n * h * w))
    with pytest.raises(TypeError):                  # keyword-only
        r.render_views(buf, fmt, scene, cams, np.zeros((n, h, w), np.int32))
    assert scene.locked == 0


def test_device_scene_aov_names():
    from ntracer_b200.backend import _new_aovs, aov_shape
    fmt = _capi.make_image_format(6, 4, _capi.RGB8)
    arrays, a = _new_aovs(('normals', 'ids'), 2, fmt, 5)
    assert sorted(arrays) == ['ids', 'normals']
    assert arrays['ids'].shape == (2, 4, 6) and arrays['ids'].dtype == np.int32
    assert arrays['normals'].shape == (2, 4, 6, 5) and arrays['normals'].dtype == np.float32
    assert a.depth is None and a.ids_len == 48 and a.normals_len == 240
    assert aov_shape('depth', 3, fmt, 4) == (3, 4, 6)
    with pytest.raises(ValueError):
        _new_aovs(('colour',), 1, fmt, 4)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------

_SEEN = set()
_RAN = set()


def _launches(text):
    return [(int(a), int(b)) for a, b in re.findall(r'ntr launch family=(\d+) flags=(\d+) grid=\d+', text)]


@pytest.fixture
def log(monkeypatch, capfd):
    """log(aov_call) -> the launches since the last call; an AOV call's NTR_F_AOV launches are recorded, any other call may
    launch none"""
    monkeypatch.setenv('NTR_LAUNCH_LOG', '1')
    capfd.readouterr()

    def read(aov_call):
        got = _launches(capfd.readouterr().err)
        aov = {x for x in got if x[1] & F_AOV}
        if aov_call:
            assert aov, 'an AOV call launched no NTR_F_AOV build'
            _SEEN.update(aov)
        else:
            assert not aov, aov
        return got
    return read


@pytest.fixture
def env(monkeypatch):
    from tests.test_kernel_matrix import SWITCHES

    def set_(**kw):
        for k in SWITCHES + ('NTR_VIEWS_PER_LAUNCH', 'NTR_QUEUE_INIT'):
            monkeypatch.delenv(k, raising=False)
        for k, v in kw.items():
            monkeypatch.setenv(k, str(v))
    set_()
    return set_


def _hit_ids(ds, fmt, cams):
    """primary_hit_ids per view -> (ids, depth) [n, h, w]"""
    ids, depth = [], []
    for o, a in cams:
        ds.set_camera(o, a)
        i, d = ds.primary_hit_ids(fmt.width, fmt.height)
        ids.append(np.asarray(i).reshape(fmt.height, fmt.width))
        depth.append(np.asarray(d).reshape(fmt.height, fmt.width))
    return np.stack(ids), np.stack(depth)


def _check_frames(got, ref, exact, what):
    if exact:
        assert np.array_equal(got, ref), (what, int((got != ref).sum()))
    else:
        assert np.abs(got.astype(np.int32) - ref.astype(np.int32)).max() <= 1, what


def _check_aovs(sc, cams, aovs, ref_ids, ref_depth, what, normals_vs_oracle=True):
    assert np.array_equal(aovs['ids'], ref_ids), (what, int((aovs['ids'] != ref_ids).sum()))
    assert np.array_equal(aovs['depth'].view(np.uint32), ref_depth.view(np.uint32)), what
    if not normals_vs_oracle:
        return
    n, h, w = ref_ids.shape
    for k, cam in enumerate(cams):
        r = ea.aov_pass(sc, w, h, cam=cam)          # the plain rays' directions (and the host's own AOVs)
        r = dict(r, ids=aovs['ids'][k], depth=aovs['depth'][k], normals=aovs['normals'][k])
        check_against_oracle(sc, cam, r, tol=GPU_NORMAL_TOL, what=(what, k))


def _run(ds, fmt, cams, what, exact, instrumented=False):
    """render_views vs render_views_aovs on one scene: frames, counters, ids / depth vs primary_hit_ids"""
    ref = ds.render_views(fmt, cams)
    cnt = ds.counters()
    frames, aovs = ds.render_views_aovs(fmt, cams)
    _check_frames(frames, ref, exact, what)
    got = ds.counters()
    keys = ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits') + \
           (('node_steps', 'simplex_tests', 'solid_tests') if instrumented else ())
    for k in keys:
        assert got[k] == cnt[k], (what, k, got[k], cnt[k])
    return frames, aovs


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
@pytest.mark.parametrize('kind', ['giant_opaque', 'giant_general', 'soup_refl'])
def test_aovs_on_the_kernel_matrix(dim, generic, kind, env, log):
    from ntracer_b200.backend import DeviceScene
    env(**({'NTR_FORCE_GENERIC': 1} if generic else {}))
    if kind.startswith('giant'):
        sc = giant_leaf_soup(dim, transparent=kind == 'giant_general')
    else:
        sc = fx.batched_soup(dim, 40)
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    cams = cameras(sc, 3)
    with DeviceScene(sc) as ds:
        ref_ids, ref_depth = _hit_ids(ds, fmt, cams)
        for instrumented in (False, True):
            ds.set_instrumented(instrumented)
            log(False)
            _, aovs = _run(ds, fmt, cams, (dim, generic, kind, instrumented), kind != 'soup_refl', instrumented)
            log(True)
            _check_aovs(sc, cams, aovs, ref_ids, ref_depth, (dim, generic, kind), normals_vs_oracle=not instrumented)
    _RAN.add('matrix')


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['box3', 'box4', 'box6', 'box9'])
def test_box_scene_aovs(name, env, log):
    from ntracer_b200.backend import DeviceScene
    sc, _ = fx.load(name)
    fmt = _capi.make_image_format(W, 48, _capi.RGB8)
    d = int(sc['dim'])
    cams = [(np.array([0, 0, -5 - 0.5 * k] + [0] * (d - 3), np.float32), np.eye(d, dtype=np.float32)) for k in range(2)]
    cams += cameras(dict(sc, cam_origin=cams[0][0], cam_axes=cams[0][1]), 3, 12)[1:]
    with DeviceScene(sc) as ds:
        ref_ids, ref_depth = _hit_ids(ds, fmt, cams)
        for ss in (1, 2, 3):
            ds.set_supersampling(ss)
            _, aovs = _run(ds, fmt, cams, (name, ss), True)
            log(True)
            _check_aovs(sc, cams, aovs, ref_ids, ref_depth, (name, ss))


@pytest.mark.gpu
@pytest.mark.parametrize('reflective', [False, True], ids=['single_pass', 'passes'])
def test_supersampled_and_adaptive_aovs(reflective, env, log):
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('refl_transp') if reflective else pass_free(_ggs(None))
    fmt = _capi.make_image_format(48, 30, _capi.RGB8)
    cams = cameras(sc, 3)
    with DeviceScene(sc) as ds:
        ref_ids, ref_depth = _hit_ids(ds, fmt, cams)
        for ss in (2, 3):
            ds.set_supersampling(ss)
            _, aovs = _run(ds, fmt, cams, ss, not reflective)
            log(True)
            _check_aovs(sc, cams, aovs, ref_ids, ref_depth, ss, normals_vs_oracle=ss == 2)
        ds.set_supersampling(3)
        ds.set_supersampling_threshold(4 / 255)
        ref = ds.render_views(fmt, cams)
        cnt = ds.counters()
        mask = ds.refine_mask()
        log(False)
        frames, aovs = ds.render_views_aovs(fmt, cams)
        log(True)                   # the AOVs of each view: a one-view NTR_F_AOV launch at factor 1
        _check_frames(frames, ref, not reflective, 'adaptive')
        assert ds.counters()['primary_rays'] == cnt['primary_rays']
        m, c = ds.refine_mask()
        assert np.array_equal(m, mask[0]) and c == mask[1]
        _check_aovs(sc, cams, aovs, ref_ids, ref_depth, 'adaptive', normals_vs_oracle=False)


@pytest.mark.gpu
@pytest.mark.parametrize('reflective', [False, True], ids=['single_pass', 'passes'])
def test_every_route_of_an_aov_call(reflective, env, log):
    """pageable and pinned host destinations, device tensors on a stream, launch splits and queue regrowth, subsets"""
    import torch
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('refl_transp') if reflective else pass_free(_ggs(None))
    w, h, pitch = 40, 24, 128
    fmt = _capi.make_image_format(w, h, _capi.RGB8, pitch)
    cams = cameras(sc, 5)
    n, D = len(cams), int(sc['dim'])
    with DeviceScene(sc) as ds:
        ref_ids, ref_depth = _hit_ids(ds, fmt, cams)
        frames, aovs = _run(ds, fmt, cams, 'host', not reflective)
        log(True)
        _check_aovs(sc, cams, aovs, ref_ids, ref_depth, 'host')
        # pinned destinations
        pinned = {k: torch.from_numpy(np.zeros_like(v)).pin_memory() for k, v in aovs.items()}
        pf = torch.zeros(n * pitch * h, dtype=torch.uint8).pin_memory()
        a = {k: (t.data_ptr(), t.numel()) for k, t in pinned.items()}
        from ntracer_b200.backend import aov_struct
        o, ax = np.stack([c[0] for c in cams]).astype(np.float32), np.stack([c[1] for c in cams]).astype(np.float32)
        _capi.check(ds._lib.ntr_render_views_aovs(ds._h, n, o.ctypes.data, ax.ctypes.data, C.byref(fmt), pf.data_ptr(),
                                                  pf.numel(), C.byref(aov_struct(a))))
        _check_frames(pf.numpy().reshape(n, -1), frames, not reflective, 'pinned')
        for k in aovs:
            assert np.array_equal(pinned[k].numpy().view(np.uint32), aovs[k].view(np.uint32)), ('pinned', k)
        log(True)
        # device tensors on a stream
        dev = torch.zeros((n, h, pitch), dtype=torch.uint8, device='cuda')
        dt = {'ids': torch.full((n, h, w), 5, dtype=torch.int32, device='cuda'),
              'depth': torch.full((n, h, w), 5, dtype=torch.float32, device='cuda'),
              'normals': torch.full((n, h, w, D), 5, dtype=torch.float32, device='cuda')}
        stream = torch.cuda.Stream()
        ds.render_views_aovs_device(fmt, cams, dev.data_ptr(), dev.numel(), dt, stream.cuda_stream)
        stream.synchronize()
        log(True)
        _check_frames(dev.cpu().numpy().reshape(n, -1), frames, not reflective, 'device')
        for k in aovs:
            assert np.array_equal(dt[k].cpu().numpy().view(np.uint32), aovs[k].view(np.uint32)), ('device', k)
        # a subset
        _, sub = ds.render_views_aovs(fmt, cams, aovs=('depth',))
        assert list(sub) == ['depth'] and np.array_equal(sub['depth'], aovs['depth'])
        log(True)
        with pytest.raises(ValueError):             # short buffers are refused before any work
            ds.render_views_aovs_device(fmt, cams, dev.data_ptr(), dev.numel(), {'ids': (dt['ids'].data_ptr(), n * h * w - 1)})
        with pytest.raises(ValueError):
            ds.render_views_aovs_device(fmt, cams, dev.data_ptr(), dev.numel(), {'normals': (dt['normals'].data_ptr(), n * h * w * D - 1)})
    env(NTR_VIEWS_PER_LAUNCH=2)
    with DeviceScene(sc) as ds:
        f2, a2 = ds.render_views_aovs(fmt, cams)
    got = log(True)
    assert sum(1 for x in got if x[1] & F_AOV) == 3            # 5 views in launches of 2
    _check_frames(f2, frames, not reflective, 'split')
    for k in aovs:
        assert np.array_equal(a2[k].view(np.uint32), aovs[k].view(np.uint32)), ('split', k)
    if reflective:
        env(NTR_QUEUE_INIT=512)
        with DeviceScene(sc) as ds:
            f3, a3 = ds.render_views_aovs(fmt, cams)
            assert ds.counters()['queue_overflows'] > 0
        log(True)
        _check_frames(f3, frames, False, 'regrow')
        for k in aovs:
            assert np.array_equal(a3[k].view(np.uint32), aovs[k].view(np.uint32)), ('regrow', k)


@pytest.mark.gpu
def test_abort_of_an_aov_call(monkeypatch):
    """Following test_views.py's abort test, with all three AOVs"""
    import threading
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
    ids = np.zeros((3, 540, 960), np.int32)
    depth = np.zeros((3, 540, 960), np.float32)
    normals = np.zeros((3, 540, 960, 10), np.float32)
    kw = dict(ids=ids, depth=depth, normals=normals)
    r = BlockingRenderer()
    t0 = time.perf_counter()
    assert r.render_views(buf, fmt, scene, cams, **kw) is True
    full = time.perf_counter() - t0
    ref = ids.copy()
    result = {}
    th = threading.Thread(target=lambda: result.setdefault('rc', r.render_views(buf, fmt, scene, cams, **kw)))
    t0 = time.perf_counter()
    th.start()
    time.sleep(min(0.05, full / 10))
    r.signal_abort()
    th.join()
    aborted = time.perf_counter() - t0
    if full > 0.3:
        assert result['rc'] is False
        assert aborted < 0.8 * full
    assert r.render_views(buf, fmt, scene, cams, **kw) is True
    assert np.array_equal(ids, ref)
    ds.close()


@pytest.mark.gpu
def test_group_aovs(env, log):
    """A group (one device listed twice on a one-GPU box) equals single-device render_views_aovs"""
    from ntracer_b200.backend import DeviceGroup, DeviceScene, device_count
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    devices = [0, 1] if device_count() >= 2 else [0, 0]
    for sc, exact in ((pass_free(_ggs(None)), True), (_ggs('refl_transp'), False)):
        cams = cameras(sc)
        with DeviceScene(sc) as ds:
            ref, ref_aovs = ds.render_views_aovs(fmt, cams)
            cnt = ds.counters()
        log(True)
        with DeviceGroup(sc, devices=devices) as g:
            got, aovs = g.render_views_aovs(fmt, cams)
            gcnt = g.counters()
        launches = [x for x in log(True) if x[1] & F_AOV]
        assert len(launches) == len(devices)
        _check_frames(got, ref, exact, 'group')
        for k in aovs:
            assert np.array_equal(aovs[k].view(np.uint32), ref_aovs[k].view(np.uint32)), ('group', k)
        for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert gcnt[k] == cnt[k], k
        with DeviceGroup(sc, devices=devices) as g:       # adaptive: view after view, the AOVs on the first device
            g.set_supersampling(2)
            g.set_supersampling_threshold(4 / 255)
            _, aa = g.render_views_aovs(fmt, cams[:2])
        log(True)
        for k in aovs:
            assert np.array_equal(aa[k].view(np.uint32), ref_aovs[k][:2].view(np.uint32)), ('group adaptive', k)


@pytest.mark.gpu
def test_every_aov_build_ran():
    """All 36 NTR_F_VIEWS | NTR_F_AOV builds (4 per dimension family) appear among this module's AOV calls"""
    if 'matrix' not in _RAN:
        pytest.skip('the AOV matrix did not run in this session')
    assert AOV_BUILDS <= _SEEN, sorted(AOV_BUILDS - _SEEN)
    assert len(AOV_BUILDS) == 36
