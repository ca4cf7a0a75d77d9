"""Every shipped build of render_pass_kernel, and the tile and ray schedules that carry state from frame to frame.

The host picks one build per pass from the scene and the NTR_* switches (capi.cu: enqueue_frame): 8 base builds per
dimension family (NTR_F_GENERAL x NTR_F_COUNT x NTR_F_WARP), 4 NTR_F_SS and 4 NTR_F_LIST builds, and 4 NTR_F_WIDE builds
in 3..5 dimensions -- 156 in all over the families 3..10 and the run-time family (0).  NTR_LAUNCH_LOG=1 prints one stderr
line per launch naming the build, so the module can check that every one of them ran here.

The scene that reaches them all is the giant-leaf soup: fixtures.batched_soup geometry under a hand-built tree whose two
leaves list every item (bulk.build_kdtree splits every cell of 128 items or more, so it cannot make this tree).  Its
leaves of 256 items or more switch on the warp-form bounce passes, the exact mailbox (transparent variant), heavy-first
sorting and, from 64 tiles on, the longest-first tile order.

Slab and frame-sequence tests render ggs120: a frame cut into slabs runs the slabs side by side on their own streams,
each with a tile schedule of its own."""
import re

import numpy as np
import pytest

from ntracer_b200 import _capi
from tests import emul_lib as el
from tests import fixtures as fx
from tests import oracle_lib as ol
from tests.test_supersampling import box_sum

W, H = 64, 36
SWITCHES = ('NTR_WARP', 'NTR_WIDE', 'NTR_FORCE_GENERIC', 'NTR_TILE_SCHED', 'NTR_HEAVY_FIRST', 'NTR_NO_RAY_SORT',
            'NTR_ADAPTIVE_FETCH', 'NTR_FETCH_SIZES', 'NTR_EXACT_MAILBOX', 'NTR_NO_SLABS', 'NTR_ZEROCOPY', 'NTR_PASS_TIMING',
            'NTR_QUEUE_INIT', 'NTR_NO_STAGING')
F_GENERAL, F_COUNT, F_WARP, F_WIDE, F_SS, F_LIST = 1, 2, 4, 8, 16, 32
FAMILIES = (3, 4, 5, 6, 7, 8, 9, 10, 0)
ALL_BUILDS = ({(fam, fl) for fam in FAMILIES for fl in list(range(8)) + [F_SS | k for k in range(4)] + [F_LIST | k for k in range(4)]}
              | {(fam, F_GENERAL | F_WIDE | k) for fam in (3, 4, 5) for k in (0, 2, 4, 6)})
# (dimension, NTR_FORCE_GENERIC): every fixed family, and the run-time family forced in 4-D and native above 10
CASES = [(d, False) for d in range(3, 11)] + [(4, True), (11, False), (13, False), (16, False)]
CASE_IDS = ['dn%d' % d if g or d > 10 else 'd%d' % d for d, g in CASES]


def giant_leaf_soup(dim, batch=4, transparent=True, n_batches=None):
    """batched_soup geometry under one branch (axis 0 at 0) over two leaves that each list every item, batches first.
    transparent=True: material 1 is transparent and reflective, two reflection passes (the general builds, bounce passes);
    False: every material opaque and no reflections (a single-pass frame of the non-general builds)."""
    if n_batches is None:
        n_batches = 320 if batch == 4 else 256          # leaves of 325 / 261 items: past the 256 of the big-leaf switches
    sc = fx.batched_soup(dim, n_batches, batch=batch)
    n_items = n_batches + 5
    refs = np.array([(1 << 30) | (k * batch) for k in range(n_batches)] + [n_batches * batch + k for k in range(5)], np.uint32)
    split = int(np.float32(0).view(np.uint32))
    sc['nodes'] = np.array([[0, split, 1, 2],
                            [0x80000000 | n_batches, 0, n_items, 0],
                            [0x80000000 | n_batches, n_items, n_items, 0]], np.uint32)
    sc['leaf_refs'] = np.concatenate([refs, refs])
    sc['root'] = np.int64(0)
    mats = sc['materials'].copy()
    params = np.array(sc['params'], np.float64)
    if transparent:
        mats[1, 6] = 0.6
    else:
        mats[1, 7] = 0.0
        params[3] = 0
    sc['materials'], sc['params'] = mats, params
    return sc


def pass_free(sc):
    p = np.array(sc['params'], np.float64)
    p[3] = 0
    return dict(sc, params=p)


def q8_diff(a, b):
    return int(np.abs(np.asarray(a, np.int32) - np.asarray(b, np.int32)).max())


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier: the host emulation of the device code (tests/host_emul) against the oracle
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('dim', [3, 4, 9, 16])
@pytest.mark.parametrize('batch', [4, 8])
def test_emulated_giant_leaf_soup_matches_the_oracle(dim, batch):
    sc = giant_leaf_soup(dim, batch)
    o, ocnt = ol.render_float(sc, W, H, with_counters=True)
    for generic in ((False, True) if batch == 4 and dim <= 10 else (True,)):
        img, cnt = el.render(sc, W, H, generic=generic)
        assert np.abs(img - o).max() <= 1e-6, (dim, batch, generic, float(np.abs(img - o).max()))
        for k in ('reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests'):
            assert cnt[k] == ocnt[k], (dim, batch, generic, k, cnt[k], ocnt[k])


@pytest.mark.parametrize('dim', [3, 4, 7])
@pytest.mark.parametrize('batch', [8, 16])
def test_emulated_batch_widths_8_and_16_match_the_oracle(dim, batch):
    """The layouts of the reference's AVX and AVX-512 builds: the host sends them to the run-time-dimension family."""
    sc = fx.batched_soup(dim, 40, batch=batch)
    o, ocnt = ol.render_float(sc, W, H, with_counters=True)
    img, cnt = el.render(sc, W, H, generic=True)
    assert fx.lsb_stats(img, o)[0] <= 0.001
    for k in ('reflection_rays', 'shadow_rays'):
        assert abs(cnt[k] - ocnt[k]) <= 0.002 * max(ocnt[k], 1) + 2, (k, cnt[k], ocnt[k])


def test_giant_leaf_soup_has_the_tree_the_big_leaf_switches_need():
    sc = giant_leaf_soup(4)
    leaves = sc['nodes'][sc['nodes'][:, 0] & 0x80000000 != 0]
    assert len(leaves) == 2 and (leaves[:, 2] == 325).all() and (leaves[:, 0] & 0x7FFFFFFF == 320).all()
    assert giant_leaf_soup(4, batch=8)['nodes'][1, 2] == 261


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------

_SEEN = set()               # (family, flags) of every render_pass_kernel launch in this module
_RAN = set()                # the producer tests that ran to the end, for the coverage check


def _launches(text):
    return [(int(a), int(b)) for a, b in re.findall(r'ntr launch family=(\d+) flags=(\d+) grid=\d+', text)]


@pytest.fixture(scope='module')
def launch_log():
    mp = pytest.MonkeyPatch()
    mp.setenv('NTR_LAUNCH_LOG', '1')
    yield _SEEN
    mp.undo()


@pytest.fixture
def env(monkeypatch, launch_log):
    """set(**switches): clears every NTR_* switch of SWITCHES and sets the given ones (read when a scene is created)."""
    def set_(**kw):
        for k in SWITCHES:
            monkeypatch.delenv(k, raising=False)
        for k, v in kw.items():
            monkeypatch.setenv(k, str(v))
    set_()
    return set_


@pytest.fixture
def log(capfd, launch_log):
    """log() -> the stderr written since the last call; the launches in it are added to the module's record"""
    def read():
        err = capfd.readouterr().err
        _SEEN.update(_launches(err))
        return err
    return read


def _frames(sc, instrumented, fmt):
    from ntracer_b200.backend import DeviceScene
    with DeviceScene(sc) as ds:
        ds.set_instrumented(instrumented)
        fl = ds.render_float(W, H)
        cnt = ds.counters()
        ids, dist = ds.primary_hit_ids(W, H)
        img = ds.render(fmt)
    return dict(fl=fl, cnt=cnt, ids=ids, dist=dist, img=img)


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
@pytest.mark.parametrize('transparent', [False, True], ids=['opaque', 'general'])
def test_every_form_of_every_family(dim, generic, transparent, env, log):
    """Per-lane and warp-synchronous forms (NTR_WARP=0/1/2), instrumented or not, and the 96-register build in 3..5 D:
    against the oracle, against each other, and the instrumented traversal counts against the host emulation."""
    sc = giant_leaf_soup(dim, transparent=transparent)
    single_pass = not transparent
    fmt = _capi.make_image_format(W, H, _capi.RGB8)
    o, ocnt = ol.render_float(sc, W, H, with_counters=True)
    oids, odist = ol.primary_hit_ids(sc, W, H)
    _, ecnt = el.render(sc, W, H, generic=generic or dim > 10)
    forms = [dict(NTR_WARP=w) for w in (0, 1, 2)]
    if transparent and dim <= 5 and not generic:
        forms += [dict(NTR_WARP=w, NTR_WIDE=1) for w in (0, 1)]
    base = None
    for form in forms:
        plain = None
        for instrumented in (False, True):
            env(**form, **({'NTR_FORCE_GENERIC': 1} if generic else {}))
            r = _frames(sc, instrumented, fmt)
            log()
            what = (dim, generic, transparent, form, instrumented)
            bad, mx = fx.lsb_stats(r['fl'], o)
            assert bad <= 0.001, what + (bad, mx)
            assert fx.id_agreement(r['ids'], oids, r['dist'], odist)[0] >= 0.9999, what
            for k in ('primary_rays', 'reflection_rays', 'shadow_rays'):
                assert abs(r['cnt'][k] - ocnt[k]) <= 0.002 * max(ocnt[k], 1) + 2, what + (k, r['cnt'][k], ocnt[k])
            if instrumented:
                for k in ('node_steps', 'simplex_tests'):
                    assert r['cnt'][k] == ecnt[k], what + (k, r['cnt'][k], ecnt[k])
            else:
                assert r['cnt']['node_steps'] == 0 and r['cnt']['simplex_tests'] == 0, what
            base = base or r
            plain = plain or r
            for ref in (base, plain):           # the first form, and this form uninstrumented
                assert np.array_equal(r['ids'], ref['ids']), what
                for k in ('reflection_rays', 'shadow_rays', 'shaded_hits'):
                    assert r['cnt'][k] == ref['cnt'][k], what + (k, r['cnt'][k], ref['cnt'][k])
                if single_pass:
                    assert np.array_equal(r['img'], ref['img']), what
                else:
                    assert q8_diff(r['img'], ref['img']) <= 1, what
    _RAN.add(('forms', dim, generic, transparent))


@pytest.mark.gpu
@pytest.mark.parametrize('dim,generic', CASES, ids=CASE_IDS)
def test_supersampling_in_every_family(dim, generic, env, log):
    """s = 2 without passes is the box sum of the 2W x 2H view, bit for bit; adaptive at t = 4/255 gives the refined
    pixels the full-SS colour and every other pixel the plain one -- in the non-general and the general builds,
    instrumented or not (the NTR_F_SS and NTR_F_LIST builds)."""
    from ntracer_b200.backend import DeviceScene
    for transparent in (False, True):
        sc = pass_free(giant_leaf_soup(dim, transparent=transparent))
        for instrumented in (False, True):
            env(**({'NTR_FORCE_GENERIC': 1} if generic else {}))
            what = (dim, generic, transparent, instrumented)
            with DeviceScene(sc) as ds:
                ds.set_instrumented(instrumented)
                plain = ds.render_float(W, H)
                big = ds.render_float(2 * W, 2 * H)
                ds.set_supersampling(2)
                full = ds.render_float(W, H)
                ds.set_supersampling_threshold(4 / 255)
                adaptive = ds.render_float(W, H)
                mask, count = ds.refine_mask()
            log()
            assert np.array_equal(full, box_sum(big, 2)), what
            m = mask.astype(bool)
            assert 0 < count == int(m.sum()) < W * H, what + (count,)
            assert np.array_equal(adaptive[m], full[m]) and np.array_equal(adaptive[~m], plain[~m]), what
    _RAN.add(('ss', dim, generic))


@pytest.mark.gpu
@pytest.mark.parametrize('dim', [4, 9])
@pytest.mark.parametrize('batch', [8, 16])
def test_batch_widths_8_and_16_match_the_oracle(dim, batch, env, log):
    from ntracer_b200.backend import DeviceScene
    sc = giant_leaf_soup(dim, batch=batch)
    o, ocnt = ol.render_float(sc, W, H, with_counters=True)
    oids, odist = ol.primary_hit_ids(sc, W, H)
    with DeviceScene(sc) as ds:
        fl = ds.render_float(W, H)
        cnt = ds.counters()
        ids, dist = ds.primary_hit_ids(W, H)
    assert {fam for fam, _ in _launches(log())} == {0}
    assert fx.lsb_stats(fl, o)[0] <= 0.001
    assert fx.id_agreement(ids, oids, dist, odist)[0] >= 0.9999
    for k in ('primary_rays', 'reflection_rays', 'shadow_rays'):
        assert abs(cnt[k] - ocnt[k]) <= 0.002 * max(ocnt[k], 1) + 2, (k, cnt[k], ocnt[k])


# ---- slabs and frame sequences -------------------------------------------------------------------------------------

def _ggs(variant):
    sc, g = fx.load('ggs120')
    return fx.variant(sc, g, variant)


def _pinned(n):
    import torch
    return torch.empty(n, dtype=torch.uint8).pin_memory().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize('w,h', [(256, 1024), (1280, 720)])
def test_slabs_and_frame_sequences_on_every_route(w, h, env, log):
    """A single-pass frame of a scene with giant leaves (ggs120 camlight_lights: the longest-first tile order is on) on
    every ntr_render route and through ntr_render_device and begin/end, over 7 frames of a moving camera: every frame
    is, byte for byte, the packed float frame of a fresh scene at that camera.  The slab routes cut the frame into 4
    slabs on 4 streams, each with its own tile order (3 launches per slab: pass, order, decay)."""
    import torch
    from ntracer_b200 import stream
    from ntracer_b200.backend import DeviceScene
    sc = _ggs('camlight_lights')
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    n = fmt.pitch * h
    cams = stream.rotation_cameras(sc['cam_origin'], sc['cam_axes'], 7)
    want = []
    for k, cam in enumerate(cams):
        with DeviceScene(sc) as ds:
            ds.set_camera(*cam)
            fl = ds.render_float(w, h)
        want.append(ol.pack(fmt, fl))
        if k == 0:
            y0 = h // 2 - 4
            band = ol.render_float(sc, w, h, window=(0, y0, w, y0 + 8))
            assert fx.lsb_stats(fl[y0:y0 + 8], band[y0:y0 + 8], exclude=fx.center_column_mask(w, 8))[0] <= 0.001
    log()
    slabs = min(4, (h + 31) // 32 // 4)

    def check(route, frames):
        for k, img in enumerate(frames):
            assert np.array_equal(np.frombuffer(img, np.uint8)[:n], want[k]), (route, w, h, k)

    for route in ('bytearray', 'pinned', 'no_slabs', 'zerocopy', 'device', 'begin_end'):
        env(**({'NTR_NO_SLABS': 1} if route == 'no_slabs' else {'NTR_ZEROCOPY': 1} if route == 'zerocopy' else {}))
        frames = []
        with DeviceScene(sc) as ds:
            if route == 'begin_end':
                bufs = [bytearray(n), bytearray(n)]
                stream.render_sequence(ds, fmt, cams, bufs, sink=lambda k, b: frames.append(bytes(b)))
            for cam in (cams if route != 'begin_end' else ()):
                ds.set_camera(*cam)
                before = ds.launch_count()
                if route == 'device':
                    out = torch.zeros(n, dtype=torch.uint8, device='cuda')
                    ds.render_device(fmt, out.data_ptr(), n)
                    torch.cuda.synchronize()
                    frames.append(out.cpu().numpy())
                else:
                    dest = bytearray(n) if route in ('bytearray', 'no_slabs') else _pinned(n)
                    frames.append(bytes(ds.render(fmt, dest)))
                launched = _launches(log())
                if route in ('bytearray', 'pinned'):
                    assert len(launched) == slabs and ds.launch_count() - before == 3 * slabs, (route, launched)
                else:
                    assert len(launched) == 1, (route, launched)
        log()
        check(route, frames)


def _pass_log(text):
    """the NTR_PASS_TIMING line of one frame -> (ms between the pass events, rays per bounce pass)"""
    m = re.findall(r'ntr pass ms:([\d. ]+) rays:([\d ]+)', text)
    assert len(m) == 1, text[-2000:]
    return [float(v) for v in m[0][0].split()], [int(v) for v in m[0][1].split()]


@pytest.mark.gpu
@pytest.mark.parametrize('scene', ['ggs120', 'soup'])
def test_state_carried_between_frames(scene, env, log):
    """One scene renders a sequence that changes size, interleaves tile rows, evaluates single pixels and changes the
    reflection depth; every frame equals a fresh scene's first frame (within 1 LSB: bounce passes add in float atomics)
    with the same ray counters.  The launch counts show that the ray sort (+2 per bounce pass whose previous size was
    >= 32768 rays, when the previous frame's passes cost more than 1.5 ns per ray), the tile order (+2) and nothing else
    ran, from the pass sizes and times of the previous frame (NTR_PASS_TIMING)."""
    import torch
    from ntracer_b200.backend import DeviceScene
    if scene == 'ggs120':
        sc, (wa, ha), (wb, hb) = _ggs('refl_transp'), (640, 360), (480, 400)
    else:
        sc, (wa, ha), (wb, hb) = giant_leaf_soup(4), (512, 288), (448, 320)
    depth = int(sc['params'][3])
    shallow = dict(sc, params=np.array([sc['params'][0], sc['params'][1], sc['params'][2], 1, sc['params'][4]]))

    env(NTR_PASS_TIMING=1)
    fresh = {}
    for key, s, w, h in (('a', sc, wa, ha), ('b', sc, wb, hb), ('a1', shallow, wa, ha)):
        with DeviceScene(s) as ds:
            fresh[key] = (ds.render_float(w, h), ds.counters())
    log()

    def same(key, fl, cnt, what):
        ref, rcnt = fresh[key]
        assert q8_diff(fx.quant8(fl), fx.quant8(ref)) <= 1, what
        for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert cnt[k] == rcnt[k], what + (k, cnt[k], rcnt[k])

    state = {'ns': 0.0, 'rays': [], 'sorted': 0}     # what the scene keeps from its last frame with bounce passes

    def note(text, d):
        """one frame's pass log -> the pass cost per ray and the pass sizes the next frame sorts by (capi.cu: frame_collect)"""
        ms, rays = _pass_log(text)
        if sum(rays[:d]):
            state['ns'] = sum(ms[1:]) * 1e6 / sum(rays[:d])
        state['rays'] = rays

    with DeviceScene(sc) as ds:
        def frame(key, w, h, d, what):
            before = ds.launch_count()
            fl = ds.render_float(w, h)
            text = log()
            expect = 1 + d + (2 if ((w + 31) // 32) * ((h + 31) // 32) >= 64 else 0)
            if abs(state['ns'] - 1.5) > 0.15:          # a cost right at the threshold cannot be told apart in the log
                n_sorted = sum(1 for r in state['rays'][:d] if r >= 32768) if state['ns'] > 1.5 else 0
                state['sorted'] += n_sorted
                expect += 2 * n_sorted
                assert ds.launch_count() - before == expect, what + (state, ds.launch_count() - before, expect)
            note(text, d)
            same(key, fl, ds.counters(), what)

        frame('a', wa, ha, depth, ('first',))
        frame('a', wa, ha, depth, ('second',))
        frame('b', wb, hb, depth, ('resized',))
        frame('a', wa, ha, depth, ('back',))
        # interleaved strips of the frame: 2 ranks, compact
        fmt = _capi.make_image_format(wa, ha, _capi.RGB8)
        want = ol.pack(fmt, fresh['a'][0]).reshape(ha, fmt.pitch).astype(np.int32)
        for rank in range(2):
            rows = [ty for ty in range((ha + 31) // 32) if ty % 2 == rank]
            strip = torch.zeros(len(rows) * 32 * fmt.pitch, dtype=torch.uint8, device='cuda')
            ds.render_device(fmt, strip.data_ptr(), strip.numel(), 0, rank, 2, True)
            torch.cuda.synchronize()
            s = strip.cpu().numpy().reshape(len(rows) * 32, fmt.pitch).astype(np.int32)
            for k, ty in enumerate(rows):
                m = min(32, ha - ty * 32)
                assert q8_diff(s[k * 32:k * 32 + m], want[ty * 32:ty * 32 + m]) <= 1, (scene, rank, ty)
            note(log(), depth)
        # single pixels: tiny passes, so the next frame must not sort
        rng = np.random.RandomState(5)
        for _ in range(4):
            x, y = int(rng.randint(wa)), int(rng.randint(ha))
            c = ds.calculate_color(x, y, wa, ha)
            assert q8_diff(fx.quant8(c), fx.quant8(fresh['a'][0][y, x])) <= 1, (scene, x, y)
            note(log(), depth)
        frame('a', wa, ha, depth, ('after pixels',))
        ds.set_params(shallow)
        frame('a1', wa, ha, 1, ('depth 1',))
        ds.set_params(sc)
        frame('a', wa, ha, depth, ('depth back',))
        frame('a', wa, ha, depth, ('last',))
    if scene == 'ggs120':
        assert state['sorted'] >= 2         # star polytopes: 6-16 ns per bounce ray, the sort must have engaged


@pytest.mark.gpu
def test_schedule_switches_change_nothing(env, log):
    """NTR_TILE_SCHED, NTR_HEAVY_FIRST, NTR_NO_RAY_SORT, NTR_ADAPTIVE_FETCH / NTR_FETCH_SIZES only change when a tile or ray
    is traced: the second frame of a view (sorted by the first one's pass sizes) is the default's within 1 LSB, with the
    same ray counters; NTR_EXACT_MAILBOX=0 on the opaque soup is the same picture."""
    from ntracer_b200.backend import DeviceScene
    sc = giant_leaf_soup(4)
    w, h = 512, 288

    def two_frames(**sw):
        env(**sw)
        with DeviceScene(sc) as ds:
            ds.render_float(w, h)
            n0 = ds.launch_count()
            fl = ds.render_float(w, h)
            return fl, ds.counters(), ds.launch_count() - n0

    ref, rcnt, rn = two_frames()
    for sw in (dict(NTR_TILE_SCHED=0), dict(NTR_TILE_SCHED=1), dict(NTR_HEAVY_FIRST=0), dict(NTR_HEAVY_FIRST=1),
               dict(NTR_NO_RAY_SORT=1), dict(NTR_ADAPTIVE_FETCH=1, NTR_FETCH_SIZES='1,2,3')):
        fl, cnt, n = two_frames(**sw)
        assert q8_diff(fx.quant8(fl), fx.quant8(ref)) <= 1, sw
        for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
            assert cnt[k] == rcnt[k], (sw, k, cnt[k], rcnt[k])
        if 'NTR_TILE_SCHED' in sw and sw['NTR_TILE_SCHED'] == 0:
            assert n == rn - 2, (sw, n, rn)
        if 'NTR_NO_RAY_SORT' in sw:
            assert n <= rn, (sw, n, rn)
        if 'NTR_ADAPTIVE_FETCH' in sw:
            assert n >= rn, (sw, n, rn)          # + a ring-bounds kernel per sorted pass
    log()
    opaque = giant_leaf_soup(4, transparent=False)
    fmt = _capi.make_image_format(w, h, _capi.RGB8)
    pics = []
    for mbx in (None, 0):
        env(**({} if mbx is None else {'NTR_EXACT_MAILBOX': mbx}))
        with DeviceScene(opaque) as ds:
            pics.append(ds.render(fmt))
    assert np.array_equal(pics[0], pics[1])


@pytest.mark.gpu
def test_exact_mailbox_forced_on_fuzz_scenes(env, log):
    """NTR_EXACT_MAILBOX=1 on scenes whose leaves fit the bounded mailbox: the same traversal as the bounded mailbox (node
    steps and simplex tests identical, pictures within 1 LSB) and the oracle's pictures.  Against the oracle the counts
    agree to 0.5 %: FMA contraction moves rays that pass near a split plane into other leaves (the host emulation built
    with -ffp-contract=fast -mfma reproduces seed 0's 330,464 tests on the GPU exactly, against the oracle's 330,162)."""
    from ntracer_b200.backend import DeviceScene
    for seed in range(10):
        dim = 3 + seed % 5
        sc = fx.fuzz_scene(dim, seed)
        o, mask, ocnt = ol.render_float(sc, W, H, with_mask=True, with_counters=True)
        out = []
        for mbx in (1, None):
            env(**({} if mbx is None else {'NTR_EXACT_MAILBOX': mbx}))
            with DeviceScene(sc) as ds:
                ds.set_instrumented(True)
                out.append((ds.render_float(W, H), ds.counters()))
        (img, cnt), (bimg, bcnt) = out
        for k in ('reflection_rays', 'shadow_rays', 'shaded_hits', 'node_steps', 'simplex_tests', 'solid_tests'):
            assert cnt[k] == bcnt[k], (seed, dim, k, cnt[k], bcnt[k])
        assert q8_diff(fx.quant8(img), fx.quant8(bimg)) <= 1, (seed, dim)
        d = np.abs(fx.quant8(img) - fx.quant8(o)).max(axis=2)
        clean = mask == 0
        if clean.any():
            assert np.mean(d[clean] > 1) <= 0.005, (seed, dim)
        assert abs(cnt['simplex_tests'] - ocnt['simplex_tests']) <= 0.005 * ocnt['simplex_tests'], \
            (seed, dim, cnt['simplex_tests'], ocnt['simplex_tests'])
    log()


@pytest.mark.gpu
def test_every_build_ran():
    """All 156 (family, flags) builds of render_pass_kernel appear in this module's launch log."""
    need = {('forms', d, g, t) for d, g in CASES for t in (False, True)} | {('ss', d, g) for d, g in CASES}
    if not need <= _RAN:
        pytest.skip('the whole module has to run for the coverage check')
    assert len(ALL_BUILDS) == 156
    missing = sorted(ALL_BUILDS - _SEEN)
    assert not missing, missing
    assert _SEEN <= ALL_BUILDS, sorted(_SEEN - ALL_BUILDS)
