"""Differential fuzzing of the product's per-ray device code (compiled for the host, tests/emul_lib.py) against the
oracle: random scenes mixing 4-lane batches, single simplexes, hypercubes, hyperspheres, opaque / transparent /
reflective materials, shadows and bounce depths, in 3 to 7 dimensions, through the fixed-dimension and the
run-time-dimension instantiations."""
import numpy as np

from tests import emul_lib as el
from tests import fixtures as fx
from tests import oracle_lib as ol


def test_random_mixed_scenes_match_the_oracle():
    w, h = 48, 27
    defined_scenes = solids = transparent_hits = 0
    for seed in range(120):
        dim = 3 + seed % 5
        sc = fx.fuzz_scene(dim, seed)
        a, mask, cnt_o = ol.render_float(sc, w, h, with_mask=True, with_counters=True)
        b, cnt_e = el.render(sc, w, h)
        g, _ = el.render(sc, w, h, generic=True)
        ok = mask == 0                       # pixels where the reference's own lists stay inside their preallocation (and
                                             # no opaque hit is shaded off its own surface: oracle mask bit 2)
        d = np.abs(a - b).max(axis=2)
        assert (d[ok].max() if ok.any() else 0) <= 2e-5, (seed, dim)
        assert np.mean(d > 1e-3) <= 0.01, (seed, dim)          # and even outside that domain nothing drifts far
        assert np.abs(b - g).max() <= 2e-5, (seed, dim)        # fixed- and run-time-dimension code agree
        if ((mask & 3) == 0).all():
            for k in ('primary_rays', 'reflection_rays', 'shadow_rays', 'shaded_hits'):
                assert cnt_o[k] == cnt_e[k], (seed, dim, k)
            defined_scenes += 1
        solids += cnt_o['solid_tests'] > 0
        transparent_hits += cnt_o['reflection_rays'] > 0
    assert defined_scenes >= 40 and solids >= 40 and transparent_hits >= 60      # the corpus exercises what it claims


def test_random_rays_with_skip_primitives_match_the_oracle():
    """KDNode.intersects / occludes hooks on the same corpus: random rays, random `source` primitives and batch lanes
    to skip (tracer.hpp:998-1001), random light distances."""
    rays = 0
    for seed in range(40):
        dim = 3 + seed % 5
        sc = fx.fuzz_scene(dim, seed)
        rng = np.random.RandomState(seed + 999)
        n = 200
        o = np.zeros((n, dim), np.float32)
        o[:, :3] = rng.uniform(-3, 3, (n, 3))
        o[:, 3:] = rng.uniform(-0.05, 0.05, (n, dim - 3))
        target = np.zeros((n, dim), np.float32)
        target[:, :3] = rng.uniform(-1, 1, (n, 3))
        d = (target - o).astype(np.float32)
        refs = np.unique(sc['leaf_refs'])
        skip_ref = rng.choice(refs, size=n).astype(np.uint32)
        skip_lane = np.where((skip_ref >> 30) == 1, rng.randint(-1, 4, size=n), -1).astype(np.int32)
        light = rng.uniform(0.5, 6, n).astype(np.float32)
        oi, od, ont = ol.trace_rays(sc, o, d, skip_ref=skip_ref, skip_lane=skip_lane)
        oocc, _ = ol.occludes_rays(sc, o, d, light, skip_ref, skip_lane)
        for generic in (False, True):
            ids, dist, nt = el.trace_rays(sc, o, d, skip_ref=skip_ref, skip_lane=skip_lane, generic=generic)
            assert np.array_equal(ids, oi) and np.array_equal(nt, ont), (seed, generic)
            assert np.allclose(dist, od, rtol=1e-6, atol=1e-6)
        occ, _ = el.occludes_rays(sc, o, d, light, skip_ref, skip_lane)
        assert np.array_equal(occ, oocc), seed
        rays += n
        assert (oi >= 0).any()
    assert rays == 8000


def test_chunked_leaf_scan_is_bit_identical_to_the_sequential_one(tmp_path):
    """-DNTR_CHUNKED_LEAVES=1: leaves evaluated chunk by chunk against the state at the start of the chunk and then
    replayed in leaf order (trace_core.cuh: leaf_general_chunked, the groundwork for splitting one ray's leaf scan over
    the lanes of a warp) must give exactly what the item-by-item scan gives -- images, counters, ray hooks."""
    import ctypes as C
    import os
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    base = el.lib()
    variants = []
    for chunk in (3, 32):
        so = str(tmp_path / ('libhostemul_chunk%d.so' % chunk))
        subprocess.run(['/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++', '-std=c++17', '-O0', '-fPIC', '-shared',
                        '-fvisibility=hidden', '-I/usr/local/cuda/include', '-Wno-unknown-pragmas', '-DNTR_CHUNKED_LEAVES=1',
                        '-DNTR_CHUNK=%d' % chunk, '-o', so, os.path.join(here, 'host_emul', 'emul.cpp')], check=True)
        variants.append(C.CDLL(so))
    scenes = [fx.fuzz_scene(3 + seed % 5, seed) for seed in range(40)]
    sizes = [(32, 18)] * len(scenes)
    for name, v in (('cell120', 'refl_transp'), ('ggs120', 'refl_transp'), ('solids6', None), ('mixed3', None)):
        sc, g = fx.load(name)
        scenes.append(fx.variant(sc, g, v) if v else sc)
        sizes.append((32, 18))
    mixed, gm = fx.load('mixed3')
    try:
        for sc, (w, h) in zip(scenes, sizes):
            el._lib = base
            a, ca = el.render(sc, w, h)
            for var in variants:
                el._lib = var
                b, cb = el.render(sc, w, h)
                assert np.array_equal(a, b)
                for k in ('reflection_rays', 'shadow_rays', 'shaded_hits', 'node_steps'):
                    assert ca[k] == cb[k], k
                # (a hypercube hit demoted by a stale cutoff is tested again: solid tests may be more)
                assert ca['simplex_tests'] == cb['simplex_tests'], (ca['simplex_tests'], cb['simplex_tests'])
                assert np.array_equal(el.render(sc, w, h, generic=True)[0], a)
        for var in variants:
            el._lib = var
            ids, dist, nt = el.trace_rays(mixed, gm['ray_origins'], gm['ray_dirs'])
            assert np.array_equal(ids, gm['ray_ids']) and np.array_equal(nt, gm['ray_ntrans'])
    finally:
        el._lib = base


def test_warp_synchronous_path_on_an_emulated_warp(tmp_path):
    """trace_warp.cuh is what the render kernels run: the 32 rays of a warp traced together, big leaves split over the
    lanes (coop_leaf_opaque / coop_leaf_general / coop_leaf_occludes), shadow rays of a warp in one occlusion traversal.
    Here it runs on an emulated warp -- 32 host threads, every __shfl_sync / __ballot_sync / __any_sync /
    __reduce_*_sync a rendezvous of the 32 (tests/host_emul/emul.cpp, -DNTR_EMULATE_WARP) -- once with cooperation
    forced onto almost every leaf (leaf minimum 4 items, no overhead term in the cost model) and once with the shipped
    thresholds, and must reproduce the per-ray form (trace_core.cuh, itself checked against the oracle) bit for bit:
    images, ray counters and node steps, and with the shipped thresholds the primitive tests too.  A lane sequence that
    diverged between warp intrinsics would hang here (the test is under a timeout) or change the image.  (The wider sweep -- 200 random scenes at 24x14, the 1,600-item leaves of
    {5/2,3,3} at 48x27 -- was run once with the same result, DESIGN.md section 5.)"""
    import ctypes as C
    import os
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    gxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
    libs = []
    for name, flags in (('forced', ['-DNTR_COOP_LEAF_MIN=4', '-DNTR_COOP_OVERHEAD=0']), ('shipped', [])):
        so = str(tmp_path / ('libhostemul_warp_%s.so' % name))
        subprocess.run([gxx, '-std=c++17', '-O1', '-fPIC', '-shared', '-fvisibility=hidden', '-I/usr/local/cuda/include',
                        '-Wno-unknown-pragmas', '-pthread', '-DNTR_EMULATE_WARP'] + flags +
                       ['-o', so, os.path.join(here, 'host_emul', 'emul.cpp')], check=True)
        libs.append(C.CDLL(so))
    base = el.lib()
    cases = [(fx.fuzz_scene(3 + seed % 5, seed), 16, 10) for seed in range(16)]
    cases += [(fx.batched_soup(5, 60), 16, 10), (fx.batched_soup(10, 40), 12, 8)]      # opaque: batches + singles, reflective
    for name, v, w, h in (('mixed3', None, 24, 18), ('ssc120', 'refl_transp', 16, 9), ('ggs120', 'refl_transp', 24, 14),
                          ('ggs120', 'refl', 16, 9), ('cell120', 'shadows', 16, 9), ('solids6', None, 16, 9)):
        sc, g = fx.load(name)
        cases.append((fx.variant(sc, g, v) if v else sc, w, h))
    general = opaque = 0
    try:
        for sc, w, h in cases:
            el._lib = base
            a, ca = el.render(sc, w, h)
            for lib in libs:
                el._lib = lib
                b, cb = el.render(sc, w, h)
                assert np.array_equal(a, b)
                for k in ('reflection_rays', 'shadow_rays', 'shaded_hits', 'node_steps'):
                    assert ca[k] == cb[k], k
                if lib is libs[1]:
                    # with cooperation forced onto small leaves, lanes also test items the owner's mailbox would skip and
                    # the rest of a chunk behind a shadow ray's blocker: more tests, the same answers
                    for k in ('simplex_tests', 'solid_tests'):
                        assert ca[k] == cb[k], (k, ca[k], cb[k])
            is_general = bool(np.any(sc['materials'][:, 6] < 1)) or len(sc['solids']) > 0
            general += is_general
            opaque += not is_general
    finally:
        el._lib = base
    assert general >= 10 and opaque >= 3
