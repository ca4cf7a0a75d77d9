"""ntracer_b200.pygame_render (the reference's lib/ntracer/pygame_render.py on this backend) without pygame: a small
stand-in module provides what the front end touches (Surface queries, the event queue, the quit hook).  The channel
lists are compared with values recorded from the reference's own channels_from_surface and, when NTRACER_REFERENCE
names the reference's source tree, with that function run on the same stand-in; the renderer is driven end to end on
the emulated device of tests/test_facade_emulated.py (CPU tier: Python side of the C ABI)."""
import importlib
import os
import sys
import threading
import types

import numpy as np
import pytest

REF = os.path.join(os.environ['NTRACER_REFERENCE'], 'lib', 'ntracer', 'pygame_render.py') if os.environ.get('NTRACER_REFERENCE') else None


class FakeSurface:
    def __init__(self, w, h, nbytes, masks, shifts, losses, pad=0):
        self.w, self.h, self.nbytes, self.masks, self.shifts, self.losses = w, h, nbytes, masks, shifts, losses
        self.pitch = w * nbytes + pad
        self.buf = bytearray(b'\xEE' * (self.pitch * h))

    def get_bytesize(self): return self.nbytes
    def get_bitsize(self): return self.nbytes * 8
    def get_masks(self): return self.masks
    def get_shifts(self): return self.shifts
    def get_losses(self): return self.losses
    def get_width(self): return self.w
    def get_height(self): return self.h
    def get_pitch(self): return self.pitch
    def get_view(self): return self.buf


FORMATS = {
    # name: (bytes, masks, shifts, losses), expected channels as (bits, f_r, f_g, f_b, f_c)
    'xrgb8888': ((4, (0xFF0000, 0xFF00, 0xFF, 0), (16, 8, 0, 0), (0, 0, 0, 8)),
                 [(8, 0, 0, 0, 0), (8, 1, 0, 0, 0), (8, 0, 1, 0, 0), (8, 0, 0, 1, 0)]),
    'rgba8888': ((4, (0xFF000000, 0xFF0000, 0xFF00, 0xFF), (24, 16, 8, 0), (0, 0, 0, 0)),
                 [(8, 1, 0, 0, 0), (8, 0, 1, 0, 0), (8, 0, 0, 1, 0), (8, 0, 0, 0, 1)]),
    'bgr888': ((3, (0xFF, 0xFF00, 0xFF0000, 0), (0, 8, 16, 0), (0, 0, 0, 8)),
               [(8, 0, 0, 1, 0), (8, 0, 1, 0, 0), (8, 1, 0, 0, 0)]),
    'rgb565': ((2, (0xF800, 0x7E0, 0x1F, 0), (11, 5, 0, 0), (3, 2, 3, 8)),
               [(5, 1, 0, 0, 0), (6, 0, 1, 0, 0), (5, 0, 0, 1, 0)]),
    'xbgr1555': ((2, (0x1F, 0x3E0, 0x7C00, 0), (0, 5, 10, 0), (3, 3, 3, 8)),
                 [(1, 0, 0, 0, 0), (5, 0, 0, 1, 0), (5, 0, 1, 0, 0), (5, 1, 0, 0, 0)]),
}


@pytest.fixture
def fake_pygame(monkeypatch):
    pg = types.ModuleType('pygame')
    pg.USEREVENT, pg.NUMEVENTS, pg.LIL_ENDIAN, pg.BIG_ENDIAN = 24, 32, 1234, 4321
    pg.get_sdl_byteorder = lambda: pg.LIL_ENDIAN
    pg.posted, pg.arrived, pg.quit_hooks = [], threading.Event(), []

    class Event:
        def __init__(self, type, **attrs):
            self.type = type
            self.__dict__.update(attrs)
    ev = types.ModuleType('pygame.event')
    ev.Event = Event
    ev.post = lambda e: (pg.posted.append(e), pg.arrived.set())
    pg.event = ev
    pg.register_quit = pg.quit_hooks.append
    monkeypatch.setitem(sys.modules, 'pygame', pg)
    monkeypatch.setitem(sys.modules, 'pygame.event', ev)
    sys.modules.pop('ntracer_b200.pygame_render', None)
    mod = importlib.import_module('ntracer_b200.pygame_render')
    yield pg, mod
    sys.modules.pop('ntracer_b200.pygame_render', None)


def _tuples(channels):
    return [(c.bit_size, float(c.f_r), float(c.f_g), float(c.f_b), float(c.f_c)) for c in channels]


def test_channels_from_surface(fake_pygame):
    pg, mod = fake_pygame
    ref_fn = None
    if REF and os.path.exists(REF):
        # the reference's own function, executed on the same stand-in (its `ntracer.render.Channel` replaced by a recorder)
        class Chan:
            def __init__(self, bit_size, f_r, f_g, f_b, f_c=0):
                self.bit_size, self.f_r, self.f_g, self.f_b, self.f_c = bit_size, f_r, f_g, f_b, f_c

            def tfloat(self): return False
        nt, ntr = types.ModuleType('ntracer'), types.ModuleType('ntracer.render')
        ntr.Channel, ntr.CallbackRenderer = Chan, object
        nt.render = ntr
        saved = {k: sys.modules.get(k) for k in ('ntracer', 'ntracer.render')}
        sys.modules['ntracer'], sys.modules['ntracer.render'] = nt, ntr
        try:
            ns = {'__name__': 'ref_pygame_render'}
            exec(compile(open(REF).read(), REF, 'exec'), ns)
            ref_fn = ns['channels_from_surface']
        finally:
            for k, v in saved.items():
                if v is None:
                    sys.modules.pop(k, None)
                else:
                    sys.modules[k] = v
    for name, ((nbytes, masks, shifts, losses), expected) in FORMATS.items():
        s = FakeSurface(4, 2, nbytes, masks, shifts, losses)
        got = _tuples(mod.channels_from_surface(s))
        assert got == [tuple(float(v) if i else v for i, v in enumerate(e)) for e in expected], name
        assert sum(c[0] for c in got) <= nbytes * 8
        if ref_fn:
            assert got == _tuples(ref_fn(s)), name
    with pytest.raises(TypeError):
        mod.channels_from_surface(FakeSurface(4, 2, 1, (0, 0, 0, 0), (0, 0, 0, 0), (8, 8, 8, 8)))
    assert pg.quit_hooks and callable(pg.quit_hooks[0])


@pytest.mark.parametrize('name', ['xrgb8888', 'bgr888', 'rgb565'])
def test_pygame_renderer_draws_the_surface_and_posts_the_event(name, fake_pygame, monkeypatch):
    pg, mod = fake_pygame
    from ntracer_b200 import NTracer, BlockingRenderer, ImageFormat, tracern
    from tests.test_facade_emulated import _EmulatedFullDevice
    monkeypatch.setattr(tracern, 'DeviceScene', _EmulatedFullDevice)
    nt = NTracer(4)
    scene = nt.BoxScene()
    cam = nt.Camera()
    cam.translate(nt.Vector.axis(2, -3))
    scene.set_camera(cam)
    (nbytes, masks, shifts, losses), _ = FORMATS[name]
    surf = FakeSurface(40, 24, nbytes, masks, shifts, losses, pad=3)
    r = mod.PygameRenderer()
    assert r in mod.PygameRenderer.instances and r.ON_COMPLETE == pg.USEREVENT
    r.begin_render(surf, scene)
    assert pg.arrived.wait(60)
    r.abort_render()                                         # joins the worker; the frame is complete already
    e = pg.posted[0]
    assert (e.type, e.source, e.scene, e.surface) == (pg.USEREVENT, r, scene, surf)
    assert scene.locked == 0
    # the same frame through BlockingRenderer with the format the front end derived
    fmt = ImageFormat(40, 24, mod.channels_from_surface(surf), surf.pitch, True)
    want = bytearray(b'\xEE' * len(surf.buf))
    assert BlockingRenderer().render(want, fmt, scene)
    assert surf.buf == want
    rows = np.frombuffer(surf.buf, np.uint8).reshape(24, surf.pitch)
    assert (rows[:, 40 * nbytes:] == 0xEE).all() and len(set(bytes(rows[:, :40 * nbytes].tobytes()))) > 4
    assert r.last_channels[0] == (nbytes * 8, masks)
    cached = r.last_channels[1]
    pg.arrived.clear()
    r.begin_render(surf, scene)                              # same layout: the channel list is reused
    assert pg.arrived.wait(60)
    r.abort_render()
    assert r.last_channels[1] is cached and len(pg.posted) == 2
    pg.quit_hooks[0]()                                       # the quit hook aborts whatever is running; nothing is
