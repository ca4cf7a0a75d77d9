"""ntracer_b200.render -- host-side mirror of the reference's `ntracer.render` module (src/render.cpp) for the
render path: Color, Material, Channel, ImageFormat, BlockingRenderer, CallbackRenderer, Scene, LockedError.
Same names, arguments and error behaviour; the frames are produced by the CUDA backend (ntr_render)."""
import ctypes as C
import threading

import numpy as np

from . import _capi


class LockedError(Exception):
    """Raised when a scene is modified while a renderer is using it (src/ntracer_body.hpp:235-240)."""


def _color_tuple(c):
    if isinstance(c, Color):
        return (c.r, c.g, c.b)
    t = tuple(float(x) for x in c)
    if len(t) != 3:
        raise TypeError('object must be an instance of Color or a sequence with three numbers')
    return t


class Color:
    """Color(r,g,b) (src/light.hpp, doc/ntracer.rst:158-256)"""
    __slots__ = ('r', 'g', 'b')

    def __init__(self, r, g, b):
        f = np.float32
        self.r, self.g, self.b = float(f(r)), float(f(g)), float(f(b))

    def __len__(self): return 3
    def __getitem__(self, i): return (self.r, self.g, self.b)[i]
    def __iter__(self): return iter((self.r, self.g, self.b))
    def __repr__(self): return 'Color(%r,%r,%r)' % (self.r, self.g, self.b)
    def __eq__(self, b): return isinstance(b, Color) and tuple(self) == tuple(b)
    def __ne__(self, b): return not self.__eq__(b)
    def __hash__(self): return hash(tuple(self))
    def __neg__(self): return Color(-self.r, -self.g, -self.b)
    def __buffer__(self, flags): return memoryview(np.array(tuple(self), np.float32))

    def _bin(self, b, op):
        if isinstance(b, Color):
            return Color(op(self.r, b.r), op(self.g, b.g), op(self.b, b.b))
        return Color(op(self.r, b), op(self.g, b), op(self.b, b))

    def __add__(self, b): return self._bin(b, lambda x, y: x + y)
    def __sub__(self, b): return self._bin(b, lambda x, y: x - y)
    def __mul__(self, b): return self._bin(b, lambda x, y: x * y)
    __rmul__ = __mul__
    def __truediv__(self, b): return self._bin(b, lambda x, y: x / y)
    __div__ = __truediv__
    def apply(self, f): return Color(f(self.r), f(self.g), f(self.b))
    def __reduce__(self): return (_color_unpickle, (_encode_floats(tuple(self)),))       # render.cpp:1094-1101


class Material:
    """Material(color[,opacity=1,reflectivity=0,specular_intensity=1,specular_exp=8,specular_color=(1,1,1)])
    (src/render.hpp:56-73, src/render.cpp:1249-1274).  Attributes are mutable, like the reference's."""
    def __init__(self, color, opacity=1, reflectivity=0, specular_intensity=1, specular_exp=8, specular_color=(1, 1, 1)):
        self.color = Color(*_color_tuple(color))
        self.opacity, self.reflectivity = float(opacity), float(reflectivity)
        self.specular_intensity, self.specular_exp = float(specular_intensity), float(specular_exp)
        self.specular = Color(*_color_tuple(specular_color))

    def __setattr__(self, k, v):
        if k in ('color', 'specular'):
            v = v if isinstance(v, Color) else Color(*_color_tuple(v))
        elif k in ('opacity', 'reflectivity', 'specular_intensity', 'specular_exp'):
            v = float(v)
            if k in ('opacity', 'reflectivity'):
                v = min(max(v, 0.0), 1.0)           # the reference clamps both to [0,1] (render.cpp:1211-1232)
        object.__setattr__(self, k, v)

    def _row(self):
        return np.array([self.color.r, self.color.g, self.color.b, self.specular.r, self.specular.g, self.specular.b,
                         self.opacity, self.reflectivity, self.specular_intensity, self.specular_exp], np.float32)

    def __eq__(self, b): return isinstance(b, Material) and bool(np.all(self._row() == b._row()))
    def __reduce__(self): return (_material_unpickle, (_encode_floats(self._row()),))     # render.cpp:1197-1208
    def __hash__(self): return id(self)
    def __repr__(self):
        return 'Material(%r,%r,%r,%r,%r,%r)' % (tuple(self.color), self.opacity, self.reflectivity, self.specular_intensity,
                                                self.specular_exp, tuple(self.specular))


# ---- the reference's pickle encodings (src/render.cpp:1391-1657, 1698-1746) ------------------------------------------
# Every picklable value type reduces to (render._<type>_unpickle, args) with its floats as big-endian IEEE-754 bytes;
# the functions below take exactly the arguments the reference's take and fail the same way, so a pickle written by
# either side names the same functions with the same payload (ntracer_b200.compat maps the module names).
def _encode_floats(values):
    return np.asarray(values, dtype='>f4').tobytes()


def _decode_floats(data, count, what):
    if not isinstance(data, (bytes, bytearray)):
        raise TypeError('object is not an instance of bytes')
    if len(data) != 4 * count:
        raise ValueError('%s data is malformed' % what)
    return np.frombuffer(bytes(data), dtype='>f4').astype(np.float32)


def _check_args(args, n, name):
    if len(args) != n:
        raise TypeError('%s takes exactly %d arguments' % (name, n))


def _color_unpickle(data):
    return Color(*_decode_floats(data, 3, 'color'))


def _material_unpickle(data):
    v = [float(x) for x in _decode_floats(data, 10, 'material')]
    m = Material(v[0:3], 1, 0, v[8], v[9], v[3:6])
    object.__setattr__(m, 'opacity', v[6])          # stored as they are: the reference's unpickle does not clamp
    object.__setattr__(m, 'reflectivity', v[7])
    return m


def _vector_unpickle(*args):
    from . import tracern
    _check_args(args, 2, '_vector_unpickle')
    dim = tracern._check_dimension(args[0])
    return tracern.Vector._wrap(_decode_floats(args[1], dim, 'vector'))


def _matrix_unpickle(*args):
    from . import tracern
    _check_args(args, 2, '_matrix_unpickle')
    dim = tracern._check_dimension(args[0])
    return tracern.Matrix._wrap(_decode_floats(args[1], dim * dim, 'matrix').reshape(dim, dim))


def _triangle_unpickle(*args):
    from . import tracern
    _check_args(args, 3, '_triangle_unpickle')
    dim = tracern._check_dimension(args[0])
    rows = _decode_floats(args[1], dim * (dim + 1), 'triangle').reshape(dim + 1, dim)        # p1, face_normal, edge normals
    if not isinstance(args[2], Material):
        raise TypeError('object is not an instance of Material')
    V = tracern.Vector._wrap
    return tracern.Triangle(V(rows[0]), V(rows[1]), [V(r) for r in rows[2:]], args[2])           # d is recomputed, like triangle_extra


def _triangle_batch_unpickle(*args):
    from . import tracern
    if len(args) < 3:
        raise TypeError('wrong number of arguments')
    dim = tracern._check_dimension(args[1])
    B = tracern.BATCH_SIZE
    if int(args[0]) != B:
        raise TypeError('The TriangleBatch instance was pickled with a different batch size. It cannot be loaded here.')
    if len(args) != 3 + B:
        raise TypeError('wrong number of arguments')
    rows = _decode_floats(args[2], B * dim * (dim + 1), 'triangle batch').reshape(dim + 1, dim, B)    # [row][coordinate][lane]
    for m in args[3:]:
        if not isinstance(m, Material):
            raise TypeError('object is not an instance of Material')
    V = tracern.Vector._wrap
    return tracern.TriangleBatch([tracern.Triangle(V(rows[0, :, k]), V(rows[1, :, k]), [V(rows[2 + e, :, k]) for e in range(dim - 1)],
                                                   args[3 + k]) for k in range(B)])


def _solid_unpickle(*args):
    from . import tracern
    _check_args(args, 3, '_solid_unpickle')
    dim = tracern._check_dimension(args[0])
    data = args[1]
    if not isinstance(data, (bytes, bytearray)):
        raise TypeError('object is not an instance of bytes')
    if len(data) != 4 * dim * (dim + 1) + 1:
        raise ValueError('solid data is malformed')
    if data[0] not in (tracern.CUBE, tracern.SPHERE):
        raise ValueError('solid data is corrupt')
    if not isinstance(args[2], Material):
        raise TypeError('object is not an instance of Material')
    vals = _decode_floats(data[1:], dim * (dim + 1), 'solid')
    return tracern.Solid(int(data[0]), tracern.Vector._wrap(vals[dim * dim:]), tracern.Matrix._wrap(vals[:dim * dim].reshape(dim, dim)), args[2])


def _aabb_unpickle(*args):
    from . import tracern
    _check_args(args, 2, '_aabb_unpickle')
    dim = tracern._check_dimension(args[0])
    vals = _decode_floats(args[1], 2 * dim, 'AABB')
    return tracern.AABB(dim, tracern.Vector._wrap(vals[:dim]), tracern.Vector._wrap(vals[dim:]))


class Channel:
    """Channel(bit_size,f_r,f_g,f_b[,f_c=0,tfloat=False]) (src/render.cpp:95-164)"""
    __slots__ = ('bit_size', 'f_r', 'f_g', 'f_b', 'f_c', 'tfloat')

    def __init__(self, bit_size, f_r, f_g, f_b, f_c=0, tfloat=False):
        bit_size = int(bit_size)
        if tfloat:
            if bit_size != 32:
                raise ValueError('if "tfloat" is true, "bit_size" can only be 32')
        elif bit_size > 31:
            raise ValueError('"bit_size" cannot be greater than 31 (unless "tfloat" is true)')
        elif bit_size < 1:
            raise ValueError('"bit_size" cannot be less than 1')
        object.__setattr__(self, 'bit_size', bit_size)
        for n, v in (('f_r', f_r), ('f_g', f_g), ('f_b', f_b), ('f_c', f_c)):
            object.__setattr__(self, n, float(np.float32(v)))
        object.__setattr__(self, 'tfloat', bool(tfloat))

    def __setattr__(self, k, v):
        raise AttributeError('readonly attribute')

    def _tuple(self): return (self.bit_size, self.f_r, self.f_g, self.f_b, self.f_c, self.tfloat)


class ImageFormat:
    """ImageFormat(width,height,channels[,pitch=0,reversed=False]) (src/render.cpp:167-288)"""
    def __init__(self, width, height, channels, pitch=0, reversed=False):
        self.width, self.height, self.reversed = int(width), int(height), bool(reversed)
        self.set_channels(channels)
        f = _capi.make_image_format(self.width, self.height, [c._tuple() for c in self._channels], int(pitch), self.reversed)
        self.pitch = f.pitch

    def set_channels(self, new_channels):
        chans = list(new_channels)
        for c in chans:
            if not isinstance(c, Channel):
                raise TypeError('object is not an instance of Channel')
        bits = sum(c.bit_size for c in chans)
        if bits > 16 * 8:
            raise ValueError('Too many bytes per pixel. The maximum is 16.')
        self._channels = tuple(chans)
        self._bpp = (bits + 7) // 8

    channels = property(lambda self: self._channels)
    bytes_per_pixel = property(lambda self: self._bpp)

    def _native(self):
        return _capi.make_image_format(self.width, self.height, [c._tuple() for c in self._channels], self.pitch, self.reversed)


class Scene:
    """Abstract scene (src/render.hpp:8-26): anything with _prepare() -> DeviceScene and a `locked` counter."""
    def calculate_color(self, x, y, width, height):
        raise NotImplementedError


def _writable_buffer(dest):
    mv = memoryview(dest)
    if mv.readonly:
        raise BufferError('Object is not writable.')
    return np.frombuffer(mv, dtype=np.uint8)


def _gpus_for(threads):
    """How many GPUs trace a frame.  The reference's `threads` is its worker count (0 / -1: one per core,
    src/render.cpp:829-838); here a value above 1 asks for that many B200s of the box (interleaved tile rows, every GPU
    storing its rows into one frame on the first over NVLink: ntr_group_*), anything else for one.  NTR_GPUS overrides."""
    import os
    from .backend import device_count
    want = int(os.environ.get('NTR_GPUS', '0') or 0) or int(threads)
    return max(1, min(want, device_count())) if want > 1 else 1


def _render_call(dev):
    return dev._lib.ntr_group_render if hasattr(dev, 'size') else dev._lib.ntr_render


class BlockingRenderer:
    """BlockingRenderer([threads=-1]) (src/render.cpp:829-929).  threads > 1: that many GPUs trace the frame."""
    def __init__(self, threads=-1):
        self._lock = threading.Lock()
        self._dev = None
        self._gpus = _gpus_for(threads)

    def render(self, dest, format, scene):
        """-> True, or False if signal_abort() was called while rendering."""
        if not isinstance(format, ImageFormat):
            raise TypeError('object is not an instance of ImageFormat')
        if not isinstance(scene, Scene):
            raise TypeError('object is not an instance of Scene')
        buf = _writable_buffer(dest)
        fmt = format._native()
        if buf.size < fmt.pitch * fmt.height:
            raise ValueError('the buffer is too small for an image with the given dimensions')
        if not self._lock.acquire(blocking=False):
            raise RuntimeError('the renderer is already running')
        try:
            scene.locked += 1
            try:
                dev = scene._prepare(self._gpus) if self._gpus > 1 else scene._prepare()
                self._dev = dev
                rc = _render_call(dev)(dev._h, C.byref(fmt), buf.ctypes.data_as(C.c_void_p), buf.size)
                if rc == _capi.NTR_ERR_ABORTED:
                    return False
                _capi.check(rc)
                return True
            finally:
                self._dev = None
                scene.locked -= 1
        finally:
            self._lock.release()

    def render_views(self, dest, format, scene, cameras, *, ids=None, depth=None, normals=None):
        """Extension without a reference counterpart: one frame per camera in one call, frame k at byte offset
        k * pitch * height of `dest` (ntr_render_views).  Frame k is what render() gives after scene.set_camera(cameras[k]);
        the scene's camera is left as it is.  cameras: Camera objects of the scene's dimension or (origin, axes) pairs
        (stream.rotation_cameras).  With threads > 1 (or NTR_GPUS) whole views are dealt to the GPUs.
        ids / depth / normals: writable buffers that also receive the per-pixel AOVs of every view, in the same launches
        (ntr_render_views_aovs): int32 hit ids (n x height x width, -1 on a miss), float32 hit distances (n x height x width)
        and float32 normals (n x height x width x dimension) of each pixel's plain primary ray.  A numpy array must have
        that dtype.
        -> True, or False if signal_abort() was called while rendering."""
        from .backend import AOV_DTYPES, aov_shape, aov_struct, camera_arrays
        if not isinstance(format, ImageFormat):
            raise TypeError('object is not an instance of ImageFormat')
        if not isinstance(scene, Scene):
            raise TypeError('object is not an instance of Scene')
        origins, axes = camera_arrays(cameras, scene.dimension)
        n = len(origins)
        buf = _writable_buffer(dest)
        fmt = format._native()
        if buf.size < n * fmt.pitch * fmt.height:
            raise ValueError('the buffer is too small for %d images with the given dimensions' % n)
        aovs = {}
        for name, b in (('ids', ids), ('depth', depth), ('normals', normals)):
            if b is None:
                continue
            if isinstance(b, np.ndarray) and b.dtype != AOV_DTYPES[name]:
                raise TypeError('the %s buffer must hold %s' % (name, np.dtype(AOV_DTYPES[name]).name))
            v = _writable_buffer(b)
            if v.size < 4 * int(np.prod(aov_shape(name, n, fmt, scene.dimension))):
                raise ValueError('the %s buffer is too small for %d images with the given dimensions' % (name, n))
            aovs[name] = (v.ctypes.data, v.size // 4)
        if not self._lock.acquire(blocking=False):
            raise RuntimeError('the renderer is already running')
        try:
            scene.locked += 1
            try:
                dev = scene._prepare(self._gpus) if self._gpus > 1 else scene._prepare()
                self._dev = dev
                args = (dev._h, n, origins.ctypes.data_as(C.c_void_p), axes.ctypes.data_as(C.c_void_p), C.byref(fmt),
                        buf.ctypes.data_as(C.c_void_p), buf.size)
                if aovs:
                    fn = dev._lib.ntr_group_render_views_aovs if hasattr(dev, 'size') else dev._lib.ntr_render_views_aovs
                    rc = fn(*args, C.byref(aov_struct(aovs)))
                else:
                    fn = dev._lib.ntr_group_render_views if hasattr(dev, 'size') else dev._lib.ntr_render_views
                    rc = fn(*args)
                if rc == _capi.NTR_ERR_ABORTED:
                    return False
                _capi.check(rc)
                return True
            finally:
                self._dev = None
                scene.locked -= 1
        finally:
            self._lock.release()

    def signal_abort(self):
        dev = self._dev
        if dev is not None:
            dev.abort()


class CallbackRenderer:
    """CallbackRenderer([threads=0]) (src/render.cpp:495-728): begin_render returns immediately; `callback(self)`
    runs on a worker thread once the frame is complete (not when aborted)."""
    def __init__(self, threads=0):
        self._thread = None
        self._dev = None
        self._lock = threading.Lock()
        self._gpus = _gpus_for(threads)

    def begin_render(self, dest, format, scene, callback):
        if not isinstance(format, ImageFormat):
            raise TypeError('object is not an instance of ImageFormat')
        if not isinstance(scene, Scene):
            raise TypeError('object is not an instance of Scene')
        buf = _writable_buffer(dest)
        fmt = format._native()
        if buf.size < fmt.pitch * fmt.height:
            raise ValueError('the buffer is too small for an image with the given dimensions')
        with self._lock:
            if self._thread is not None and self._thread.is_alive() and threading.current_thread() is not self._thread:
                raise RuntimeError('the renderer is already running')
            scene.locked += 1
            try:
                dev = scene._prepare(self._gpus) if self._gpus > 1 else scene._prepare()
            except Exception:
                scene.locked -= 1
                raise
            self._dev = dev

            def work():
                try:
                    rc = _render_call(dev)(dev._h, C.byref(fmt), buf.ctypes.data_as(C.c_void_p), buf.size)
                finally:
                    scene.locked -= 1
                    self._dev = None
                if rc == _capi.NTR_OK:
                    callback(self)

            self._thread = threading.Thread(target=work, daemon=True)
            self._thread.start()

    def abort_render(self):
        dev, t = self._dev, self._thread
        if dev is not None:
            dev.abort()
        if t is not None and t is not threading.current_thread():
            t.join()


class StreamRenderer:
    """Extension without a reference counterpart: the interactive loop of scripts/polytope.py:505-557 (begin_render ->
    completion callback -> move the camera -> begin_render ...) with two frames in flight, so that frame k+1 is traced
    while frame k crosses PCIe (ntr_render_begin / ntr_render_end).  The reference cannot overlap frames: its scene is
    locked, camera included, until the frame is complete (src/tracer.hpp:1922-1926).

        t0 = r.submit(buf0, fmt, scene); scene.set_camera(cam1)
        t1 = r.submit(buf1, fmt, scene); r.wait(t0)  # buf0 is complete ...

    The camera and scene parameters are captured by submit(); geometry must not change while frames are open."""
    def __init__(self):
        self._open = {}

    def submit(self, dest, format, scene):
        if not isinstance(format, ImageFormat):
            raise TypeError('object is not an instance of ImageFormat')
        if not isinstance(scene, Scene):
            raise TypeError('object is not an instance of Scene')
        buf = _writable_buffer(dest)
        fmt = format._native()
        if buf.size < fmt.pitch * fmt.height:
            raise ValueError('the buffer is too small for an image with the given dimensions')
        dev = scene._prepare()
        ticket = dev.render_begin(fmt, buf)
        self._open[ticket] = dev
        return ticket

    def wait(self, ticket):
        """-> True, or False if abort() hit the frame."""
        dev = self._open.pop(ticket)
        try:
            dev.render_end(ticket)
        except _capi.AbortedError:
            return False
        return True

    def abort(self):
        for dev in set(self._open.values()):
            dev.abort()
