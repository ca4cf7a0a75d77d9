"""DeviceScene: thin object wrapper over the C ABI (include/ntracer_b200.h).

One DeviceScene = one scene arena resident on one B200.  The reference-compatible classes in
ntracer_b200.tracern / ntracer_b200.render build flat scene dicts and drive this class; tests and
bench.py use it directly.  Every method goes through libntracer_b200.so -- there is no CPU path.
"""
import ctypes as C

import numpy as np

from . import _capi

FLT_MAX = 3.4028234663852886e38


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def camera_arrays(cameras, dim):
    """The cameras of a views call -> (origins [n, dim], axes [n, dim, dim]) float32, C-contiguous.  `cameras` is a sequence
    of tracern.Camera objects or (origin, axes) pairs (what stream.rotation_cameras returns), or a mix of both.
    TypeError: not such a sequence; ValueError: no camera, or one of another dimension."""
    from .tracern import Camera
    try:
        items = list(cameras)
    except TypeError:
        raise TypeError('cameras must be a sequence of Camera objects or (origin, axes) pairs') from None
    if not items:
        raise ValueError('at least one camera is needed')
    origins = np.empty((len(items), dim), np.float32)
    axes = np.empty((len(items), dim, dim), np.float32)
    for k, c in enumerate(items):
        if isinstance(c, Camera):
            o, a = c._origin, c._axes
        elif isinstance(c, (tuple, list)) and len(c) == 2:
            try:
                o, a = np.asarray(c[0], np.float32), np.asarray(c[1], np.float32)
            except (TypeError, ValueError):
                raise TypeError('camera %d: origin and axes must be arrays of numbers' % k) from None
        else:
            raise TypeError('camera %d is neither a Camera nor an (origin, axes) pair' % k)
        if o.shape != (dim,) or a.shape != (dim, dim):
            raise ValueError('camera %d: the scene and camera must have the same dimension (%d)' % (k, dim))
        origins[k], axes[k] = o, a
    return origins, axes


def _views_dest(dest, n, fmt):
    """-> (what render_views returns, the uint8 view of it the library writes)"""
    need = n * fmt.pitch * fmt.height
    if dest is None:
        out = np.zeros((n, fmt.pitch * fmt.height), dtype=np.uint8)
        return out, out
    buf = np.frombuffer(dest, dtype=np.uint8)
    if buf.size < need:
        raise ValueError('the buffer is too small for %d images with the given dimensions' % n)
    return dest, buf


AOV_NAMES = ('ids', 'depth', 'normals')
AOV_DTYPES = {'ids': np.int32, 'depth': np.float32, 'normals': np.float32}


def aov_shape(name, n, fmt, dim):
    """shape of AOV `name` of n views: (n, height, width), and (n, height, width, dim) for the normals"""
    return (n, fmt.height, fmt.width) + ((dim,) if name == 'normals' else ())


def _aov_names(aovs):
    names = tuple(aovs)
    for name in names:
        if name not in AOV_NAMES:
            raise ValueError('unknown AOV %r (known: %s)' % (name, ', '.join(AOV_NAMES)))
    return names


def aov_struct(ptrs):
    """{name: (address, length in elements)} -> _capi.AovBuffers (the AOVs not named are not wanted)"""
    a = _capi.AovBuffers()
    for name, (ptr, length) in ptrs.items():
        setattr(a, name, ptr)
        setattr(a, name + '_len', int(length))
    return a


def _new_aovs(aovs, n, fmt, dim):
    """-> ({name: new array}, AovBuffers over them)"""
    arrays = {name: np.zeros(aov_shape(name, n, fmt, dim), AOV_DTYPES[name]) for name in _aov_names(aovs)}
    return arrays, aov_struct({k: (v.ctypes.data, v.size) for k, v in arrays.items()})


def _refine_mask(fn, handle, w, h):
    mask = np.zeros((h, w), dtype=np.uint8)
    count = C.c_uint64(0)
    _capi.check(fn(handle, _p(mask) if mask.size else None, mask.size, C.byref(count)))
    return mask, int(count.value)


class DeviceScene:
    def __init__(self, scene, device=-1):
        """scene: flat scene dict (DESIGN.md 'scene file'; ntracer_b200.scene_io.load_scene)."""
        self._lib = _capi.load()
        self._h = C.c_void_p()
        self.dim = int(scene['dim'])
        self.kind = int(scene['kind'])
        self._scene = scene
        self._open = {}
        self.supersampling = 1
        self.supersampling_threshold = None
        self._window = None                     # (width, height) of the last frame's window: the shape of refine_mask()
        desc, keep = _capi.make_desc(scene)
        _capi.check(self._lib.ntr_scene_create(C.byref(desc), device, C.byref(self._h)))
        if 'cam_origin' in scene and 'cam_axes' in scene:
            self.set_camera(scene['cam_origin'], scene['cam_axes'])

    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            self._lib.ntr_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- state ----
    def set_camera(self, origin, axes):
        o = np.ascontiguousarray(origin, dtype=np.float32).reshape(self.dim)
        a = np.ascontiguousarray(axes, dtype=np.float32).reshape(self.dim, self.dim)
        _capi.check(self._lib.ntr_scene_set_camera(self._h, _p(o), _p(a)))

    def set_params(self, scene):
        """Re-send fov / shadows / camera_light / max_reflect_depth / background / ambient / lights."""
        desc, keep = _capi.make_desc(scene)
        _capi.check(self._lib.ntr_scene_set_params(self._h, C.byref(desc)))
        self._scene = scene

    def set_instrumented(self, on):
        _capi.check(self._lib.ntr_set_instrumented(self._h, int(bool(on))))

    def set_supersampling(self, factor):
        """Anti-aliasing: every pixel becomes the mean of factor x factor samples (1..8; 1 = one ray per pixel)."""
        _capi.check(self._lib.ntr_scene_set_supersampling(self._h, int(factor)))
        self.supersampling = int(factor)

    def set_supersampling_threshold(self, threshold):
        """Adaptive supersampling: with a factor above 1, only pixels whose corner colours differ by more than `threshold`
        in some channel get the factor x factor samples (None = off: every pixel does)."""
        _capi.check(self._lib.ntr_scene_set_supersampling_threshold(self._h, -1.0 if threshold is None else float(threshold)))
        self.supersampling_threshold = None if threshold is None else float(threshold)

    def refine_mask(self):
        """-> (mask, count): the refine mask of the last frame as a (height, width) uint8 array over its window (1 =
        refined; rows a sharded render does not own stay 0) and the number of refined pixels."""
        w, h = self._window if self._window else (0, 0)
        return _refine_mask(self._lib.ntr_last_refine_mask, self._h, w, h)

    # ---- the hot path ----
    def render(self, fmt, dest=None):
        """BlockingRenderer.render: packs the frame into `dest` (any writable buffer) or a new uint8 array."""
        need = fmt.pitch * fmt.height
        if dest is None:
            out = np.zeros(need, dtype=np.uint8)
            buf = out
        else:
            out = dest
            buf = np.frombuffer(dest, dtype=np.uint8)
            if buf.size < need:
                raise ValueError('the buffer is too small for an image with the given dimensions')
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render(self._h, C.byref(fmt), _p(buf), buf.size))
        return out

    def render_views(self, fmt, cameras, dest=None):
        """One frame per camera in one call (ntr_render_views): frame k of `dest` (any writable buffer) at byte offset
        k * pitch * height, or a new (n, pitch * height) uint8 array.  cameras: Camera objects or (origin, axes) pairs.
        Frame k is what render() gives with camera k; the scene's own camera is left as it is."""
        origins, axes = camera_arrays(cameras, self.dim)
        out, buf = _views_dest(dest, len(origins), fmt)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_views(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt), _p(buf), buf.size))
        return out

    def render_views_device(self, fmt, cameras, dev_ptr, nbytes, stream=0):
        """render_views into device memory (a (n, height, pitch) uint8 torch tensor's data_ptr()) on a CUDA stream handle:
        asynchronous for frames without reflection passes, synchronous on the stream with them."""
        origins, axes = camera_arrays(cameras, self.dim)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_views_device(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt),
                                                      C.c_void_p(dev_ptr), int(nbytes), C.c_void_p(stream)))

    def render_views_aovs(self, fmt, cameras, aovs=AOV_NAMES, dest=None):
        """render_views plus per-pixel AOVs of every view in the same launches (ntr_render_views_aovs) -> (frames, {name:
        array}) for the names in `aovs`: 'ids' int32 (n, height, width), the flat id of the plain primary ray's opaque hit
        (-1: a miss) as primary_hit_ids gives it; 'depth' float32 (n, height, width), its distance (0 on a miss); 'normals'
        float32 (n, height, width, dim), the normal that shades the hit (zeros on a miss).  Frames and counters are those of
        render_views."""
        origins, axes = camera_arrays(cameras, self.dim)
        out, buf = _views_dest(dest, len(origins), fmt)
        arrays, a = _new_aovs(aovs, len(origins), fmt, self.dim)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_views_aovs(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt), _p(buf), buf.size,
                                                    C.byref(a)))
        return out, arrays

    def render_views_aovs_device(self, fmt, cameras, dev_ptr, nbytes, aovs, stream=0):
        """render_views_aovs into device memory on a CUDA stream handle: the frames as render_views_device, `aovs` maps AOV
        names to torch tensors on the scene's device (int32 ids, float32 depth and normals, in render_views_aovs's shapes) or
        to (device address, length in elements) pairs."""
        origins, axes = camera_arrays(cameras, self.dim)
        ptrs = {}
        for name in _aov_names(aovs):
            t = aovs[name]
            ptrs[name] = (t.data_ptr(), t.numel()) if hasattr(t, 'data_ptr') else (int(t[0]), int(t[1]))
        a = aov_struct(ptrs)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_views_aovs_device(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt),
                                                           C.c_void_p(dev_ptr), int(nbytes), C.byref(a), C.c_void_p(stream)))

    def render_begin(self, fmt, dest):
        """Enqueue one frame with the current camera and return a ticket (the interactive loop: frame k+1 is traced
        while frame k is copied back; at most two frames open).  `dest` must stay alive until render_end(ticket)."""
        buf = np.frombuffer(dest, dtype=np.uint8)
        if buf.size < fmt.pitch * fmt.height:
            raise ValueError('the buffer is too small for an image with the given dimensions')
        ticket = C.c_uint64(0)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_begin(self._h, C.byref(fmt), _p(buf), buf.size, C.byref(ticket)))
        self._open[ticket.value] = buf          # keeps the exported buffer alive while the copy engine writes it
        return ticket.value

    def render_end(self, ticket):
        """Wait for the frame of `ticket` and finish the copy into its destination."""
        try:
            _capi.check(self._lib.ntr_render_end(self._h, C.c_uint64(ticket)))
        finally:
            self._open.pop(ticket, None)

    def render_device(self, fmt, dev_ptr, nbytes, stream=0, tile_row_first=0, tile_row_step=1, compact=False):
        """Asynchronous render into device memory (a torch tensor's data_ptr()) on a CUDA stream handle."""
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_render_device(self._h, C.byref(fmt), C.c_void_p(dev_ptr), nbytes,
                                                C.c_void_p(stream), tile_row_first, tile_row_step, int(compact)))

    def render_float(self, width, height):
        out = np.zeros((height, width, 3), dtype=np.float32)
        self._window = (width, height)
        _capi.check(self._lib.ntr_render_float(self._h, width, height, _p(out)))
        return out

    def calculate_color(self, x, y, width, height):
        out = (C.c_float * 3)()
        self._window = (1, 1)
        _capi.check(self._lib.ntr_calculate_color(self._h, x, y, width, height, out))
        return np.array(list(out), dtype=np.float32)

    def primary_hit_ids(self, width, height):
        ids = np.zeros((height, width), dtype=np.int32)
        dist = np.zeros((height, width), dtype=np.float32)
        _capi.check(self._lib.ntr_primary_hit_ids(self._h, width, height, _p(ids), _p(dist)))
        return ids, dist

    def trace_rays(self, origins, dirs, t_near=-FLT_MAX, t_far=FLT_MAX, skip_ref=None, skip_lane=None):
        origins = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, self.dim)
        dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, self.dim)
        n = origins.shape[0]
        ids = np.zeros(n, dtype=np.int32)
        dist = np.zeros(n, dtype=np.float32)
        nt = np.zeros(n, dtype=np.int32)
        sr = None if skip_ref is None else np.ascontiguousarray(skip_ref, dtype=np.uint32)
        sl = None if skip_lane is None else np.ascontiguousarray(skip_lane, dtype=np.int32)
        _capi.check(self._lib.ntr_trace_rays(self._h, n, _p(origins), _p(dirs), t_near, t_far, _p(sr), _p(sl),
                                             _p(ids), _p(dist), _p(nt)))
        return ids, dist, nt

    def trace_rays_hits(self, origins, dirs, t_near=-FLT_MAX, t_far=FLT_MAX, skip_ref=None, skip_lane=None, max_hits=16):
        """trace_rays plus the surviving transparent hits of every ray: (ids, dist, n_transparent, hit_ids [n, max_hits]
        (-1 = unused), hit_dists [n, max_hits]) -- what KDNode.intersects returns ahead of the opaque hit."""
        origins = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, self.dim)
        dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, self.dim)
        n = origins.shape[0]
        ids = np.zeros(n, dtype=np.int32)
        dist = np.zeros(n, dtype=np.float32)
        nt = np.zeros(n, dtype=np.int32)
        hid = np.full((n, max_hits), -1, dtype=np.int32)
        hdist = np.zeros((n, max_hits), dtype=np.float32)
        sr = None if skip_ref is None else np.ascontiguousarray(skip_ref, dtype=np.uint32)
        sl = None if skip_lane is None else np.ascontiguousarray(skip_lane, dtype=np.int32)
        _capi.check(self._lib.ntr_trace_rays_hits(self._h, n, _p(origins), _p(dirs), t_near, t_far, _p(sr), _p(sl),
                                                  _p(ids), _p(dist), _p(nt), int(max_hits), _p(hid), _p(hdist)))
        return ids, dist, nt, hid, hdist

    def occludes_rays(self, origins, dirs, distance=None, skip_ref=None, skip_lane=None):
        origins = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, self.dim)
        dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, self.dim)
        n = origins.shape[0]
        occ = np.zeros(n, dtype=np.int32)
        nt = np.zeros(n, dtype=np.int32)
        dd = None if distance is None else np.ascontiguousarray(distance, dtype=np.float32)
        sr = None if skip_ref is None else np.ascontiguousarray(skip_ref, dtype=np.uint32)
        sl = None if skip_lane is None else np.ascontiguousarray(skip_lane, dtype=np.int32)
        _capi.check(self._lib.ntr_occludes_rays(self._h, n, _p(origins), _p(dirs), _p(dd), _p(sr), _p(sl),
                                                _p(occ), _p(nt)))
        return occ, nt

    # ---- control / introspection ----
    def abort(self):
        _capi.check(self._lib.ntr_abort(self._h))

    def counters(self):
        c = _capi.Counters()
        _capi.check(self._lib.ntr_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    def last_kernel_ms(self):
        ms = C.c_float()
        _capi.check(self._lib.ntr_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        return int(self._lib.ntr_launch_count(self._h))


class DeviceGroup:
    """One scene replicated on several B200s of one box (ntr_group_*): a frame is split by interleaved 32-pixel tile rows
    and every device stores its rows straight into one frame buffer on the first device over NVLink."""
    def __init__(self, scene, n=0, devices=None):
        self._lib = _capi.load()
        self._h = C.c_void_p()
        self.dim = int(scene['dim'])
        desc, keep = _capi.make_desc(scene)
        devs = None if devices is None else (C.c_int * len(devices))(*[int(d) for d in devices])
        _capi.check(self._lib.ntr_group_create(C.byref(desc), len(devices) if devices is not None else int(n), devs, C.byref(self._h)))
        self.size = int(self._lib.ntr_group_size(self._h))
        self.supersampling = 1
        self.supersampling_threshold = None
        self._window = None
        if 'cam_origin' in scene and 'cam_axes' in scene:
            self.set_camera(scene['cam_origin'], scene['cam_axes'])

    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            self._lib.ntr_group_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_camera(self, origin, axes):
        o = np.ascontiguousarray(origin, dtype=np.float32).reshape(self.dim)
        a = np.ascontiguousarray(axes, dtype=np.float32).reshape(self.dim, self.dim)
        _capi.check(self._lib.ntr_group_set_camera(self._h, _p(o), _p(a)))

    def set_params(self, scene):
        desc, keep = _capi.make_desc(scene)
        _capi.check(self._lib.ntr_group_set_params(self._h, C.byref(desc)))

    def set_supersampling(self, factor):
        _capi.check(self._lib.ntr_group_set_supersampling(self._h, int(factor)))
        self.supersampling = int(factor)

    def set_supersampling_threshold(self, threshold):
        _capi.check(self._lib.ntr_group_set_supersampling_threshold(self._h, -1.0 if threshold is None else float(threshold)))
        self.supersampling_threshold = None if threshold is None else float(threshold)

    def refine_mask(self):
        """DeviceScene.refine_mask of the last group frame: every device's rows, their refined pixels summed."""
        w, h = self._window if self._window else (0, 0)
        return _refine_mask(self._lib.ntr_group_last_refine_mask, self._h, w, h)

    def render(self, fmt, dest=None):
        need = fmt.pitch * fmt.height
        out = np.zeros(need, dtype=np.uint8) if dest is None else dest
        buf = out if dest is None else np.frombuffer(dest, dtype=np.uint8)
        if buf.size < need:
            raise ValueError('the buffer is too small for an image with the given dimensions')
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_group_render(self._h, C.byref(fmt), _p(buf), buf.size))
        return out

    def render_views(self, fmt, cameras, dest=None):
        """DeviceScene.render_views over the group: whole views dealt to the devices in contiguous runs
        (ntr_group_render_views)."""
        origins, axes = camera_arrays(cameras, self.dim)
        out, buf = _views_dest(dest, len(origins), fmt)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_group_render_views(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt), _p(buf), buf.size))
        return out

    def render_views_aovs(self, fmt, cameras, aovs=AOV_NAMES, dest=None):
        """DeviceScene.render_views_aovs over the group: every device writes the frames and AOVs of its own views
        (ntr_group_render_views_aovs)."""
        origins, axes = camera_arrays(cameras, self.dim)
        out, buf = _views_dest(dest, len(origins), fmt)
        arrays, a = _new_aovs(aovs, len(origins), fmt, self.dim)
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_group_render_views_aovs(self._h, len(origins), _p(origins), _p(axes), C.byref(fmt), _p(buf),
                                                          buf.size, C.byref(a)))
        return out, arrays

    def render_device(self, fmt):
        """-> address of the frame on the first device (valid until the next render)"""
        ptr = C.c_void_p()
        self._window = (fmt.width, fmt.height)
        _capi.check(self._lib.ntr_group_render_device(self._h, C.byref(fmt), C.byref(ptr)))
        return ptr.value

    def abort(self):
        _capi.check(self._lib.ntr_group_abort(self._h))

    def counters(self):
        c = _capi.Counters()
        _capi.check(self._lib.ntr_group_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    def last_kernel_ms(self):
        ms = C.c_float()
        _capi.check(self._lib.ntr_group_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        return int(self._lib.ntr_group_launch_count(self._h))


class SharedFrame:
    """A frame buffer in the memory of one GPU that kernels of OTHER processes store into (one process per GPU):
    rank 0 allocates and exports it, the others import the handle (CUDA IPC)."""
    def __init__(self, device, nbytes=0, handle=None):
        self._lib = _capi.load()
        self.device, self.owner = int(device), handle is None
        ptr = C.c_void_p()
        if self.owner:
            _capi.check(self._lib.ntr_frame_alloc(self.device, int(nbytes), C.byref(ptr)))
        else:
            h = (C.c_ubyte * 64).from_buffer_copy(bytes(handle))
            _capi.check(self._lib.ntr_frame_import(self.device, h, C.byref(ptr)))
        self.ptr = ptr.value

    def export(self):
        h = (C.c_ubyte * 64)()
        _capi.check(self._lib.ntr_frame_export(C.c_void_p(self.ptr), h))
        return bytes(h)

    def fill(self, value, nbytes, stream=0):
        _capi.check(self._lib.ntr_frame_fill(self.device, C.c_void_p(self.ptr), int(value), int(nbytes), C.c_void_p(stream)))

    def download(self, fmt, dest, stream=0):
        buf = np.frombuffer(dest, dtype=np.uint8)
        _capi.check(self._lib.ntr_frame_download(self.device, C.c_void_p(self.ptr), C.byref(fmt), _p(buf), buf.size, C.c_void_p(stream)))

    def close(self):
        if self.ptr:
            (self._lib.ntr_frame_free if self.owner else self._lib.ntr_frame_release)(self.device, C.c_void_p(self.ptr))
            self.ptr = None


def device_count():
    return int(_capi.load().ntr_device_count())


def measure_fp32_peak(device=-1):
    out = C.c_float()
    _capi.check(_capi.load().ntr_measure_fp32_peak(device, C.byref(out)))
    return float(out.value)
