"""ctypes mirror of include/ntracer_b200.h and loader of the CUDA backend (libntracer_b200.so).

The product has no CPU path: if the shared library is missing, or it reports no sm_100 device,
every compute call raises.  Nothing here imports or falls back to oracle/.
"""
import ctypes as C
import os

import numpy as np

NTR_MAX_DIM = 16
NTR_MAX_CHANNELS = 16
NULL_NODE = 0xFFFFFFFF
LEAF_FLAG = 0x80000000
REF_SIMPLEX, REF_BATCH, REF_SOLID = 0, 1, 2
SCENE_BOX, SCENE_COMPOSITE = 0, 1

NTR_OK = 0
NTR_MAX_SUPERSAMPLING = 8
NTR_ERR_VALUE, NTR_ERR_MEMORY, NTR_ERR_RUNTIME, NTR_ERR_NO_DEVICE, NTR_ERR_ABORTED = -1, -2, -3, -4, -5


class Node(C.Structure):
    _fields_ = [('meta', C.c_uint32), ('w1', C.c_uint32), ('w2', C.c_uint32), ('w3', C.c_uint32)]


class SceneDesc(C.Structure):
    _fields_ = [
        ('dim', C.c_int32), ('kind', C.c_int32), ('batch_size', C.c_int32), ('root', C.c_uint32),
        ('n_nodes', C.c_uint32), ('nodes', C.c_void_p),
        ('n_leaf_refs', C.c_uint32), ('leaf_refs', C.c_void_p),
        ('n_simplex', C.c_uint32), ('simplex', C.c_void_p), ('simplex_mat', C.c_void_p),
        ('n_solids', C.c_uint32), ('solids', C.c_void_p), ('solid_mat', C.c_void_p),
        ('n_materials', C.c_uint32), ('materials', C.c_void_p),
        ('boundary', C.c_void_p),
        ('fov', C.c_float), ('shadows', C.c_int32), ('camera_light', C.c_int32),
        ('max_reflect_depth', C.c_int32), ('bg_gradient_axis', C.c_int32),
        ('ambient', C.c_float * 3), ('bg1', C.c_float * 3), ('bg2', C.c_float * 3), ('bg3', C.c_float * 3),
        ('n_point_lights', C.c_uint32), ('point_lights', C.c_void_p),
        ('n_global_lights', C.c_uint32), ('global_lights', C.c_void_p),
    ]


class Channel(C.Structure):
    _fields_ = [('f_r', C.c_float), ('f_g', C.c_float), ('f_b', C.c_float), ('f_c', C.c_float),
                ('bit_size', C.c_uint8), ('tfloat', C.c_uint8), ('pad_', C.c_uint8 * 2)]


class ImageFormat(C.Structure):
    _fields_ = [('width', C.c_int32), ('height', C.c_int32), ('pitch', C.c_int32), ('n_channels', C.c_int32),
                ('channels', Channel * NTR_MAX_CHANNELS),
                ('bytes_per_pixel', C.c_uint8), ('reversed', C.c_uint8), ('pad_', C.c_uint8 * 2)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        'primary_rays', 'reflection_rays', 'shadow_rays', 'node_steps', 'simplex_tests', 'solid_tests',
        'shaded_hits', 'queue_overflows', 'truncated_hit_lists')]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def make_image_format(width, height, channels, pitch=0, reversed=False):
    """channels: iterable of (bit_size, f_r, f_g, f_b[, f_c[, tfloat]]).  Validation follows
    ImageFormat.__new__ / im_set_channels (reference src/render.cpp:192-209,249-288)."""
    chans = [tuple(c) for c in channels]
    if len(chans) > NTR_MAX_CHANNELS:
        raise ValueError('too many channels')
    f = ImageFormat()
    bits = 0
    for i, c in enumerate(chans):
        bit_size, f_r, f_g, f_b = c[:4]
        f_c = c[4] if len(c) > 4 else 0.0
        tfloat = bool(c[5]) if len(c) > 5 else False
        if tfloat:
            if bit_size != 32:
                raise ValueError('if "tfloat" is true, "bit_size" can only be 32')
        elif bit_size > 31:
            raise ValueError('"bit_size" cannot be greater than 31 (unless "tfloat" is true)')
        elif bit_size < 1:
            raise ValueError('"bit_size" cannot be less than 1')
        f.channels[i] = Channel(f_r, f_g, f_b, f_c, bit_size, int(tfloat))
        bits += bit_size
    if bits > 16 * 8:
        raise ValueError('Too many bytes per pixel. The maximum is 16.')
    f.n_channels = len(chans)
    f.bytes_per_pixel = (bits + 7) // 8
    if width < 1 or height < 1:
        raise ValueError('width and height must be at least 1')
    if pitch < 0:
        raise ValueError('pitch cannot be negative')
    if pitch:
        if pitch < width * f.bytes_per_pixel:
            raise ValueError('"pitch" must be at least "width" times the size of one pixel in bytes')
    else:
        pitch = width * f.bytes_per_pixel
    f.width, f.height, f.pitch, f.reversed = width, height, pitch, int(bool(reversed))
    return f


class AovBuffers(C.Structure):
    """ntr_aov_buffers: per-pixel ids / depth / normals of a views call (NULL = not wanted), lengths in elements"""
    _fields_ = [('ids', C.c_void_p), ('depth', C.c_void_p), ('normals', C.c_void_p),
                ('ids_len', C.c_size_t), ('depth_len', C.c_size_t), ('normals_len', C.c_size_t)]


RGB8 = ((8, 1, 0, 0), (8, 0, 1, 0), (8, 0, 0, 1))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def make_desc(sc):
    """Build an ntr_scene_desc from a flat scene dict (see DESIGN.md 'scene file').
    Returns (desc, keepalive): keepalive holds the contiguous numpy arrays the pointers refer to."""
    dim = int(sc['dim'])
    kind = int(sc['kind'])
    d = SceneDesc()
    keep = {}

    def arr(name, dtype, shape=None):
        a = sc.get(name)
        if a is None:
            a = np.zeros((0,) if shape is None else shape, dtype=dtype)
        a = np.ascontiguousarray(a, dtype=dtype)
        keep[name] = a
        return a

    d.dim, d.kind = dim, kind
    d.batch_size = int(sc.get('batch_size', 1))
    params = np.asarray(sc['params'], dtype=np.float64)
    d.fov = float(params[0])
    d.root = NULL_NODE
    if kind == SCENE_COMPOSITE:
        nodes = arr('nodes', np.uint32).reshape(-1, 4)
        refs = arr('leaf_refs', np.uint32)
        simplex = arr('simplex', np.float32)
        smat = arr('simplex_mat', np.int32)
        solids = arr('solids', np.float32)
        solmat = arr('solid_mat', np.int32)
        mats = arr('materials', np.float32)
        bnd = arr('boundary', np.float32)
        pl = arr('point_lights', np.float32)
        gl = arr('global_lights', np.float32)
        stride = (dim + 1) * dim + 1
        sol_stride = 1 + 2 * dim * dim + dim
        if simplex.size % stride or solids.size % sol_stride or mats.size % 10 or nodes.size % 4:
            raise ValueError('scene arrays do not match the record sizes of a %d-dimensional scene' % dim)
        if smat.size != simplex.size // stride or solmat.size != solids.size // sol_stride:
            raise ValueError('one material index per simplex / solid is required')
        if bnd.size != 2 * dim:
            raise ValueError('boundary must hold 2 x %d floats' % dim)
        if pl.size % (dim + 3) or gl.size % (dim + 3):
            raise ValueError('lights are rows of %d floats' % (dim + 3))
        d.root = int(sc['root']) & 0xFFFFFFFF
        d.n_nodes, d.nodes = nodes.shape[0], _ptr(nodes)
        d.n_leaf_refs, d.leaf_refs = refs.size, _ptr(refs)
        d.n_simplex = simplex.size // stride
        d.simplex, d.simplex_mat = _ptr(simplex), _ptr(smat)
        d.n_solids = solids.size // (1 + 2 * dim * dim + dim)
        d.solids, d.solid_mat = _ptr(solids), _ptr(solmat)
        d.n_materials, d.materials = mats.size // 10, _ptr(mats)
        d.boundary = _ptr(bnd)
        d.shadows, d.camera_light = int(params[1]), int(params[2])
        d.max_reflect_depth, d.bg_gradient_axis = int(params[3]), int(params[4])
        for name in ('ambient', 'bg1', 'bg2', 'bg3'):
            v = np.asarray(sc[name], dtype=np.float32)
            setattr(d, name, (C.c_float * 3)(*[float(x) for x in v]))
        d.n_point_lights, d.point_lights = pl.size // (dim + 3), _ptr(pl)
        d.n_global_lights, d.global_lights = gl.size // (dim + 3), _ptr(gl)
    return d, keep


_LIB = None
_LIB_PATH = os.environ.get('NTR_B200_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libntracer_b200.so')


class BackendError(RuntimeError):
    pass


def lib_path():
    return _LIB_PATH


def load():
    """Load libntracer_b200.so (built in-tree by __graft_entry__.build()).  Raises if it is missing:
    there is deliberately no fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise BackendError('CUDA backend %s is not built (run `python -c "import __graft_entry__ as g; g.build()"`); '
                           'ntracer_b200 has no CPU fallback' % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    vp, i32, u32, f32p = C.c_void_p, C.c_int, C.c_uint32, C.POINTER(C.c_float)
    sig = {
        'ntr_abi_version': (C.c_int, []),
        'ntr_last_error': (C.c_char_p, []),
        'ntr_device_count': (C.c_int, []),
        'ntr_scene_create': (C.c_int, [C.POINTER(SceneDesc), i32, C.POINTER(vp)]),
        'ntr_scene_destroy': (None, [vp]),
        'ntr_scene_set_camera': (C.c_int, [vp, vp, vp]),
        'ntr_scene_set_params': (C.c_int, [vp, C.POINTER(SceneDesc)]),
        'ntr_scene_set_supersampling': (C.c_int, [vp, i32]),
        'ntr_scene_set_supersampling_threshold': (C.c_int, [vp, C.c_float]),
        'ntr_scene_set_projection': (C.c_int, [vp, i32, C.c_float]),
        'ntr_camera_rays': (C.c_int, [vp, i32, i32, vp, vp]),
        'ntr_camera_rays_device': (C.c_int, [vp, i32, i32, vp, vp, vp]),
        'ntr_last_refine_mask': (C.c_int, [vp, vp, C.c_size_t, C.POINTER(C.c_uint64)]),
        'ntr_render': (C.c_int, [vp, C.POINTER(ImageFormat), vp, C.c_size_t]),
        'ntr_render_device': (C.c_int, [vp, C.POINTER(ImageFormat), vp, C.c_size_t, vp, i32, i32, i32]),
        'ntr_render_begin': (C.c_int, [vp, C.POINTER(ImageFormat), vp, C.c_size_t, C.POINTER(C.c_uint64)]),
        'ntr_render_end': (C.c_int, [vp, C.c_uint64]),
        'ntr_render_views': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t]),
        'ntr_render_views_device': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t, vp]),
        'ntr_render_views_aovs': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t, C.POINTER(AovBuffers)]),
        'ntr_render_views_aovs_device': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t,
                                                   C.POINTER(AovBuffers), vp]),
        'ntr_render_rays': (C.c_int, [vp, u32, vp, vp, vp, C.POINTER(AovBuffers)]),
        'ntr_render_rays_device': (C.c_int, [vp, u32, vp, vp, vp, C.POINTER(AovBuffers), vp]),
        'ntr_render_float': (C.c_int, [vp, i32, i32, vp]),
        'ntr_calculate_color': (C.c_int, [vp, i32, i32, i32, i32, f32p]),
        'ntr_primary_hit_ids': (C.c_int, [vp, i32, i32, vp, vp]),
        'ntr_trace_rays': (C.c_int, [vp, u32, vp, vp, C.c_float, C.c_float, vp, vp, vp, vp, vp]),
        'ntr_trace_rays_hits': (C.c_int, [vp, u32, vp, vp, C.c_float, C.c_float, vp, vp, vp, vp, vp, i32, vp, vp]),
        'ntr_occludes_rays': (C.c_int, [vp, u32, vp, vp, vp, vp, vp, vp, vp]),
        'ntr_abort': (C.c_int, [vp]),
        'ntr_get_counters': (C.c_int, [vp, C.POINTER(Counters)]),
        'ntr_set_instrumented': (C.c_int, [vp, i32]),
        'ntr_last_kernel_ms': (C.c_int, [vp, f32p]),
        'ntr_launch_count': (C.c_uint64, [vp]),
        'ntr_measure_fp32_peak': (C.c_int, [i32, f32p]),
        'ntr_simplex_from_points': (C.c_int, [i32, u32, vp, vp]),
        'ntr_build_kdtree': (C.c_int, [i32, u32, vp, vp, i32, i32, C.c_float, C.c_float, C.POINTER(vp), C.POINTER(u32),
                                       C.POINTER(vp), C.POINTER(u32), C.POINTER(u32), vp]),
        'ntr_build_kdtree_culled': (C.c_int, [i32, u32, vp, vp, vp, u32, vp, vp, vp, i32, i32, C.c_float, C.c_float, C.POINTER(vp),
                                              C.POINTER(u32), C.POINTER(vp), C.POINTER(u32), C.POINTER(u32), vp]),
        'ntr_free': (None, [vp]),
        'ntr_group_items': (C.c_int, [i32, u32, vp, vp, i32, vp]),
        'ntr_group_create': (C.c_int, [C.POINTER(SceneDesc), i32, vp, C.POINTER(vp)]),
        'ntr_group_destroy': (None, [vp]),
        'ntr_group_size': (C.c_int, [vp]),
        'ntr_group_set_camera': (C.c_int, [vp, vp, vp]),
        'ntr_group_set_params': (C.c_int, [vp, C.POINTER(SceneDesc)]),
        'ntr_group_set_supersampling': (C.c_int, [vp, i32]),
        'ntr_group_set_supersampling_threshold': (C.c_int, [vp, C.c_float]),
        'ntr_group_set_projection': (C.c_int, [vp, i32, C.c_float]),
        'ntr_group_last_refine_mask': (C.c_int, [vp, vp, C.c_size_t, C.POINTER(C.c_uint64)]),
        'ntr_group_render': (C.c_int, [vp, C.POINTER(ImageFormat), vp, C.c_size_t]),
        'ntr_group_render_device': (C.c_int, [vp, C.POINTER(ImageFormat), C.POINTER(vp)]),
        'ntr_group_render_views': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t]),
        'ntr_group_render_views_aovs': (C.c_int, [vp, i32, vp, vp, C.POINTER(ImageFormat), vp, C.c_size_t, C.POINTER(AovBuffers)]),
        'ntr_group_render_rays': (C.c_int, [vp, u32, vp, vp, vp, C.POINTER(AovBuffers)]),
        'ntr_group_abort': (C.c_int, [vp]),
        'ntr_group_get_counters': (C.c_int, [vp, C.POINTER(Counters)]),
        'ntr_group_last_kernel_ms': (C.c_int, [vp, f32p]),
        'ntr_group_launch_count': (C.c_uint64, [vp]),
        'ntr_frame_alloc': (C.c_int, [i32, C.c_size_t, C.POINTER(vp)]),
        'ntr_frame_free': (C.c_int, [i32, vp]),
        'ntr_frame_export': (C.c_int, [vp, vp]),
        'ntr_frame_import': (C.c_int, [i32, vp, C.POINTER(vp)]),
        'ntr_frame_release': (C.c_int, [i32, vp]),
        'ntr_frame_fill': (C.c_int, [i32, vp, i32, C.c_size_t, vp]),
        'ntr_frame_download': (C.c_int, [i32, vp, C.POINTER(ImageFormat), vp, C.c_size_t, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export what the header declares
        fn.restype, fn.argtypes = res, args
    _LIB = lib
    return lib


EXPORTED_SYMBOLS = (
    'ntr_abi_version', 'ntr_last_error', 'ntr_device_count', 'ntr_scene_create', 'ntr_scene_destroy',
    'ntr_scene_set_camera', 'ntr_scene_set_params', 'ntr_scene_set_supersampling', 'ntr_render', 'ntr_render_device', 'ntr_render_begin',
    'ntr_render_end', 'ntr_render_views', 'ntr_render_views_device', 'ntr_render_views_aovs', 'ntr_render_views_aovs_device',
    'ntr_render_rays', 'ntr_render_rays_device', 'ntr_render_float',
    'ntr_calculate_color', 'ntr_primary_hit_ids', 'ntr_trace_rays', 'ntr_trace_rays_hits', 'ntr_occludes_rays', 'ntr_abort',
    'ntr_get_counters', 'ntr_set_instrumented', 'ntr_last_kernel_ms', 'ntr_launch_count',
    'ntr_measure_fp32_peak', 'ntr_simplex_from_points', 'ntr_build_kdtree', 'ntr_build_kdtree_culled', 'ntr_free', 'ntr_group_items',
    'ntr_group_create', 'ntr_group_destroy', 'ntr_group_size', 'ntr_group_set_camera', 'ntr_group_set_params',
    'ntr_group_set_supersampling', 'ntr_scene_set_supersampling_threshold', 'ntr_last_refine_mask',
    'ntr_group_set_supersampling_threshold', 'ntr_group_last_refine_mask',
    'ntr_scene_set_projection', 'ntr_group_set_projection', 'ntr_camera_rays', 'ntr_camera_rays_device',
    'ntr_group_render', 'ntr_group_render_device', 'ntr_group_render_views', 'ntr_group_render_views_aovs', 'ntr_group_render_rays',
    'ntr_group_abort', 'ntr_group_get_counters',
    'ntr_group_last_kernel_ms', 'ntr_group_launch_count',
    'ntr_frame_alloc', 'ntr_frame_free', 'ntr_frame_export', 'ntr_frame_import', 'ntr_frame_release',
    'ntr_frame_fill', 'ntr_frame_download')


class AbortedError(RuntimeError):
    """A render call ended early because ntr_abort() was called (NTR_ERR_ABORTED)."""


def check(status):
    """Translate an ntr_status into the exception the reference raises for the same condition
    (PY_EXCEPT_HANDLERS, reference src/py_common.hpp:39-47)."""
    if status == NTR_OK:
        return
    msg = (load().ntr_last_error() or b'').decode('utf-8', 'replace')
    if status == NTR_ERR_VALUE:
        raise ValueError(msg)
    if status == NTR_ERR_MEMORY:
        raise MemoryError(msg)
    if status == NTR_ERR_NO_DEVICE:
        raise BackendError(msg or 'no sm_100 CUDA device: ntracer_b200 has no CPU fallback')
    if status == NTR_ERR_ABORTED:
        raise AbortedError(msg)
    raise RuntimeError(msg)
