"""ntracer_b200.tracern -- host-side mirror of the reference's `ntracer.tracern` / `tracer{3..8}` modules
(reference src/ntracer_body.hpp: the 31 Python types and 5 module functions, doc/ntracer.rst:452-1975) for
the render path: the geometry / scene classes a script builds, flattened into the device arena and rendered
by the CUDA backend through the C ABI.

Same names, argument meaning and error behaviour as the reference; the arithmetic of the *render path*
(Scene.calculate_color, KDNode.intersects / occludes, the renderers) runs on the GPU.  Host-side helper math
(vectors, matrices, Triangle.from_points, the k-d tree builder) is plain numpy float32 -- it is scene set-up,
not the hot path.  The dimension is a run-time attribute like in the reference's generic module.
"""
import math
import numbers

import numpy as np

from . import _capi
from .backend import DeviceGroup, DeviceScene, FLT_MAX, projection_args
from . import render as _render
from .render import Color, LockedError, Material, Scene, _color_tuple, _encode_floats

BATCH_SIZE = 4      # lanes of a TriangleBatch; the reference's SSE build has v_real::size == 4
CUBE, SPHERE = 1, 2
_F = np.float32
ROUNDING_FUZZ = _F(10) * np.finfo(np.float32).eps        # src/tracer.hpp:25


def _check_dimension(d):
    if d < 3:
        raise ValueError('dimension cannot be smaller than 3')
    if d > _capi.NTR_MAX_DIM:
        raise ValueError('dimension cannot be greater than %d' % _capi.NTR_MAX_DIM)
    return int(d)


# ---------------------------------------------------------------------------------------------------------
class Vector:
    """Vector(dimension[,values]) -- doc/ntracer.rst:1704-1822"""
    __slots__ = ('_v',)

    def __init__(self, dimension, values=None):
        if isinstance(dimension, Vector) and values is None:
            self._v = dimension._v.copy()
            return
        _check_dimension(dimension)
        if values is None:
            self._v = np.zeros(dimension, _F)
        else:
            v = np.array([float(x) for x in values], _F)
            if v.size != dimension:
                raise TypeError('this object has a dimension of %d and cannot be initialized with %d values' % (dimension, v.size))
            self._v = v

    @classmethod
    def _wrap(cls, arr):
        o = object.__new__(Vector)
        o._v = np.ascontiguousarray(arr, _F)
        return o

    @staticmethod
    def axis(dimension, axis, length=1):
        _check_dimension(dimension)
        if not 0 <= axis < dimension:
            raise ValueError('axis must be between 0 and dimension-1')
        v = np.zeros(dimension, _F)
        v[axis] = length
        return Vector._wrap(v)

    dimension = property(lambda self: int(self._v.size))

    def __len__(self): return int(self._v.size)
    def __getitem__(self, i): return float(self._v[i])
    def __iter__(self): return (float(x) for x in self._v)
    def __buffer__(self, flags): return memoryview(self._v)
    def __array__(self, dtype=None, copy=None): return self._v.astype(dtype) if dtype else self._v
    def __repr__(self): return 'Vector(%d,(%s))' % (self._v.size, ','.join(repr(float(x)) for x in self._v))
    def __str__(self): return '<%s>' % ','.join('%g' % float(x) for x in self._v)
    def __hash__(self): return hash(self._v.tobytes())

    def _coerce(self, b):
        if isinstance(b, Vector):
            if b._v.size != self._v.size:
                raise TypeError('cannot perform vector operations on vectors of different dimension')
            return b._v
        return None

    def __add__(self, b):
        o = self._coerce(_as_vector(b, self._v.size))
        return Vector._wrap(self._v + o)

    def __sub__(self, b):
        o = self._coerce(_as_vector(b, self._v.size))
        return Vector._wrap(self._v - o)

    def __mul__(self, b):
        if isinstance(b, (Vector, Matrix)):
            return NotImplemented
        return Vector._wrap(self._v * _F(b))
    __rmul__ = __mul__

    def __truediv__(self, b): return Vector._wrap(self._v / _F(b))
    __div__ = __truediv__
    def __neg__(self): return Vector._wrap(-self._v)
    def __abs__(self): return self.absolute()
    def __eq__(self, b): return isinstance(b, Vector) and b._v.size == self._v.size and bool(np.all(self._v == b._v))
    def __reduce__(self): return (_render._vector_unpickle, (self.dimension, _encode_floats(self._v)))       # ntracer_body.hpp:2016-2020
    def __ne__(self, b): return not self.__eq__(b)

    def square(self): return float(np.dot(self._v, self._v))
    def absolute(self): return float(np.sqrt(_F(np.dot(self._v, self._v))))
    def unit(self): return Vector._wrap(self._v / np.sqrt(_F(np.dot(self._v, self._v))))
    def apply(self, f): return Vector(self._v.size, [f(float(x)) for x in self._v])

    def set_c(self, index, value):
        v = self._v.copy()
        v[index] = value
        return Vector._wrap(v)


def _as_vector(x, dim=None):
    if isinstance(x, Vector):
        v = x
    else:
        seq = list(x)
        v = Vector(len(seq) if dim is None else dim, seq)
    if dim is not None and v.dimension != dim:
        raise TypeError('object has a dimension of %d instead of %d' % (v.dimension, dim))
    return v


class Matrix:
    """Matrix(dimension,values) -- doc/ntracer.rst:1114-1207; row-major, `values` is the flat sequence"""
    __slots__ = ('_m',)

    def __init__(self, dimension, values=None):
        _check_dimension(dimension)
        if values is None:
            self._m = np.zeros((dimension, dimension), _F)
            return
        vals = list(values)
        if len(vals) == dimension * dimension:
            m = np.array([float(x) for x in vals], _F).reshape(dimension, dimension)
        elif len(vals) == dimension:
            m = np.array([[float(x) for x in row] for row in vals], _F)
            if m.shape != (dimension, dimension):
                raise TypeError('matrix rows must have %d items' % dimension)
        else:
            raise TypeError('a matrix of dimension %d needs %d values or %d rows' % (dimension, dimension ** 2, dimension))
        self._m = m

    @classmethod
    def _wrap(cls, arr):
        o = object.__new__(Matrix)
        o._m = np.ascontiguousarray(arr, _F)
        return o

    dimension = property(lambda self: int(self._m.shape[0]))
    values = property(lambda self: tuple(float(x) for x in self._m.ravel()))

    def __len__(self): return int(self._m.shape[0])
    def __getitem__(self, i): return Vector._wrap(self._m[i].copy())
    def __eq__(self, b): return isinstance(b, Matrix) and self._m.shape == b._m.shape and bool(np.all(self._m == b._m))
    def __reduce__(self): return (_render._matrix_unpickle, (self.dimension, _encode_floats(self._m.ravel())))  # :2347-2351
    def __repr__(self): return 'Matrix(%d,%r)' % (self.dimension, self.values)

    def __mul__(self, b):
        if isinstance(b, Matrix):
            return Matrix._wrap(self._m @ b._m)
        if isinstance(b, Vector):
            return Vector._wrap(self._m @ b._v)
        return NotImplemented

    def determinant(self): return float(np.linalg.det(self._m.astype(np.float64)))

    def inverse(self):
        try:
            return Matrix._wrap(np.linalg.inv(self._m.astype(np.float64)))
        except np.linalg.LinAlgError:
            raise ValueError('matrix is singular')

    def transpose(self): return Matrix._wrap(self._m.T.copy())

    @staticmethod
    def identity(dimension):
        _check_dimension(dimension)
        return Matrix._wrap(np.eye(dimension, dtype=_F))

    @staticmethod
    def scale(*args):
        if len(args) == 1:
            v = _as_vector(args[0])
            return Matrix._wrap(np.diag(v._v))
        d, mag = args
        _check_dimension(d)
        return Matrix._wrap(np.eye(d, dtype=_F) * _F(mag))

    @staticmethod
    def reflection(axis):
        a = _as_vector(axis)._v
        sq = _F(np.dot(a, a))
        return Matrix._wrap(np.eye(a.size, dtype=_F) - 2 * np.outer(a, a) / sq)      # geometry.hpp:602-608

    @staticmethod
    def rotation(a, b, theta):
        a, b = _as_vector(a)._v, _as_vector(b, len(a))._v
        c, s = _F(math.cos(theta) - 1), _F(math.sin(theta))
        # geometry.hpp:579-591: r[row][col] = a[row]*(a[col]*c - b[col]*s) + b[row]*(b[col]*c + a[col]*s) (+1 on the diagonal)
        m = np.outer(a, a * c - b * s) + np.outer(b, b * c + a * s) + np.eye(a.size, dtype=_F)
        return Matrix._wrap(m)


def dot(a, b):
    a = _as_vector(a)
    return float(np.dot(a._v, _as_vector(b, a.dimension)._v))


def cross(vectors):
    """Generalized cross product of D-1 vectors (geometry.hpp:858-893)."""
    vs = [_as_vector(v) for v in vectors]
    d = vs[0].dimension
    if len(vs) != d - 1:
        raise ValueError('the number of vectors must be exactly one less than their dimension')
    m = np.stack([v._v for v in vs]).astype(np.float64)        # (D-1) x D
    r = np.zeros(d, np.float64)
    f = 1.0 if d % 2 else -1.0
    for i in range(d):
        r[i] = f * np.linalg.det(np.delete(m, i, axis=1).T)
        f = -f
    return Vector._wrap(r)


# ---------------------------------------------------------------------------------------------------------
class CameraAxes:
    def __init__(self, cam): self._cam = cam
    def __len__(self): return self._cam.dimension
    def __getitem__(self, i): return Vector._wrap(self._cam._axes[i].copy())

    def __setitem__(self, i, v):
        self._cam._axes[i] = _as_vector(v, self._cam.dimension)._v


class Camera:
    """Camera(dimension) -- src/camera.hpp:7-46, doc/ntracer.rst:598-647"""
    def __init__(self, dimension):
        _check_dimension(dimension)
        self._origin = np.zeros(dimension, _F)
        self._axes = np.eye(dimension, dtype=_F)

    dimension = property(lambda self: int(self._origin.size))
    axes = property(lambda self: CameraAxes(self))

    @property
    def origin(self): return Vector._wrap(self._origin.copy())

    @origin.setter
    def origin(self, v): self._origin = _as_vector(v, self.dimension)._v.copy()

    def translate(self, offset):                 # camera.hpp:17-19
        o = _as_vector(offset, self.dimension)._v
        self._origin = self._origin + o @ self._axes

    def transform(self, m):                      # camera.hpp:21-23: t_orientation.mult_transpose(m)
        self._axes = (self._axes @ m._m.T).astype(_F)

    def normalize(self):                         # camera.hpp:25-36 (Gram-Schmidt)
        a = self._axes
        new = np.zeros_like(a)
        new[0] = a[0] / np.sqrt(np.dot(a[0], a[0]))
        for i in range(1, a.shape[0]):
            x = np.zeros(a.shape[1], _F)
            for j in range(i - 1):
                x += np.dot(a[i], a[j]) * a[j]
            v = a[i] - x
            new[i] = v / np.sqrt(np.dot(v, v))
        self._axes = new

    def _copy(self):
        c = Camera(self.dimension)
        c._origin, c._axes = self._origin.copy(), self._axes.copy()
        return c


class AABB:
    """AABB(dimension[,start,end]) -- doc/ntracer.rst:465-542"""
    def __init__(self, dimension, start=None, end=None):
        _check_dimension(dimension)
        self.start = Vector(dimension, [-FLT_MAX] * dimension) if start is None else _as_vector(start, dimension)
        self.end = Vector(dimension, [FLT_MAX] * dimension) if end is None else _as_vector(end, dimension)

    dimension = property(lambda self: self.start.dimension)

    def __reduce__(self):                       # ntracer_body.hpp:2559-2563
        return (_render._aabb_unpickle, (self.dimension, _encode_floats(np.concatenate([self.start._v, self.end._v]))))

    def left(self, axis, split):
        return AABB(self.dimension, self.start, self.end.set_c(axis, split))

    def right(self, axis, split):
        return AABB(self.dimension, self.start.set_c(axis, split), self.end)

    def _center(self):
        return (self.start._v + self.end._v) * _F(0.5)

    @staticmethod
    def _check_proto(self_dim, primitive, allowed, what):
        if isinstance(primitive, (Primitive, PrimitiveBatch)):
            raise TypeError('Instances of Primitive cannot be used directly. Use PrimitivePrototype instead.')
        if not isinstance(primitive, allowed):
            raise TypeError('object must be an instance of ' + what)
        if primitive.dimension != self_dim:
            raise TypeError('cannot perform intersection test on object with different dimension')

    def intersects(self, primitive):
        """Exact box/primitive overlap with non-zero volume (src/tracer.hpp:1459-1675): separating-axis tests for
        simplexes (face normal, then every edge normal projected onto every coordinate hyperplane), for hypercubes
        (cube normals and their projections) and a closest-point test for hyperspheres.  Touching does not count.
        Arithmetic in float32 like the reference."""
        AABB._check_proto(self.dimension, primitive, PrimitivePrototype, __name__ + '.PrimitivePrototype')
        if isinstance(primitive, TriangleBatchPrototype):
            b = primitive.boundary
            if np.any(b.start._v >= self.end._v) or np.any(b.end._v <= self.start._v):
                return False
            return any(self._simplex_overlap(t) for t in primitive._protos)     # miss.all() -> False (:1559-1585)
        if isinstance(primitive, TrianglePrototype):
            b = primitive.boundary
            if np.any(b.start._v >= self.end._v) or np.any(b.end._v <= self.start._v):
                return False
            return self._simplex_overlap(primitive)
        return self._solid_overlap(primitive)

    def _simplex_overlap(self, tp):
        """the part of aabb::intersects(triangle_prototype) after the bounding-box rejection (:1470-1509)"""
        d = self.dimension
        half = (self.end._v - self.start._v) / _F(2)
        origin = self._center()
        fn = tp.face_normal._v
        pts = np.stack([pd.point._v for pd in tp.point_data])           # D points
        n_offset = _F(np.dot(fn, pts[0]))
        po = _F(np.dot(origin, fn))
        b_max = _F(np.sum(np.abs(half * fn)))
        if po + b_max < n_offset or po - b_max > n_offset:
            return False
        for pd in tp.point_data:
            axis = pd.edge_normal._v
            for j in range(d):
                keep = np.arange(d) != j
                vals = pts[:, keep] @ axis[keep]
                t_min, t_max = _F(vals.min()), _F(vals.max())
                po = _F(np.dot(origin[keep], axis[keep]))
                b_radius = _F(np.sum(np.abs(half[keep] * axis[keep])))
                # a zero radius means the axis is parallel to the dropped coordinate: the test says nothing (:1503-1505)
                if b_radius != 0 and (po + b_radius <= t_min or po - b_radius >= t_max):
                    return False
        return True

    def intersects_flat(self, primitive, skip):
        """aabb::intersects_flat (:1512-1541, 1590-1625): the same test with coordinate `skip` ignored, used by the
        builder for primitives lying in a split plane."""
        AABB._check_proto(self.dimension, primitive, (TrianglePrototype, TriangleBatchPrototype),
                          '%s.TrianglePrototype or %s.TriangleBatchPrototype' % (__name__, __name__))
        d = self.dimension
        b = primitive.boundary
        k = np.arange(d) != skip
        if np.any(b.start._v[k] >= self.end._v[k]) or np.any(b.end._v[k] <= self.start._v[k]):
            return False
        protos = primitive._protos if isinstance(primitive, TriangleBatchPrototype) else (primitive,)
        half = (self.end._v - self.start._v) / _F(2)
        origin = self._center()

        def lane(tp):
            pts = [pd.point._v for pd in tp.point_data]
            for i, pd in enumerate(tp.point_data):
                axis = pd.edge_normal._v
                t_max = _F(np.dot(pts[0][k], axis[k]))
                t_min = _F(np.dot(pts[i if i else 1][k], axis[k]))
                if t_min > t_max:
                    t_min, t_max = t_max, t_min
                po = _F(np.dot(origin[k], axis[k]))
                b_max = _F(np.sum(np.abs(half[k] * axis[k])))
                if po + b_max <= t_min or po - b_max >= t_max:
                    return False
            return True
        return any(lane(t) for t in protos)

    def _solid_overlap(self, sp):
        """aabb::intersects(solid_prototype) (:1628-1675)"""
        d = self.dimension
        s = sp.primitive
        half = (self.end._v - self.start._v) / _F(2)
        center = self._center()
        pos = s.position._v
        if sp.type == CUBE:
            b = sp.boundary
            if np.any(self.end._v <= b.start._v) or np.any(self.start._v >= b.end._v):
                return False
            comps = s.orientation._m                                    # cube_component(i) = column i

            def separated(axis):                                        # box_axis_test (:1628-1639)
                a_po, b_po = _F(np.dot(pos, axis)), _F(np.dot(center, axis))
                a_max = _F(np.sum(np.abs(comps.T @ axis)))
                b_max = _F(np.sum(np.abs(half * axis)))
                return b_po + b_max < a_po - a_max or b_po - b_max > a_po + a_max
            for i in range(d):
                normal = s.inv_orientation._m[i]                        # cube_normal(i) = row i of the inverse
                if separated(normal):
                    return False
                sq = _F(np.dot(normal, normal))
                for j in range(d):                                      # the normal projected onto each coordinate hyperplane
                    axis = normal * -normal[j]
                    axis[j] += sq
                    if separated(axis):
                        return False
            return True
        box_p = pos - s.inv_orientation._m @ center
        closest = np.zeros(d, _F)
        for i in range(d):
            comp = s.orientation._m[i] * half[i]
            x = _F(np.dot(box_p, comp)) / _F(np.dot(comp, comp))
            closest = closest + _F(min(1.0, max(-1.0, float(x)))) * comp
        diff = pos - closest
        return bool(_F(np.dot(diff, diff)) < 1)


# ---------------------------------------------------------------------------------------------------------
_PROBE_MATERIAL = Material((1, 1, 1))       # opaque: KDNode.intersects materialises opaque hits only


class Primitive:
    def __init__(self, *a, **k):
        if type(self) is Primitive:
            raise TypeError('the Primitive type cannot be instantiated directly')

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k != '_probe'}

    def _probe_leaf(self):
        """A one-item tree around a copy of this primitive's geometry: the single-primitive ray test runs on the GPU
        through the same kernels as everything else (there is no CPU path).  Geometry is immutable, so it is cached."""
        leaf = self.__dict__.get('_probe')
        if leaf is None:
            leaf = self._probe = KDLeaf([self._twin()])
        return leaf

    def intersects(self, origin, direction):
        """-> RayIntersection or None (src/ntracer_body.hpp:1002-1019): triangle::intersects / solid::intersects for one
        ray, whatever the material's opacity."""
        hits = self._probe_leaf().intersects(origin, direction)
        if not hits:
            return None
        h = hits[-1]
        return RayIntersection(h.dist, h.origin, h.normal, self)


class PrimitiveBatch:
    def __init__(self, *a, **k):
        if type(self) is PrimitiveBatch:
            raise TypeError('the PrimitiveBatch type cannot be instantiated directly')

    __getstate__ = Primitive.__getstate__
    _probe_leaf = Primitive._probe_leaf

    def intersects(self, origin, direction, index=-1):
        """-> RayIntersection (batch_index = the lane that was hit) or None; lane `index` is ignored
        (src/ntracer_body.hpp:1038-1056, triangle_batch::intersects tracer.hpp:551-599)."""
        leaf = self._probe_leaf()
        hits = leaf.intersects(origin, direction, source=leaf[0] if index >= 0 else None, batch_index=index)
        if not hits:
            return None
        h = hits[-1]
        return RayIntersection(h.dist, h.origin, h.normal, self, h.batch_index)


class Triangle(Primitive):
    """Triangle(p1,face_normal,edge_normals,material): a (D-1)-simplex (src/tracer.hpp:392-488)"""
    def __init__(self, p1, face_normal, edge_normals, material):
        self.p1 = _as_vector(p1)
        d = self.p1.dimension
        self.face_normal = _as_vector(face_normal, d)
        en = [_as_vector(e, d) for e in edge_normals]
        if len(en) != d - 1:
            raise ValueError('a triangle needs exactly dimension-1 edge normals')
        self.edge_normals = tuple(en)
        if not isinstance(material, Material):
            raise TypeError('material must be an instance of Material')
        self.material = material
        self.d = float(-np.dot(self.face_normal._v, self.p1._v))       # recalculate_d, tracer.hpp:472-474

    dimension = property(lambda self: self.p1.dimension)

    def _rows(self):
        """p1, face_normal, edge normals: the rows of the reference's pickle payload (ntracer_body.hpp:1217-1232)"""
        return np.stack([self.p1._v, self.face_normal._v] + [e._v for e in self.edge_normals])

    def __reduce__(self):
        return (_render._triangle_unpickle, (self.dimension, _encode_floats(self._rows().ravel()), self.material))

    def _twin(self):
        return Triangle(self.p1, self.face_normal, self.edge_normals, _PROBE_MATERIAL)

    @staticmethod
    def from_points(points, material):          # tracer.hpp:442-462
        pts = [_as_vector(p) for p in points]
        n = pts[0].dimension
        if len(pts) != n:
            raise ValueError('a triangle needs exactly "dimension" points')
        vs = [pts[i + 1] - pts[0] for i in range(n - 1)]
        N = cross(vs)
        sq = N.square()
        edges = []
        for i in range(n - 1):
            tmp = list(vs)
            tmp[i] = N
            edges.append(cross(tmp) / sq)
        return Triangle(pts[0], N, edges, material)

    def to_points(self):                        # tracer.hpp:490-506
        n = self.dimension
        out = [self.p1]
        for i in range(n - 1):
            tmp = list(self.edge_normals)
            tmp[i] = self.face_normal
            out.append(cross(tmp) + self.p1)
        return tuple(out)

    def _row(self):
        return np.concatenate([self.face_normal._v, np.array([self.d], _F), self.p1._v] + [e._v for e in self.edge_normals])


class TriangleBatch(PrimitiveBatch):
    """TriangleBatch(triangles): BATCH_SIZE simplexes tested together (src/tracer.hpp:532-641)"""
    def __init__(self, triangles):
        ts = list(triangles)
        if len(ts) != BATCH_SIZE:
            raise ValueError('a TriangleBatch requires exactly %d triangles' % BATCH_SIZE)
        for t in ts:
            if not isinstance(t, Triangle):
                raise TypeError('object is not an instance of Triangle')
        self._t = tuple(ts)

    dimension = property(lambda self: self._t[0].dimension)
    def __len__(self): return BATCH_SIZE
    def __getitem__(self, i): return self._t[i]

    def __reduce__(self):                       # [row][coordinate][lane], then the lanes' materials (render.cpp:1722-1732)
        rows = np.stack([t._rows() for t in self._t], axis=-1)
        return (_render._triangle_batch_unpickle, (BATCH_SIZE, self.dimension, _encode_floats(rows.ravel())) + tuple(t.material for t in self._t))

    def _twin(self):
        return TriangleBatch([t._twin() for t in self._t])


class Solid(Primitive):
    """Solid(type,position,orientation,material) (src/tracer.hpp:231-289)"""
    def __init__(self, type, position, orientation, material):
        if type not in (CUBE, SPHERE):
            raise ValueError('invalid shape type')
        self.type = type
        self.position = _as_vector(position)
        if not isinstance(orientation, Matrix) or orientation.dimension != self.position.dimension:
            raise TypeError('the orientation and position must have the same dimension')
        self.orientation = orientation
        self.inv_orientation = orientation.inverse()
        if not isinstance(material, Material):
            raise TypeError('material must be an instance of Material')
        self.material = material

    dimension = property(lambda self: self.position.dimension)

    def __reduce__(self):                       # type byte, orientation, position (render.cpp:1733-1743)
        data = bytes([self.type]) + _encode_floats(self.orientation._m.ravel()) + _encode_floats(self.position._v)
        return (_render._solid_unpickle, (self.dimension, data, self.material))

    def _twin(self):
        return Solid(self.type, self.position, self.orientation, _PROBE_MATERIAL)

    def _hit_frame(self, o, d):
        """What solid::intersects leaves in `normal` for a ray that hits (src/tracer.hpp:126-173, 251-276), recomputed on
        the host for RayIntersection.origin / .normal: the hit is found in the solid's frame and carried back with
        `orientation` -- the normal is NOT renormalised (SURVEY 8a-Q8) and the origin follows the reference's frame
        arithmetic as written (Q5).  -> (origin, normal) as float32 arrays, or None if this arithmetic finds no hit."""
        n = self.dimension
        lo = (self.inv_orientation._m @ o - self.position._v).astype(_F)
        ld = (self.inv_orientation._m @ d).astype(_F)
        if self.type == CUBE:
            for i in range(n):
                if ld[i] == 0:
                    continue
                face = _F(1) if ld[i] < 0 else _F(-1)
                dist = (face - lo[i]) / ld[i]
                if not dist > 0:
                    continue
                p = (ld * dist + lo).astype(_F)
                p[i] = face
                others = np.arange(n) != i
                if np.any(np.abs(p[others]) > 1 + ROUNDING_FUZZ):
                    continue
                nd = np.zeros(n, _F)
                nd[i] = face
                return (self.orientation._m @ (p + self.position._v)).astype(_F), (self.orientation._m @ nd).astype(_F)
            return None
        a = _F(np.dot(ld, ld))
        b = _F(2) * _F(np.dot(ld, lo))
        c = _F(np.dot(lo, lo)) - _F(1)
        disc = b * b - _F(4) * a * c
        if disc < 0:
            return None
        dist = (-b - np.sqrt(disc)) / (_F(2) * a)
        p = (lo + ld * dist).astype(_F)
        return (self.orientation._m @ (p + self.position._v)).astype(_F), (self.orientation._m @ p).astype(_F)

    def _row(self):
        return np.concatenate([np.array([self.type], _F), self.orientation._m.ravel(), self.inv_orientation._m.ravel(), self.position._v])


class PrimitivePrototype:
    pass


class TrianglePointDatum:
    def __init__(self, point, edge_normal): self.point, self.edge_normal = point, edge_normal


class TriangleBatchPointDatum:
    """point / edge_normal of vertex j for every lane of a batch (indexable by lane)"""
    def __init__(self, point, edge_normal): self.point, self.edge_normal = point, edge_normal


class TrianglePrototype(PrimitivePrototype):
    """TrianglePrototype(points[,material]) (src/ntracer_body.hpp:2658-2720)"""
    def __init__(self, points, material=None):
        if isinstance(points, Triangle):
            if material is not None:
                raise TypeError('if "points" is an instance of Triangle, "material" must be None')
            tri, pts = points, list(points.to_points())
        else:
            if material is None:
                raise TypeError('if "points" is not an instance of Triangle, "material" cannot be None')
            pts = [_as_vector(p) for p in points]
            tri = Triangle.from_points(pts, material)
        self.primitive = tri
        arr = np.stack([p._v for p in pts])
        self.boundary = AABB(tri.dimension, Vector._wrap(arr.min(axis=0)), Vector._wrap(arr.max(axis=0)))
        first = -np.sum([e._v for e in tri.edge_normals], axis=0)
        self.point_data = tuple([TrianglePointDatum(pts[0], Vector._wrap(first))] +
                                [TrianglePointDatum(pts[i + 1], tri.edge_normals[i]) for i in range(tri.dimension - 1)])

    dimension = property(lambda self: self.primitive.dimension)
    face_normal = property(lambda self: self.primitive.face_normal)
    material = property(lambda self: self.primitive.material)


class TriangleBatchPrototype(PrimitivePrototype):
    def __init__(self, t_prototypes):
        if isinstance(t_prototypes, TriangleBatch):
            protos = [TrianglePrototype(t) for t in t_prototypes]
            self.primitive = t_prototypes
        else:
            protos = list(t_prototypes)
            self.primitive = TriangleBatch([p.primitive for p in protos])
        lo = np.min([p.boundary.start._v for p in protos], axis=0)
        hi = np.max([p.boundary.end._v for p in protos], axis=0)
        self.boundary = AABB(protos[0].dimension, Vector._wrap(lo), Vector._wrap(hi))
        self._protos = tuple(protos)

    dimension = property(lambda self: self._protos[0].dimension)
    # per-lane views of the SoA members (TriangleBatchPrototype.face_normal[i] etc., doc/ntracer.rst:1585-1650)
    face_normal = property(lambda self: tuple(p.face_normal for p in self._protos))
    material = property(lambda self: tuple(p.material for p in self._protos))

    @property
    def point_data(self):
        return tuple(TriangleBatchPointDatum(tuple(p.point_data[j].point for p in self._protos),
                                             tuple(p.point_data[j].edge_normal for p in self._protos))
                     for j in range(self.dimension))


class SolidPrototype(PrimitivePrototype):
    """SolidPrototype(type,position,orientation,material) (src/ntracer_body.hpp:2912-2961)"""
    def __init__(self, type, position, orientation, material):
        s = Solid(type, position, orientation, material)
        self.primitive = s
        d = s.dimension
        pos = s.position._v
        if type == CUBE:
            extent = np.abs(s.orientation._m).sum(axis=1)           # sum over cube_component(i) = columns of orientation
            self.boundary = AABB(d, Vector._wrap(pos - extent), Vector._wrap(pos + extent))
        else:
            lo, hi = np.zeros(d, _F), np.zeros(d, _F)
            for i in range(d):
                n = s.orientation._m[i] / np.sqrt(np.dot(s.orientation._m[i], s.orientation._m[i]))
                e = np.zeros(d, _F)
                e[i] = 1
                a, b = float(np.dot(e - pos, n)), float(np.dot(-e - pos, n))
                lo[i], hi[i] = min(a, b), max(a, b)
            self.boundary = AABB(d, Vector._wrap(lo), Vector._wrap(hi))

    dimension = property(lambda self: self.primitive.dimension)
    type = property(lambda self: self.primitive.type)
    position = property(lambda self: self.primitive.position)
    orientation = property(lambda self: self.primitive.orientation)
    inv_orientation = property(lambda self: self.primitive.inv_orientation)
    material = property(lambda self: self.primitive.material)


# ---------------------------------------------------------------------------------------------------------
class RayIntersection:
    """RayIntersection(dist,origin,normal,primitive[,batch_index=-1]) (doc/ntracer.rst:1360-1395)"""
    def __init__(self, dist, origin, normal, primitive, batch_index=-1):
        self.dist, self.origin, self.normal, self.primitive, self.batch_index = dist, origin, normal, primitive, batch_index


class KDNode:
    """Base of KDLeaf / KDBranch.  intersects / occludes run on the GPU (ntr_trace_rays / ntr_occludes_rays)."""
    def __init__(self, *a, **k):
        if type(self) is KDNode:
            raise TypeError('the KDNode type cannot be instantiated directly')

    def __getstate__(self):
        # the device copy (a handle into the CUDA library) is a cache: it never travels with a pickle
        return {k: v for k, v in self.__dict__.items() if k not in ('_dev', '_flat')}

    def _device(self):
        if getattr(self, '_dev', None) is None:
            flat = _Flattener(self.dimension)
            root = flat.walk(self)
            sc = flat.scene_dict(root, AABB(self.dimension), None)
            self._dev, self._flat = DeviceScene(sc), flat
        return self._dev, self._flat

    def _skip(self, flat, source, batch_index):
        if source is None:
            return None, None
        if not isinstance(source, (Primitive, PrimitiveBatch)):
            raise TypeError('object is not an instance of Primitive or PrimitiveBatch')
        ref = flat.item_ref.get(id(source), 0xFFFFFFFF)
        return np.array([ref], np.uint32), np.array([batch_index if isinstance(source, PrimitiveBatch) else -1], np.int32)

    def intersects(self, origin, direction, t_near=-FLT_MAX, t_far=FLT_MAX, source=None, batch_index=-1):
        """-> list of RayIntersection: the surviving transparent hits in the order the traversal's list holds them, then
        the opaque hit (if any) last (src/ntracer_body.hpp:1412-1458)."""
        o, d = _as_vector(origin, self.dimension), _as_vector(direction, self.dimension)
        dev, flat = self._device()
        sr, sl = self._skip(flat, source, batch_index)
        ids, dist, nt, hid, hdist = dev.trace_rays_hits(o._v[None], d._v[None], t_near, t_far, sr, sl)

        def materialise(flat_id, t):
            prim, lane = flat.prim_of_flat_id(int(flat_id))
            tri = prim[lane] if lane >= 0 else prim
            P = o + d * t
            if isinstance(tri, Triangle):
                n = tri.face_normal.unit()
                if dot(tri.face_normal, d) > 0:
                    n = -n
            else:
                frame = tri._hit_frame(o._v, d._v)
                n = None
                if frame is not None:
                    P, n = Vector._wrap(frame[0]), Vector._wrap(frame[1])
            return RayIntersection(t, P, n, prim, lane)

        out = [materialise(hid[0, k], float(hdist[0, k])) for k in range(min(int(nt[0]), hid.shape[1])) if hid[0, k] >= 0]
        if ids[0] >= 0:
            out.append(materialise(ids[0], float(dist[0])))
        return out

    def occludes(self, origin, direction, distance=FLT_MAX, t_near=-FLT_MAX, t_far=FLT_MAX, source=None, batch_index=-1):
        o, d = _as_vector(origin, self.dimension), _as_vector(direction, self.dimension)
        dev, flat = self._device()
        sr, sl = self._skip(flat, source, batch_index)
        occ, nt = dev.occludes_rays(o._v[None], d._v[None], np.array([distance], _F), sr, sl)
        return (bool(occ[0]), None if occ[0] else [])


class KDLeaf(KDNode):
    """KDLeaf(primitives) (doc/ntracer.rst:1026-1053); batches are kept first like kd_leaf (tracer.hpp:1142-1150)"""
    def __init__(self, primitives):
        items = list(primitives)
        if not items:
            raise ValueError('KDLeaf requires at least one item')
        for p in items:
            if not isinstance(p, (Primitive, PrimitiveBatch)):
                raise TypeError('object is not an instance of Primitive or PrimitiveBatch')
        d = items[0].dimension
        if any(p.dimension != d for p in items):
            raise TypeError('every member of KDLeaf must have the same dimension')
        self._items = tuple([p for p in items if isinstance(p, PrimitiveBatch)] + [p for p in items if not isinstance(p, PrimitiveBatch)])
        self._nbatches = sum(isinstance(p, PrimitiveBatch) for p in items)
        self.dimension = d

    def __len__(self): return len(self._items)
    def __getitem__(self, i): return self._items[i]


class KDBranch(KDNode):
    """KDBranch(axis,split[,left=None,right=None]) (doc/ntracer.rst:980-1021)"""
    def __init__(self, axis, split, left=None, right=None):
        for n in (left, right):
            if n is not None and not isinstance(n, KDNode):
                raise TypeError('"left" and "right" must be instances of KDNode')
        if left is None and right is None:
            raise TypeError('"left" and "right" can\'t both be None')
        if left is not None and right is not None and left.dimension != right.dimension:
            raise TypeError('"left" and "right" must have the same dimension')
        self.dimension = (left if left is not None else right).dimension
        if not 0 <= axis < self.dimension:
            raise ValueError('invalid axis')
        self.axis, self.split, self.left, self.right = int(axis), float(_F(split)), left, right


class _Flattener:
    """Walks a KDNode tree into the flat arrays of ntr_scene_desc (the host half of the arena upload)."""
    def __init__(self, dim):
        self.dim = dim
        self.nodes, self.refs, self.simplex, self.simplex_mat, self.solids, self.solid_mat = [], [], [], [], [], []
        self.mats, self.mat_ids, self.item_ref, self.items, self.mat_objs = [], {}, {}, [], []
        self.flat_owner = []            # flat simplex id -> (item, lane)

    def mat_id(self, m):
        k = id(m)
        if k not in self.mat_ids:
            self.mat_ids[k] = len(self.mats)
            self.mats.append(m._row())
            self.mat_objs.append(m)
        return self.mat_ids[k]

    def add_tri(self, t, owner, lane):
        self.simplex.append(t._row())
        self.simplex_mat.append(self.mat_id(t.material))
        self.flat_owner.append((owner, lane))
        return len(self.simplex) - 1

    def ref_of(self, item):
        k = id(item)
        if k in self.item_ref:
            return self.item_ref[k]
        self.items.append(item)
        if isinstance(item, TriangleBatch):
            first = self.add_tri(item[0], item, 0)
            for lane in range(1, BATCH_SIZE):
                self.add_tri(item[lane], item, lane)
            r = (_capi.REF_BATCH << 30) | first
        elif isinstance(item, Triangle):
            r = (_capi.REF_SIMPLEX << 30) | self.add_tri(item, item, -1)
        elif isinstance(item, Solid):
            self.solids.append(item._row())
            self.solid_mat.append(self.mat_id(item.material))
            r = (_capi.REF_SOLID << 30) | (len(self.solids) - 1)
        else:
            raise TypeError('unknown primitive type')
        self.item_ref[k] = r
        return r

    def walk(self, root):
        if root is None:
            return _capi.NULL_NODE
        # iterative pre-order (left subtree first) so deep trees do not hit the recursion limit
        out_root = len(self.nodes)
        stack = [(root, None, 0)]
        while stack:
            node, parent, slot = stack.pop()
            idx = len(self.nodes)
            if parent is not None:
                self.nodes[parent][slot] = idx
            if isinstance(node, KDLeaf):
                first = len(self.refs)
                for it in node._items:
                    self.refs.append(self.ref_of(it))
                self.nodes.append([_capi.LEAF_FLAG | node._nbatches, first, len(node._items), 0])
            else:
                bits = int(np.array([node.split], _F).view(np.uint32)[0])
                self.nodes.append([node.axis, bits, _capi.NULL_NODE, _capi.NULL_NODE])
                if node.right is not None:
                    stack.append((node.right, idx, 3))
                if node.left is not None:
                    stack.append((node.left, idx, 2))
        return out_root

    def prim_of_flat_id(self, fid):
        if fid < len(self.flat_owner):
            return self.flat_owner[fid]
        solids = [it for it in self.items if isinstance(it, Solid)]
        return solids[fid - len(self.flat_owner)], -1

    def material_snapshot(self):
        return np.array([m._row() for m in self.mat_objs], _F).reshape(-1, 10)

    def scene_dict(self, root, boundary, scene):
        d = self.dim
        stride = (d + 1) * d + 1
        sc = {
            'dim': np.int64(d), 'kind': np.int64(1), 'batch_size': np.int64(BATCH_SIZE), 'root': np.int64(root),
            'nodes': np.array(self.nodes, np.uint32).reshape(-1, 4), 'leaf_refs': np.array(self.refs, np.uint32),
            'simplex': np.array(self.simplex, _F).reshape(-1, stride), 'simplex_mat': np.array(self.simplex_mat, np.int32),
            'solids': np.array(self.solids, _F).reshape(-1, 1 + 2 * d * d + d), 'solid_mat': np.array(self.solid_mat, np.int32),
            'materials': self.material_snapshot(),
            'boundary': np.stack([boundary.start._v, boundary.end._v]),
        }
        sc.update(_scene_params(scene, d))
        return sc


def _scene_params(scene, d):
    if scene is None:
        return {'params': np.array([0.8, 0, 1, 4, 1], np.float64), 'ambient': np.zeros(3, _F), 'bg1': np.ones(3, _F),
                'bg2': np.zeros(3, _F), 'bg3': np.array([0, 1, 1], _F), 'point_lights': np.zeros((0, d + 3), _F),
                'global_lights': np.zeros((0, d + 3), _F)}
    return {
        'params': np.array([scene.fov, scene.shadows, scene.camera_light, scene.max_reflect_depth, scene.bg_gradient_axis], np.float64),
        'ambient': np.array(_color_tuple(scene.ambient_color), _F), 'bg1': np.array(_color_tuple(scene.bg1), _F),
        'bg2': np.array(_color_tuple(scene.bg2), _F), 'bg3': np.array(_color_tuple(scene.bg3), _F),
        'point_lights': np.array([list(l.position) + list(_color_tuple(l.color)) for l in scene.point_lights], _F).reshape(-1, d + 3),
        'global_lights': np.array([list(l.direction) + list(_color_tuple(l.color)) for l in scene.global_lights], _F).reshape(-1, d + 3),
    }


# ---------------------------------------------------------------------------------------------------------
class PointLight:
    """PointLight(position,color) (src/tracer.hpp:1678-1689)"""
    def __init__(self, position, color):
        self.position = _as_vector(position)
        self.color = Color(*_color_tuple(color))

    dimension = property(lambda self: self.position.dimension)


class GlobalLight:
    """GlobalLight(direction,color) (src/tracer.hpp:1691-1698)"""
    def __init__(self, direction, color):
        self.direction = _as_vector(direction)
        self.color = Color(*_color_tuple(color))

    dimension = property(lambda self: self.direction.dimension)


def _restore_light_list(scene, kind, items):
    lst = _LightList(scene, kind)
    list.extend(lst, items)                 # already validated when they were added
    return lst


class _LightList(list):
    def __init__(self, scene, kind):
        super().__init__()
        self._scene, self._kind = scene, kind

    def __reduce__(self):
        return _restore_light_list, (self._scene, self._kind, list(self))

    def _check(self, light):
        if not isinstance(light, self._kind):
            raise TypeError('object is not an instance of %s' % self._kind.__name__)
        if light.dimension != self._scene.dimension:
            raise TypeError('the light must have the same dimension as the scene')
        self._scene._check_unlocked()

    def append(self, light):
        self._check(light)
        super().append(light)

    def extend(self, lights):
        for l in lights:
            self.append(l)

    def __setitem__(self, i, light):
        self._check(light)
        super().__setitem__(i, light)


class _SceneBase(Scene):
    supersampling = 1           # class-level default: scenes pickled before the attribute existed load with it
    supersampling_threshold = None      # likewise: off, and a scene that never sets it pickles as before
    projection = ('perspective', None)  # likewise: the reference's pinhole camera

    def __init__(self, dimension):
        self.locked = 0
        self.fov = 0.8
        self._cam = Camera(dimension)
        self._dev = None

    dimension = property(lambda self: self._cam.dimension)

    def __getstate__(self):
        # device copy and lock count belong to this process (pickle codecs of the reference: src/render.cpp:1391-1657)
        st = {k: v for k, v in self.__dict__.items() if k not in ('_dev', '_flat', '_mat_snapshot', '_group', '_group_of', '_sc')}
        st['_dev'] = None
        st['locked'] = 0
        return st

    def _check_unlocked(self):
        if self.locked:
            raise LockedError('the scene is locked for reading')

    def set_camera(self, camera):
        self._check_unlocked()
        if not isinstance(camera, Camera) or camera.dimension != self.dimension:
            raise TypeError('the scene and camera must have the same dimension')
        self._cam = camera._copy()

    def get_camera(self): return self._cam._copy()

    def set_fov(self, fov):
        self._check_unlocked()
        self.fov = float(fov)

    def set_supersampling(self, factor, threshold=None):
        """Anti-aliasing (no counterpart in the reference, which traces one ray through the corner of every pixel): every
        pixel of a frame becomes the mean of factor x factor samples on an ordered grid over the pixel, i.e. the box-filtered
        factor-times-larger frame.  factor is an integer from 1 to 8; 1 (the default) is one ray per pixel.  Every renderer
        and calculate_color honour it.  A frame costs about factor ** 2 times the rays, and the device memory that holds the
        reflection rays of a frame grows with factor ** 2 as well.

        threshold (a real number >= 0, or None for off) makes it adaptive: the frame is traced at one ray per pixel, and
        only the pixels whose four corner colours (the pixel and its right, lower and lower-right neighbours) differ by
        more than threshold in some channel (colours in 0..1) get the factor x factor samples; the others keep their plain
        colour.  4/255 is a good default (README, "Adaptive anti-aliasing")."""
        self._check_unlocked()
        if isinstance(factor, bool) or not isinstance(factor, numbers.Integral):
            raise TypeError('the supersampling factor must be an integer')
        if not 1 <= factor <= _capi.NTR_MAX_SUPERSAMPLING:
            raise ValueError('the supersampling factor must be between 1 and %d' % _capi.NTR_MAX_SUPERSAMPLING)
        if threshold is not None:
            if isinstance(threshold, bool) or not isinstance(threshold, numbers.Real):
                raise TypeError('the supersampling threshold must be a real number or None')
            if not (math.isfinite(threshold) and threshold >= 0):
                raise ValueError('the supersampling threshold must be a finite number >= 0, or None for off')
        self.supersampling = int(factor)
        if threshold is None:
            self.__dict__.pop('supersampling_threshold', None)
        else:
            self.supersampling_threshold = float(threshold)

    def set_projection(self, kind, param=None):
        """The camera's projection (no counterpart in the reference, whose camera is a pinhole through fov): 'perspective'
        (the default; param is ignored), 'orthographic' (param: half the view's width in scene units, required; fov is
        ignored and the rays start on the image plane through the camera origin, so the camera must stand outside what it
        should see) or 'equirectangular' (param: the horizontal field angle in radians, in (0, 2 pi], default 2 pi; fov is
        ignored; a W x W/2 frame at 2 pi shows the whole sphere around the camera).  Every renderer and calculate_color
        honour it, supersampling included.  scene.projection reads it back as (kind, param)."""
        self._check_unlocked()
        kind, param = projection_args(kind, param)
        if kind == 'perspective':
            self.__dict__.pop('projection', None)
        else:
            self.projection = (kind, param)

    # ---- backend ----
    def _device_scene(self):
        raise NotImplementedError

    def _prepare(self, gpus=1):
        """-> the device copy of the scene, camera set: a DeviceScene, or a DeviceGroup over `gpus` devices (the frame split
        by interleaved tile rows, BlockingRenderer(threads=N))."""
        dev = self._device_scene()
        if gpus > 1:
            grp = getattr(self, '_group', None)
            if grp is None or grp.size != gpus or self._group_of is not dev:
                if grp is not None:
                    grp.close()
                grp = self._group = DeviceGroup(self._scene_dict(), gpus)
                self._group_of = dev            # rebuilt whenever the single-device copy is (materials changed)
            else:
                grp.set_params(self._scene_dict())
            dev = grp
        dev.set_camera(self._cam._origin, self._cam._axes)
        if getattr(dev, 'supersampling', 1) != self.supersampling:
            dev.set_supersampling(self.supersampling)
        if getattr(dev, 'supersampling_threshold', None) != self.supersampling_threshold:
            dev.set_supersampling_threshold(self.supersampling_threshold)
        if getattr(dev, 'projection', ('perspective', None)) != self.projection:
            dev.set_projection(*self.projection)
        return dev

    def calculate_color(self, x, y, width, height):
        """Scene.calculate_color (src/render.cpp:586-614)"""
        self.locked += 1
        try:
            return Color(*[float(v) for v in self._prepare().calculate_color(x, y, width, height)])
        finally:
            self.locked -= 1


class BoxScene(_SceneBase):
    """BoxScene(dimension) (src/tracer.hpp:83-123, doc/ntracer.rst:547-591)"""
    def __init__(self, dimension):
        _check_dimension(dimension)
        super().__init__(dimension)

    def _flat(self):
        return {'dim': np.int64(self.dimension), 'kind': np.int64(0), 'batch_size': np.int64(1),
                'params': np.array([self.fov, 0, 0, 0, 0], np.float64)}

    def _scene_dict(self):
        return self._flat()

    def _device_scene(self):
        if self._dev is None:
            self._dev = DeviceScene(self._flat())
            self._dev_fov = self.fov
        elif self._dev_fov != self.fov:
            self._dev.set_params(self._flat())
            self._dev_fov = self.fov
        return self._dev


class CompositeScene(_SceneBase):
    """CompositeScene(boundary,data) (src/tracer.hpp:1710-1927, doc/ntracer.rst:671-892)"""
    def __init__(self, boundary, data):
        if not isinstance(boundary, AABB):
            raise TypeError('object is not an instance of AABB')
        if not isinstance(data, KDNode):
            raise TypeError('object is not an instance of KDNode')
        if boundary.dimension != data.dimension:
            raise TypeError('"boundary" and "data" must have the same dimesion')
        super().__init__(boundary.dimension)
        self.boundary, self.root = boundary, data
        self.shadows, self.camera_light, self.max_reflect_depth, self.bg_gradient_axis = False, True, 4, 1
        self.ambient_color, self.bg1, self.bg2, self.bg3 = Color(0, 0, 0), Color(1, 1, 1), Color(0, 0, 0), Color(0, 1, 1)
        self.point_lights = _LightList(self, PointLight)
        self.global_lights = _LightList(self, GlobalLight)
        self._flat = None

    def set_shadows(self, shadows):
        self._check_unlocked(); self.shadows = bool(shadows)

    def set_camera_light(self, camera_light):
        self._check_unlocked(); self.camera_light = bool(camera_light)

    def set_ambient_color(self, color):
        self._check_unlocked(); self.ambient_color = Color(*_color_tuple(color))

    def set_max_reflect_depth(self, depth):
        self._check_unlocked()
        if depth < 0:
            raise ValueError('depth cannot be negative')
        self.max_reflect_depth = int(depth)

    def set_background(self, c1, c2=None, c3=None, axis=1):
        self._check_unlocked()
        if not 0 <= axis < self.dimension:
            raise ValueError('"axis" must be between 0 and one less than the dimension of the scene')
        c2 = c1 if c2 is None else c2
        c3 = c1 if c3 is None else c3
        self.bg1, self.bg2, self.bg3, self.bg_gradient_axis = Color(*_color_tuple(c1)), Color(*_color_tuple(c2)), Color(*_color_tuple(c3)), int(axis)

    def add_light(self, light):
        if isinstance(light, PointLight):
            self.point_lights.append(light)
        elif isinstance(light, GlobalLight):
            self.global_lights.append(light)
        else:
            raise TypeError('object is not an instance of PointLight or GlobalLight')

    def _device_scene(self):
        # geometry is immutable once the scene exists; Material objects are not (the reference reads them through
        # pointers), so the arena is rebuilt if any referenced material changed since the upload
        if self._dev is not None and not np.array_equal(self._flat.material_snapshot(), self._mat_snapshot):
            self._dev.close()
            self._dev = None
        if self._dev is None:
            flat = _Flattener(self.dimension)
            root = flat.walk(self.root)
            self._flat = flat
            self._mat_snapshot = flat.material_snapshot()
            self._sc = flat.scene_dict(root, self.boundary, self)
            self._dev = DeviceScene(self._sc)
        else:
            sc = {'dim': np.int64(self.dimension), 'kind': np.int64(1), 'batch_size': np.int64(BATCH_SIZE), 'root': np.int64(0),
                  'boundary': np.stack([self.boundary.start._v, self.boundary.end._v])}
            sc.update(_scene_params(self, self.dimension))
            self._dev.set_params(sc)
            self._sc.update(_scene_params(self, self.dimension))
        return self._dev

    def _scene_dict(self):
        return self._sc


# ---------------------------------------------------------------------------------------------------------
def screen_coord_to_ray(cam, x, y, w, h, fov):
    """src/ntracer_body.hpp:3342-3358 / flat_origin_ray_source (src/tracer.hpp:60-76)"""
    half_w, half_h = _F(w) / _F(2), _F(h) / _F(2)
    fovI = _F(math.tan(_F(fov) / 2)) / half_w
    v = cam._axes[2] + cam._axes[0] * (fovI * (_F(x) - half_w)) - cam._axes[1] * (fovI * (_F(y) - half_h))
    return Vector._wrap(v / np.sqrt(_F(np.dot(v, v))))


def build_kdtree(primitives, extra_threads=-1, *, max_depth=None, split_threshold=None, traversal_cost=None,
                 intersection_cost=None, update_primitives=False):
    """-> (AABB, KDNode).  The tree comes from this backend's native host-side builder (csrc/builder.cpp,
    ntr_group_items + ntr_build_kdtree_culled: triangles grouped into TriangleBatch items, then a binned SAH over the
    items' bounding boxes whose candidate planes are re-evaluated with the cells' real contents).  It is NOT the reference's builder (src/tracer.hpp:1930-2455): colours and hit ids do not depend on
    the tree, except with shadows on (DESIGN.md section 2)."""
    from . import bulk
    protos = list(primitives)
    if not protos:
        raise ValueError('cannot build tree from empty sequence')
    for p in protos:
        if not isinstance(p, PrimitivePrototype):
            raise TypeError('object is not an instance of PrimitivePrototype')
    d = protos[0].dimension
    if any(p.dimension != d for p in protos):
        raise TypeError('the primitive prototypes must all have the same dimension')
    lo = np.stack([p.boundary.start._v for p in protos])
    hi = np.stack([p.boundary.end._v for p in protos])
    # group_primitives (src/tracer.hpp:2395-2427): triangles are packed into TriangleBatch items of BATCH_SIZE lanes before
    # the tree is built over the ITEMS; solids and the left-over triangles stay single primitives.  The grouping is this
    # backend's own (ntr_group_items: recursive median split of the centres, O(n log n) against the reference's O(n^2)).
    prims = [p.primitive for p in protos]
    tri = [i for i, q in enumerate(prims) if isinstance(q, Triangle)]
    items, ilo, ihi = [], [], []
    owned = []          # per item: the prototypes of its simplexes (none for a solid)
    if BATCH_SIZE > 1 and len(tri) >= BATCH_SIZE:
        order = bulk.group_items(lo[tri], hi[tri], BATCH_SIZE)
        nb = len(tri) // BATCH_SIZE
        for k in range(nb):
            members = [tri[int(j)] for j in order[k * BATCH_SIZE:(k + 1) * BATCH_SIZE]]
            items.append(TriangleBatch([prims[j] for j in members]))
            ilo.append(lo[members].min(axis=0))
            ihi.append(hi[members].max(axis=0))
            owned.append(members)
        single = [tri[int(j)] for j in order[nb * BATCH_SIZE:]] + [i for i, q in enumerate(prims) if not isinstance(q, Triangle)]
    else:
        single = list(range(len(prims)))
    for j in single:
        items.append(prims[j])
        ilo.append(lo[j])
        ihi.append(hi[j])
        owned.append([j] if isinstance(prims[j], Triangle) else [])
    # The simplexes behind the items go to the builder too, so that -- like the reference's builder with its exact
    # overlap tests (src/tracer.hpp:1465-1675) -- an item is listed only in the cells its geometry can touch
    # (ntr_build_kdtree_culled; a rebuilt {5,3,3} scene then costs the reference algorithm the same number of simplex
    # tests per frame as on the reference's own tree, against 2.2 x with bounding boxes alone).
    flat = [j for m in owned for j in m]
    first = np.cumsum([0] + [len(m) for m in owned]).astype(np.uint32)
    recs = np.zeros((len(flat), (d + 1) * d + 1), np.float32)
    for k, j in enumerate(flat):
        recs[k] = prims[j]._row()
    cull = (first, lo[flat].reshape(-1, d), hi[flat].reshape(-1, d), recs) if flat else None
    nodes, refs, root, boundary = bulk.build_kdtree(np.stack(ilo), np.stack(ihi), max_depth or 0, split_threshold or 0,
                                                    -1.0 if traversal_cost is None else traversal_cost,
                                                    -1.0 if intersection_cost is None else intersection_cost, cull=cull)
    # children always follow their parent in the node array, so a reverse sweep builds the objects bottom-up
    objs = [None] * len(nodes)
    for i in range(len(nodes) - 1, -1, -1):
        meta, a, b, c = (int(x) for x in nodes[i])
        if meta & _capi.LEAF_FLAG:
            members = [items[j] for j in refs[a:a + b]]
            # batches first, like the reference's leaves (tracer.hpp:1142-1150)
            objs[i] = KDLeaf([m for m in members if isinstance(m, TriangleBatch)] + [m for m in members if not isinstance(m, TriangleBatch)])
        else:
            split = float(np.array([a], np.uint32).view(np.float32)[0])
            objs[i] = KDBranch(meta, split, None if b == _capi.NULL_NODE else objs[b], None if c == _capi.NULL_NODE else objs[c])
    if root == _capi.NULL_NODE:
        raise ValueError('cannot build tree from empty sequence')
    return AABB(d, Vector._wrap(boundary[0]), Vector._wrap(boundary[1])), objs[root]


def build_composite_scene(primitives, extra_threads=-1, **kw):
    boundary, root = build_kdtree(primitives, extra_threads, **kw)
    return CompositeScene(boundary, root)
