"""Host-side mirror of SPOMSO's object / functional API for the SDF hot path.

Same class names, method names, argument meaning and error behaviour as the reference front end, but instead
of wrapping NumPy closures (Code/spomso/spomso/cores/modifications.py:88-98) every object records an explicit
tree: node = Euclidean state + ordered modification list + (leaf primitive | combine children | nested node).
`create(co)` flattens the tree (program.py) and runs it on the B200 (engine.py). There is no NumPy evaluation
path in this package; the CPU restatement lives in oracle/ and is test infrastructure only.

Reference interfaces mirrored here:
  EuclideanTransform           Code/spomso/spomso/cores/transformations.py:12-264
  ModifyObject                 Code/spomso/spomso/cores/modifications.py:30-1663 (hot-path subset, SURVEY §8a)
  GenericGeometry              Code/spomso/spomso/cores/geom.py:15-74
  CombineGeometry              Code/spomso/spomso/cores/combine.py:37-163
  primitives                   Code/spomso/spomso/cores/geom_3d.py, geom_2d.py
"""
from __future__ import annotations

import numpy as np

# ----------------------------------------------------------------------------------------------------------------
# leaf descriptors (stand-ins for the module-level sdf_* functions of sdf_3D.py / sdf_2D.py)


class LeafSDF:
    """Stands for one of SPOMSO's `sdf_*` functions. Calling it evaluates on the GPU (functional API)."""

    def __init__(self, name: str):
        self.name = name
        self.__name__ = name

    def __call__(self, co, *params):
        return GenericGeometry(self, *params).create(co)

    def __repr__(self):
        return f"<aegolius_b200 leaf {self.name}>"


_LEAF_NAMES = [
    "sdf_x", "sdf_y", "sdf_z", "sdf_sphere", "sdf_cylinder", "sdf_box", "sdf_torus", "sdf_chainlink", "sdf_braid",
    "sdf_arc_3d", "sdf_plane", "sudf_plane", "sdf_segment_3d", "sdf_cone", "sdf_oriented_infinite_cone",
    "sdf_infinite_cone", "sdf_solid_angle", "sdf_triangle_3d", "sdf_quad_3d", "sdf_segmented_line_3d",
    "sdf_point_cloud_3d", "sdf_circle", "sdf_neu_circle", "sdf_box_2d", "sdf_segment_2d", "sdf_rounded_box_2d",
    "sdf_triangle_2d", "sdf_arc", "sdf_sector", "sdf_inf_sector", "sdf_ngon", "sdf_segmented_line_2d",
    "sdf_point_cloud_2d", "sdf_closed_segmented_line_2d", "sdf_closed_segmented_line_3d", "sdf_polygon_2d",
    "sdf_parametric_curve_2d", "sdf_parametric_curve_3d", "sdf_closed_parametric_curve_2d",
    "sdf_closed_parametric_curve_3d", "sdf_segmented_curve_2d", "sdf_segmented_curve_3d",
    "sdf_closed_segmented_curve_2d", "sdf_closed_segmented_curve_3d",
]
LEAVES = {n: LeafSDF(n) for n in _LEAF_NAMES}
globals().update(LEAVES)


def rotation_matrix_from_rotvec(rotvec) -> np.ndarray:
    """Rodrigues formula; equals scipy's Rotation.from_rotvec(v).as_matrix() (transformations.py:160)."""
    v = np.asarray(rotvec, dtype=np.float64)
    theta = float(np.linalg.norm(v))
    if theta == 0.0:
        return np.eye(3)
    k = v / theta
    K = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
    return np.eye(3) + np.sin(theta) * K + (1.0 - np.cos(theta)) * (K @ K)


def _rotvec_matrix(rotvec):
    """The reference calls scipy's Rotation.from_rotvec (transformations.py:160); use the same routine when scipy is
    importable so that rotation matrices are bit-identical to SPOMSO's, else the Rodrigues form (<= 2e-16 apart)."""
    try:
        from scipy.spatial.transform import Rotation
        return Rotation.from_rotvec(np.asarray(rotvec, dtype=np.float64)).as_matrix()
    except ImportError:  # pragma: no cover
        return rotation_matrix_from_rotvec(rotvec)


# ----------------------------------------------------------------------------------------------------------------
# Euclidean state (transformations.py:12-264)


class EuclideanTransform:
    def __init__(self):
        self._et = []
        self._center = np.asarray((0.0, 0.0, 0.0))
        self._scale = 1.0
        self._rot_matrix = np.eye(3)

    @property
    def transformations(self):
        return self._et

    @property
    def center(self):
        return self._center

    @property
    def scale(self):
        return self._scale

    @property
    def rotation_matrix(self):
        return self._rot_matrix

    def set_location(self, center):
        self._et.append("set_location")
        center = np.asarray(center)
        if center.size <= 3:
            self._center[:center.size] = center
        else:
            raise SyntaxError(f"Array {center} is of incorrect size!")

    def move(self, move_vector):
        self._et.append("move")
        vector = np.asarray(move_vector)
        if vector.size <= 3:
            self._center += vector  # same broadcasting rules (and failures) as transformations.py:104
        else:
            raise SyntaxError(f"Array {vector} is of incorrect size!")

    def set_scale(self, scale):
        self._et.append("set_scale")
        if isinstance(scale, (float, int)):
            self._scale = scale
        else:
            raise TypeError("Scale must be a float or an int")

    def rescale(self, scale):
        self._et.append("rescale")
        if isinstance(scale, (float, int)):
            self._scale *= scale
        else:
            raise TypeError("Scale must be a float or an int")

    @staticmethod
    def get_rotation_matrix(angle, axis):
        axis = np.asarray(axis)
        if axis.size <= 3:
            axis_ = np.zeros(3)
            axis_[:axis.size] = axis
        else:
            raise SyntaxError(f"Array {axis} is of incorrect size!")
        if not isinstance(angle, (float, int)):
            raise TypeError("Rotation angle must be a float or an int")
        return _rotvec_matrix(angle * axis_), angle, axis_

    def set_rotation(self, angle, axis):
        # NB: like transformations.py:163-173 the axis is NOT normalised here
        self._et.append("set_rotation")
        self._rot_matrix, _, _ = self.get_rotation_matrix(angle, axis)

    def rotate_rotvec(self, angle, axis):
        axis = np.asarray(axis)
        if np.array_equal(axis, np.zeros(3)[:axis.size]):
            raise ValueError("Axis cannot be zero!")
        axis = axis / np.linalg.norm(axis)
        rot_matrix, _, _ = self.get_rotation_matrix(angle, axis)
        self.rotate_matrix(rot_matrix)

    def rotate_matrix(self, rotation_matrix):
        # accumulates by LEFT multiplication (transformations.py:200)
        self._rot_matrix = np.matmul(rotation_matrix, self._rot_matrix)

    def rotate(self, *inputs):
        self._et.append("rotate")
        if len(inputs) == 1:
            # the reference wraps the matrix as (1,3,3) (transformations.py:221-223), which later fails in
            # create(); here a plain 3x3 is accepted and a wrapped one rejected up front.
            m = np.asarray(inputs[0], dtype=np.float64)
            if m.shape != (3, 3):
                raise ValueError(f"rotation matrix must have shape (3, 3), got {m.shape}")
            self.rotate_matrix(m)
        elif len(inputs) == 2:
            angle, axis = inputs
            self.rotate_rotvec(angle, np.asarray(axis))
        else:
            raise SyntaxError("Wrong number of inputs!")


# ----------------------------------------------------------------------------------------------------------------
# modifications (modifications.py): recorded, not executed


class ModifyObject:
    def __init__(self):
        self._mod = []
        self._mods = []  # [(name, params dict)] in call order

    @property
    def modifications(self):
        return self._mod

    def _add(self, name, **params):
        self._mod.append(name)
        self._mods.append((name, params))
        return self

    # coordinate warps ---------------------------------------------------------------------------------------
    def elongation(self, elongate_vector):
        return self._add("elongation", ev=np.asarray(elongate_vector, dtype=np.float64))

    def twist(self, pitch):
        return self._add("twist", pitch=pitch)

    def bend(self, radius, angle):
        return self._add("bend", radius=radius, angle=angle)

    def shear_xz(self, angle):
        return self._add("shear_xz", angle=angle)

    def shear_yz(self, angle):
        return self._add("shear_yz", angle=angle)

    def shear_xy(self, angle):
        return self._add("shear_xy", angle=angle)

    def shear_zy(self, angle):
        return self._add("shear_zy", angle=angle)

    def shear_yx(self, angle):
        return self._add("shear_yx", angle=angle)

    def shear_zx(self, angle):
        return self._add("shear_zx", angle=angle)

    def shear(self, angle, sheared_axis, fixed_axis):
        return self._add("shear", angle=angle, sheared_axis=sheared_axis, fixed_axis=fixed_axis)

    def infinite_repetition(self, distances):
        return self._add("infinite_repetition", distances=distances)

    def finite_repetition(self, size, repetitions):
        return self._add("finite_repetition", size=np.asarray(size), rep=np.asarray(repetitions))

    def finite_repetition_rescaled(self, size, repetitions, instance_size, padding):
        return self._add("finite_repetition_rescaled", size=np.asarray(size), rep=np.asarray(repetitions),
                         f=np.asarray(instance_size), padding=np.asarray(padding))

    def symmetry(self, axis):
        return self._add("symmetry", axis=axis)

    def mirror(self, a, b):
        return self._add("mirror", a=np.asarray(a), b=np.asarray(b))

    def rotational_symmetry(self, n, radius, phase):
        return self._add("rotational_symmetry", angle=2 * np.pi / n, radius=radius, phase=phase)

    def linear_instancing(self, n, a, b):
        return self._add("linear_instancing", n=n, a=np.asarray(a), b=np.asarray(b))

    def curve_instancing(self, f, f_parameters, t_range):
        return self._add("curve_instancing", f=f, f_parameters=f_parameters, t_range=t_range)

    def aligned_curve_instancing(self, f, f_parameters, t_range):
        return self._add("aligned_curve_instancing", f=f, f_parameters=f_parameters, t_range=t_range, tol=0.001)

    def fully_aligned_curve_instancing(self, f, f_parameters, t_range):
        return self._add("fully_aligned_curve_instancing", f=f, f_parameters=f_parameters, t_range=t_range,
                         tol=0.001)

    def revolution(self, radius):
        return self._add("revolution", radius=radius)

    def axis_revolution(self, radius, angle):
        return self._add("axis_revolution", radius=radius, angle=angle)

    def move_sdf(self, move_vector):
        return self._add("move_sdf", move_vector=move_vector)

    def scale_sdf(self, scale_factor):
        return self._add("scale_sdf", scale_factor=scale_factor)

    def rotate_sdf(self, rotation_matrix):
        return self._add("rotate_sdf", rotation_matrix=rotation_matrix)

    # value / mixed -----------------------------------------------------------------------------------------
    def rounding(self, rounding_radius):
        return self._add("rounding", rounding_radius=rounding_radius)

    def rounding_cs(self, rounding_radius, bb_size):
        return self._add("rounding_cs", rounding_radius=rounding_radius, bb_size=bb_size)

    def boundary(self):
        return self._add("boundary")

    def invert(self, direct=False):
        if direct:  # modifications.py:297-299: the closure is returned but not installed
            self._mod.append("invert")
            return self
        return self._add("invert")

    def sign(self, direct=False):
        if direct:
            self._mod.append("sign")
            return self
        return self._add("sign")

    def onion(self, thickness):
        return self._add("onion", thickness=thickness)

    def concentric(self, width):
        return self._add("concentric", width=width)

    def extrusion(self, distance):
        return self._add("extrusion", distance=distance)

    # post-processing value maps (modifications.py:1361-1587) -----------------------------------------------------
    def sigmoid_falloff(self, amplitude, width):
        return self._add("sigmoid_falloff", amplitude=amplitude, width=width)

    def positive_sigmoid_falloff(self, amplitude, width):
        return self._add("positive_sigmoid_falloff", amplitude=amplitude, width=width)

    def capped_exponential(self, amplitude, width):
        return self._add("capped_exponential", amplitude=amplitude, width=width)

    def hard_binarization(self, threshold):
        return self._add("hard_binarization", threshold=threshold)

    def linear_falloff(self, amplitude, width):
        return self._add("linear_falloff", amplitude=amplitude, width=width)

    def relu(self, width=1):
        return self._add("relu", width=width)

    def smooth_relu(self, smooth_width, width=1, threshold=0.01):
        return self._add("smooth_relu", smooth_width=smooth_width, width=width, threshold=threshold)

    def slowstart(self, smooth_width, width=1, threshold=0.01, ground=True):
        return self._add("slowstart", smooth_width=smooth_width, width=width, threshold=threshold, ground=ground)

    def gaussian_boundary(self, amplitude, width):
        return self._add("gaussian_boundary", amplitude=amplitude, width=width)

    def gaussian_falloff(self, amplitude, width):
        return self._add("gaussian_falloff", amplitude=amplitude, width=width)

    # not representable in an op list (user Python callables / grid stencils) -----------------------------------
    def _unsupported(self, name):
        raise NotImplementedError(
            f"'{name}' takes a Python callable or a grid stencil and cannot enter the GPU op list "
            f"(SURVEY §8a exclusions); evaluate this object with SPOMSO itself.")

    def custom_modification(self, *a, **k):
        self._unsupported("custom_modification")

    def custom_post_process(self, *a, **k):
        self._unsupported("custom_post_process")

    def displacement(self, *a, **k):
        self._unsupported("displacement")

    def define_volume(self, *a, **k):
        self._unsupported("define_volume")

    def recover_volume(self, *a, **k):
        self._unsupported("recover_volume")

    def signed(self, co_resolution):
        """modifications.py:220-275: unsigned -> signed distance field on a 3D grid (a whole-grid post-pass, like the
        convolution modifications: flattened into a stencil stage, engine._staged_torch)."""
        return self._add("signed", co_resolution=co_resolution)

    # grid stencils (modifications.py:1586-1637): evaluated by separate kernels between two interpreter launches
    def conv_averaging(self, kernel_size, iterations, co_resolution):
        return self._add("conv_averaging", kernel_size=kernel_size, iterations=iterations, co_resolution=co_resolution)

    def conv_edge_detection(self, co_resolution):
        return self._add("conv_edge_detection", co_resolution=co_resolution)


# ----------------------------------------------------------------------------------------------------------------
# nodes


class GenericGeometry(EuclideanTransform, ModifyObject):
    """Node of the geometry tree (geom.py:15-60). `geo_sdf` is a LeafSDF, the bound `propagate` of another
    node (nesting, Code/examples/scalar/3D/basics_3D.py:111) or an internal combine descriptor."""

    def __init__(self, geo_sdf, *geo_parameters):
        EuclideanTransform.__init__(self)
        ModifyObject.__init__(self)
        self._geo_parameters = geo_parameters
        self.kind = None
        self.leaf = None
        self.inner = None
        self.combine_op = None
        self.children = None
        self.combine_parameter = None
        if isinstance(geo_sdf, LeafSDF):
            self.kind, self.leaf = "leaf", geo_sdf.name
        elif isinstance(geo_sdf, _CombineDescriptor):
            self.kind = "combine"
            self.combine_op = geo_sdf.op
            self.children = geo_sdf.children  # tuple of nodes, late-bound like combine.py:129-135
            self.combine_parameter = geo_sdf.parameter
        elif getattr(geo_sdf, "__func__", None) is GenericGeometry.propagate or (
                hasattr(geo_sdf, "__self__") and isinstance(geo_sdf.__self__, GenericGeometry)
                and getattr(geo_sdf, "__name__", "") in ("propagate", "create")):
            self.kind, self.inner = "nested", geo_sdf.__self__
        else:
            raise NotImplementedError(
                f"SDF callable {geo_sdf!r} is not a known primitive; arbitrary Python SDFs cannot enter the GPU "
                f"op list (SURVEY §8a exclusions).")

    def create(self, co, **kwargs):
        """Signed distance field of shape (N,) on `co` ((D,N) array or a GridSpec)  — geom.py:29-43."""
        from . import engine
        return engine.create(self, co, **kwargs)

    def propagate(self, co, *parameters_, **kwargs):
        """geom.py:45-60 — same evaluation as create; its bound method marks nesting."""
        from . import engine
        return engine.create(self, co, **kwargs)


class _CombineDescriptor:
    def __init__(self, op, children, parameter):
        self.op, self.children, self.parameter = op, children, parameter


class CombineGeometry:
    """combine.py:37-163."""

    OPERATIONS = ("UNION2", "UNION", "SUBTRACT2", "INTERSECT2", "INTERSECT", "SUM", "DIFFERENCE")
    PARAMETRIC_OPERATIONS = ("SMOOTH_UNION2_2", "SMOOTH_UNION2", "SMOOTH_INTERSECT2",
                             "SMOOTH_INTERSECT2_BOLTZMANN", "SMOOTH_SUBTRACT2", "SMOOTH_SUBTRACT2_BOLTZMANN")

    def __init__(self, operation_type: str):
        self.operation_type = operation_type
        self._combined_geometry = None

    @property
    def available_operations(self):
        print(f"Available non-parametric operations are: {list(self.OPERATIONS)}")
        return list(self.OPERATIONS)

    @property
    def available_parametric_operations(self):
        print(f"Available parametric operations are: {list(self.PARAMETRIC_OPERATIONS)}")
        return list(self.PARAMETRIC_OPERATIONS)

    @property
    def combined_geometry(self):
        return self._combined_geometry

    def combine(self, *combined_objects):
        if self.operation_type not in self.OPERATIONS:
            # the reference builds SyntaxError(msg, str) (combine.py:125-127), which CPython >= 3.10 turns into a
            # TypeError about the malformed details tuple; the intended SyntaxError is raised here
            raise SyntaxError(f"{self.operation_type} is not an implemented non-parametric operation. "
                              f"Possible operations are {self.OPERATIONS}")
        self._combined_geometry = _CombineDescriptor(self.operation_type, combined_objects, None)
        return GenericGeometry(self._combined_geometry, ())

    def combine_parametric(self, *combined_objects, parameters):
        if self.operation_type not in self.PARAMETRIC_OPERATIONS:
            raise SyntaxError(f"{self.operation_type} is not an implemented parametric operation. "
                              f"Possible parametric operations are {self.PARAMETRIC_OPERATIONS}")
        self._combined_geometry = _CombineDescriptor(self.operation_type, combined_objects, parameters)
        return GenericGeometry(self._combined_geometry, ())


# ----------------------------------------------------------------------------------------------------------------
# 3D primitives (geom_3d.py)


def _leaf(name):
    return LEAVES[name]


class X(GenericGeometry):
    def __init__(self, offset):
        GenericGeometry.__init__(self, _leaf("sdf_x"), offset)


class Y(GenericGeometry):
    def __init__(self, offset):
        GenericGeometry.__init__(self, _leaf("sdf_y"), offset)


class Z(GenericGeometry):
    def __init__(self, offset):
        GenericGeometry.__init__(self, _leaf("sdf_z"), offset)


class InfiniteCylinder(GenericGeometry):
    def __init__(self, radius):  # geom_3d.py:102 binds the 2D circle
        GenericGeometry.__init__(self, _leaf("sdf_circle"), radius)


class Cylinder(GenericGeometry):
    def __init__(self, radius, height):
        GenericGeometry.__init__(self, _leaf("sdf_cylinder"), radius, height)


class Sphere(GenericGeometry):
    def __init__(self, radius):
        GenericGeometry.__init__(self, _leaf("sdf_sphere"), radius)


class Box(GenericGeometry):
    def __init__(self, a, b, c):
        GenericGeometry.__init__(self, _leaf("sdf_box"), (a, b, c))


class Plane(GenericGeometry):
    def __init__(self, normal, thickness):  # geom_3d.py:196: unsigned slab
        GenericGeometry.__init__(self, _leaf("sudf_plane"), np.asarray(normal), thickness)


class OrientedPlane(GenericGeometry):
    def __init__(self, normal, offset):
        GenericGeometry.__init__(self, _leaf("sdf_plane"), np.asarray(normal), offset)


class Line(GenericGeometry):
    def __init__(self, a, b):
        GenericGeometry.__init__(self, _leaf("sdf_segment_3d"), a, b)


class Triangle3D(GenericGeometry):
    def __init__(self, a, b, c):
        GenericGeometry.__init__(self, _leaf("sdf_triangle_3d"), np.asarray(a), np.asarray(b), np.asarray(c))


class Quad(GenericGeometry):
    def __init__(self, a, b, c, d):
        GenericGeometry.__init__(self, _leaf("sdf_quad_3d"), np.asarray(a), np.asarray(b), np.asarray(c),
                                 np.asarray(d))


class Torus(GenericGeometry):
    def __init__(self, primary_radius, secondary_radius):
        GenericGeometry.__init__(self, _leaf("sdf_torus"), primary_radius, secondary_radius)


class ChainLink(GenericGeometry):
    def __init__(self, primary_radius, secondary_radius, length):  # geom_3d.py:368 halves the length
        GenericGeometry.__init__(self, _leaf("sdf_chainlink"), primary_radius, secondary_radius, length / 2)


class Braid(GenericGeometry):
    def __init__(self, length, primary_radius, secondary_radius, pitch):  # geom_3d.py:403
        GenericGeometry.__init__(self, _leaf("sdf_braid"), length / 2, primary_radius, secondary_radius, pitch)


class Arc3D(GenericGeometry):
    def __init__(self, radius, thickness, start_angle, end_angle):
        GenericGeometry.__init__(self, _leaf("sdf_arc_3d"), radius, thickness, start_angle, end_angle)


class Cone(GenericGeometry):
    def __init__(self, height, angle):
        GenericGeometry.__init__(self, _leaf("sdf_cone"), height, angle)


class InfiniteCone(GenericGeometry):
    def __init__(self, angle):
        GenericGeometry.__init__(self, _leaf("sdf_infinite_cone"), angle)


class OrientedInfiniteCone(GenericGeometry):
    def __init__(self, angle):
        GenericGeometry.__init__(self, _leaf("sdf_oriented_infinite_cone"), angle)


class SolidAngle(GenericGeometry):
    def __init__(self, radius, angle_1, angle_2):
        GenericGeometry.__init__(self, _leaf("sdf_solid_angle"), radius, angle_1, angle_2)


def _as_rows(points):
    pts = np.asarray(points)
    if pts.shape[1] < pts.shape[0]:
        pts = pts.T
    return pts


class SegmentedLine3D(GenericGeometry):
    def __init__(self, points, closed=False):
        self._points = _as_rows(points)
        self._closed = closed
        if not closed:
            # geom_3d.py:748-751 returns sdf_segmented_curve_3d (3 positional args) for open lines, so the
            # reference raises TypeError at create(); raise it at construction instead.
            raise TypeError("SegmentedLine3D(closed=False) is broken in the reference (wrong-arity SDF); "
                            "use closed=True or sdf_segmented_line_3d")
        GenericGeometry.__init__(self, _leaf("sdf_closed_segmented_line_3d"), self._points)

    @property
    def closed(self):
        return self._closed


class ParametricCurve3D(GenericGeometry):
    """geom_3d.py:577-648: distance to the nearest sample of f(t), t = linspace(*t_range) (+ closing segment)."""

    def __init__(self, parametric_curve, parametric_curve_parameters, t_range, closed=False):
        self._curve, self._c_params, self._t_range, self._closed = parametric_curve, parametric_curve_parameters, \
            t_range, closed
        GenericGeometry.__init__(self, _leaf("sdf_closed_parametric_curve_3d" if closed else "sdf_parametric_curve_3d"),
                                 parametric_curve, parametric_curve_parameters, self.ts)

    @property
    def ts(self):
        return np.linspace(*self._t_range)

    @property
    def closed(self):
        return self._closed


class _SegmentedParametricBase(GenericGeometry):
    """Polyline through `points`, sampled at parameters ts (point v = floor(t), fraction u = t - v): distance to the
    nearest SAMPLE (sdf_2D.py:180-188, sdf_3D.py:253-261), plus the closing segment when closed."""
    _dim = 2

    def __init__(self, points, t_range, closed=False):
        self._points = _as_rows(points)
        self._t_range = t_range
        self._closed = closed
        name = f"sdf_closed_segmented_curve_{self._dim}d" if closed else f"sdf_segmented_curve_{self._dim}d"
        GenericGeometry.__init__(self, _leaf(name), self._points, self.ts)

    @property
    def steps(self):
        return self._t_range[2]

    @property
    def t_start(self):
        return self._t_range[0]

    @property
    def t_end(self):
        return self._t_range[1]

    @property
    def closed(self):
        return self._closed


class SegmentedParametricCurve(_SegmentedParametricBase):
    """geom_2d.py:460-555."""
    _dim = 2

    def polygon(self):
        """geom_2d.py:530-555: closed curve -> polygon, d * interior_polygon(co, control points)."""
        if not self.closed:
            return self
        return self._add("polygon", points=self._points.copy())

    @property
    def ts(self):  # geom_2d.py:519-523
        tt = np.linspace(self._t_range[0], self._t_range[1] - 1, self._t_range[2])
        return np.clip(tt, 0, self._points.shape[1] - 1.0001)


class SegmentedParametricCurve3D(_SegmentedParametricBase):
    """geom_3d.py:651-714."""
    _dim = 3

    @property
    def ts(self):  # geom_3d.py:704-708: unlike the 2D class the start value is subtracted
        tt = np.linspace(self._t_range[0], self._t_range[1] - 1, self._t_range[2]) - self._t_range[0]
        return np.clip(tt, 0, self._points.shape[1] - 1.0001)


class PointCloud3D(GenericGeometry):
    def __init__(self, points):
        self._points = _as_rows(points)
        GenericGeometry.__init__(self, _leaf("sdf_point_cloud_3d"), self._points)

    @property
    def points(self):
        return self._points


# ----------------------------------------------------------------------------------------------------------------
# 2D primitives (geom_2d.py)


class Circle(GenericGeometry):
    def __init__(self, radius):
        GenericGeometry.__init__(self, _leaf("sdf_circle"), radius)


class NEUCircle(GenericGeometry):
    def __init__(self, radius, order):
        GenericGeometry.__init__(self, _leaf("sdf_neu_circle"), radius, order)


class NGon(GenericGeometry):
    def __init__(self, radius, n_sides):
        GenericGeometry.__init__(self, _leaf("sdf_ngon"), radius, n_sides)


class Rectangle(GenericGeometry):
    def __init__(self, a, b):
        GenericGeometry.__init__(self, _leaf("sdf_box_2d"), (a, b))


class RoundedRectangle(GenericGeometry):
    def __init__(self, a, b, rounding):
        GenericGeometry.__init__(self, _leaf("sdf_rounded_box_2d"), (a, b), rounding[:4])


class Segment(GenericGeometry):
    def __init__(self, a, b):
        GenericGeometry.__init__(self, _leaf("sdf_segment_2d"), a, b)


class Triangle(GenericGeometry):
    def __init__(self, a, b, c):
        GenericGeometry.__init__(self, _leaf("sdf_triangle_2d"), np.asarray(a), np.asarray(b), np.asarray(c))


class Sector(GenericGeometry):
    def __init__(self, radius, angle_1, angle_2):
        GenericGeometry.__init__(self, _leaf("sdf_sector"), radius, angle_1, angle_2)


class InfiniteSector(GenericGeometry):
    def __init__(self, angle_1, angle_2):
        GenericGeometry.__init__(self, _leaf("sdf_inf_sector"), angle_1, angle_2)


class Arc(GenericGeometry):
    def __init__(self, radius, start_angle, end_angle):
        GenericGeometry.__init__(self, _leaf("sdf_arc"), radius, start_angle, end_angle)


class Polygon(GenericGeometry):
    """geom_2d.py:102-125 (simple polygons; vertices (3, N) or (N, 3))."""

    def __init__(self, vertices):
        GenericGeometry.__init__(self, _leaf("sdf_polygon_2d"), vertices)
        vertices = np.array(vertices)
        if not (vertices.shape[1] >= 3 and vertices.shape[0] >= 3):
            raise ValueError("There must be at least 3 vertices defined by their coordinates in 3D space.")
        if 3 not in vertices.shape:
            raise ValueError("The coordinates of vertices should be defined in 3D space.")
        if not (vertices.shape[0] == 3):
            vertices = vertices.T
        self._vertices = vertices
        self._n_sides = vertices.shape[1]

    @property
    def n_sides(self):
        return self._n_sides


class ParametricCurve(GenericGeometry):
    """geom_2d.py:340-457."""

    def __init__(self, parametric_curve, parametric_curve_parameters, t_range, closed=False):
        self._curve, self._c_params, self._t_range, self._closed = parametric_curve, parametric_curve_parameters, \
            t_range, closed
        GenericGeometry.__init__(self, _leaf("sdf_closed_parametric_curve_2d" if closed else "sdf_parametric_curve_2d"),
                                 parametric_curve, parametric_curve_parameters, self.ts)

    @property
    def ts(self):
        return np.linspace(*self._t_range)

    @property
    def closed(self):
        return self._closed

    @property
    def steps(self):
        return self._t_range[2]

    def shape(self):
        """geom_2d.py:415-457: closed curve -> shape. The sign comes from the curve sampled at ts followed by t = 0
        (ts_ = zeros(steps + 1); ts_[:steps] = ts)."""
        if not self.closed:
            return self
        ts_ = np.zeros(self.steps + 1)
        ts_[:self.steps] = self.ts
        return self._add("shape", points=np.asarray(self._curve(ts_, *self._c_params), dtype=np.float64))


class SegmentedLine(GenericGeometry):
    def __init__(self, points, closed=False):
        self._points = _as_rows(points)
        self._closed = closed
        GenericGeometry.__init__(
            self, _leaf("sdf_closed_segmented_line_2d" if closed else "sdf_segmented_line_2d"), self._points)

    @property
    def closed(self):
        return self._closed

    def polygon(self):
        """geom_2d.py:601-626: closed segmented line -> polygon, d * interior_polygon(co, points)."""
        if not self.closed:
            return self
        return self._add("polygon", points=self._points.copy())


class PointCloud2D(GenericGeometry):
    def __init__(self, points):
        self._points = _as_rows(points)
        GenericGeometry.__init__(self, _leaf("sdf_point_cloud_2d"), self._points)

    @property
    def points(self):
        return self._points
