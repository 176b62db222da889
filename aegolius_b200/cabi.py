"""ctypes binding of libaegolius_b200.so (include/aegolius_b200.h). This is the stub a SPOMSO maintainer would add
(see INTEGRATION.md); nothing here evaluates anything on the CPU."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .opcodes import P_FIELD

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libaegolius_b200.so")

AB_OK, AB_EINVAL, AB_EUNSUPPORTED_OP, AB_ECUDA, AB_ETOOLARGE, AB_ENODEVICE = 0, -1, -2, -3, -4, -5
AB_F32, AB_F64 = 0, 1
AB_GRAD_NONE, AB_GRAD_SPATIAL, AB_GRAD_PARAM = 0, 1, 2


class ab_op(C.Structure):
    _fields_ = [("opcode", C.c_uint16), ("a", C.c_uint8), ("b", C.c_uint8), ("arg", C.c_uint32)]


class ab_blob(C.Structure):
    _fields_ = [("data", C.c_void_p), ("count", C.c_uint64), ("dim", C.c_int32), ("on_device", C.c_int32)]


class ab_program(C.Structure):
    _fields_ = [("ops", C.c_void_p), ("n_ops", C.c_uint32), ("args", C.c_void_p), ("n_args", C.c_uint32),
                ("dargs", C.c_void_p), ("blobs", C.POINTER(ab_blob)), ("n_blobs", C.c_uint32),
                ("n_pslots", C.c_uint32), ("n_vslots", C.c_uint32), ("dblobs", C.POINTER(ab_blob))]


class ab_grid(C.Structure):
    _fields_ = [("size", C.c_double * 3), ("res", C.c_uint32 * 3), ("slab_begin", C.c_uint32),
                ("slab_end", C.c_uint32)]


class ab_vec_op(C.Structure):
    _fields_ = [("opcode", C.c_uint32), ("kind0", C.c_uint32), ("kind1", C.c_uint32), ("c", C.c_double * 3),
                ("s0", C.c_double), ("s1", C.c_double), ("a0", C.c_void_p), ("a1", C.c_void_p),
                ("stride0", C.c_uint64), ("stride1", C.c_uint64)]


# ab_vec_opcode / ab_vec_kind / ab_vec_component_id (include/aegolius_b200.h)
(AB_VOP_ADD, AB_VOP_SUB, AB_VOP_RESCALE, AB_VOP_ROT_Z, AB_VOP_ROT_THETA, AB_VOP_ROT_X, AB_VOP_ROT_Y, AB_VOP_ROT_AXIS,
 AB_VOP_REVOLVE_X, AB_VOP_REVOLVE_Y, AB_VOP_REVOLVE_Z, AB_VOP_NORMALIZE) = range(1, 13)
AB_VK_NONE, AB_VK_SCALAR, AB_VK_VEC3, AB_VK_ARRAY, AB_VK_VEC_ARRAY = range(5)
AB_VC_X, AB_VC_Y, AB_VC_Z, AB_VC_PHI, AB_VC_THETA, AB_VC_LENGTH = range(6)
AB_MAX_VEC_OPS = 32


class AegoliusError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libaegolius_b200 error {code}: {msg}")
        self.code = code


class NoDeviceError(AegoliusError):
    pass


_lib = None

_SIGNATURES = {
    "ab_version": (C.c_int, []),
    "ab_last_error": (C.c_char_p, []),
    "ab_device_count": (C.c_int, []),
    "ab_eval_grid": (C.c_int, [C.POINTER(ab_program), C.POINTER(ab_grid), C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_uint64, C.c_int, C.c_void_p]),
    "ab_eval_grid_multicast": (C.c_int, [C.POINTER(ab_program), C.POINTER(ab_grid), C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_uint64, C.c_int, C.c_void_p]),
    "ab_eval_points": (C.c_int, [C.POINTER(ab_program), C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]),
    "ab_eval_grid_loss": (C.c_int, [C.POINTER(ab_program), C.POINTER(ab_grid), C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_void_p]),
    "ab_spec_register": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]),
    "ab_spec_clear": (C.c_int, []),
    "ab_prog_register": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64]),
    "ab_prog_clear": (C.c_int, []),
    "ab_prog_hits": (C.c_uint64, []),
    "ab_prog_enable": (C.c_int, [C.c_int]),
    "ab_prog_signature_hash": (C.c_uint64, [C.c_void_p, C.c_uint32, C.c_int, C.c_int]),
    "ab_prog_arg_layout": (C.c_int, [C.POINTER(ab_program), C.c_void_p, C.POINTER(C.c_uint32)]),
    "ab_op_tier": (C.c_int, [C.c_int]),
    "ab_spec_hits": (C.c_uint64, []),
    "ab_eval_grid_host": (C.c_int, [C.POINTER(ab_program), C.POINTER(ab_grid), C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_uint64, C.c_int]),
    "ab_eval_points_host": (C.c_int, [C.POINTER(ab_program), C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_uint64, C.c_int]),
    "ab_nn_grid": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(ab_grid), C.c_int, C.c_void_p, C.c_int,
                             C.c_void_p]),
    "ab_nn_points": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int,
                               C.c_void_p, C.c_int, C.c_void_p]),
    "ab_cloud_upload": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_uint64, C.c_int, C.c_int,
                                  C.POINTER(C.c_void_p)]),
    "ab_fd_gradient": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(ab_grid), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                 C.c_uint64, C.c_int, C.c_void_p]),
    "ab_box_filter": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_uint32, C.c_int,
                                C.c_void_p, C.c_int, C.c_void_p]),
    "ab_edge_filter": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ab_signed_field": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ab_signed_mask": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_void_p]),
    "ab_signed_field_slab": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32,
                                       C.c_uint32, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ab_signed_field_slab_tangent": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                               C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_int, C.c_void_p]),
    "ab_vec_apply": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(ab_vec_op), C.c_uint32, C.c_int, C.c_int,
                               C.c_void_p]),
    "ab_vec_component": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                   C.c_void_p]),
    "ab_device_alloc": (C.c_int, [C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    "ab_device_free": (C.c_int, [C.c_void_p, C.c_int]),
    "ab_host_alloc_pinned": (C.c_int, [C.c_uint64, C.POINTER(C.c_void_p)]),
    "ab_host_alloc_pinned_flags": (C.c_int, [C.c_uint64, C.c_uint, C.POINTER(C.c_void_p)]),
    "ab_host_free_pinned": (C.c_int, [C.c_void_p]),
    "ab_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]),
    "ab_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]),
    "ab_stream_sync": (C.c_int, [C.c_int, C.c_void_p]),
    "ab_launch_count": (C.c_uint64, []),
}
EXPORTS = tuple(_SIGNATURES)


def lib():
    """Loads the CUDA library; fails loudly if it has not been built (there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m aegolius_b200.build` (needs nvcc). "
                              f"aegolius_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc != AB_OK:
        msg = lib().ab_last_error().decode(errors="replace")
        raise (NoDeviceError if rc == AB_ENODEVICE else AegoliusError)(rc, msg)


def device_count() -> int:
    return int(lib().ab_device_count())


def launch_count() -> int:
    return int(lib().ab_launch_count())


class CProgram:
    """Keeps the numpy buffers of a Program alive and exposes an ab_program struct. `device_blobs[b]` = (pointer, count) binds
    the device field of a P_FIELD blob; `device_dblobs[b]` = (pointer, count) its tangent row (AB_GRAD_PARAM)."""

    def __init__(self, prog, device_blobs=None, device_dblobs=None):
        self._ops = np.ascontiguousarray(prog.ops)
        self._args = np.ascontiguousarray(prog.args, dtype=np.float64)
        self._blob_arrays = [np.ascontiguousarray(b, dtype=np.float64) for b in prog.blobs]
        n_blobs = len(self._blob_arrays)
        self._blobs = (ab_blob * max(1, n_blobs))()
        fields = {st["blob"] for st in getattr(prog, "stages", ())}  # P_FIELD inputs: device arrays, one value per point
        read = {int(b) for c, b in zip(prog.ops["opcode"], prog.ops["b"]) if int(c) == P_FIELD}
        for i, b in enumerate(self._blob_arrays):
            if i in fields and i not in read and (device_blobs is None or device_blobs[i] is None):
                self._blobs[i] = ab_blob(None, 0, 1, 1)  # a stage whose field this program never reads (pruned away)
            elif i in fields:
                if device_blobs is None or device_blobs[i] is None:
                    raise ValueError("this program has grid-stencil stages: evaluate it through aegolius_b200.create "
                                     "on a whole grid (the stages need the full field)")
                ptr, count = device_blobs[i]
                self._blobs[i] = ab_blob(ptr, count, 1, 1)
            elif device_blobs is not None and device_blobs[i] is not None:
                self._blobs[i] = ab_blob(device_blobs[i], b.shape[1], 3, 1)
            else:
                self._blobs[i] = ab_blob(b.ctypes.data, b.shape[1], 3, 0)
        self._dargs = None
        if getattr(prog, "dargs", None) is not None:
            self._dargs = np.ascontiguousarray(prog.dargs, dtype=np.float64)
            if self._dargs.shape != self._args.shape:
                raise ValueError("Program.dargs must have the shape of Program.args")
        self._dblobs = None
        if device_dblobs is not None:
            self._dblobs = (ab_blob * max(1, n_blobs))()
            for i, d in enumerate(device_dblobs):
                if d is not None:
                    self._dblobs[i] = ab_blob(d[0], d[1], 1, 1)
        self.struct = ab_program(self._ops.ctypes.data, self._ops.shape[0], self._args.ctypes.data,
                                 self._args.shape[0], self._dargs.ctypes.data if self._dargs is not None else None,
                                 self._blobs, n_blobs, prog.n_pslots, prog.n_vslots, self._dblobs)

    def ref(self):
        return C.byref(self.struct)


def make_grid(size, res, slab=None):
    g = ab_grid()
    for i in range(3):
        g.size[i] = float(size[i])
        g.res[i] = int(res[i])
    g.slab_begin, g.slab_end = (0, int(res[0])) if slab is None else (int(slab[0]), int(slab[1]))
    return g
