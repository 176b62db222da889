"""Evaluation front door: the drop-in for GenericGeometry.create(co) (Code/spomso/spomso/cores/geom.py:29-43),
from_sdf (vector_functions.py:130-139) and sdf_point_cloud_* (sdf_3D.py:283-286, sdf_2D.py:221-224).

    field = aegolius_b200.create(obj, co)                        # obj: SPOMSO object or frontend object
    field, grad = aegolius_b200.create(obj, co, grad="spatial")  # analytic gradient (forward-mode duals)
    aegolius_b200.patch()                                        # rebind spomso's GenericGeometry.create

Everything is computed by libaegolius_b200.so on the GPU; if the library or a device is missing the call raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import cabi
from .grid import resolution_conversion, GridSpec, detect_grid
from .program import Program, flatten
from . import opcodes as oc
from . import codegen

_DT = {"f32": (cabi.AB_F32, np.float32), "f64": (cabi.AB_F64, np.float64),
       "float32": (cabi.AB_F32, np.float32), "float64": (cabi.AB_F64, np.float64),
       np.float32: (cabi.AB_F32, np.float32), np.float64: (cabi.AB_F64, np.float64)}


def library_path():
    return cabi.LIB_PATH


def _dtype(dtype):
    try:
        return _DT[dtype]
    except (KeyError, TypeError):
        return _DT[np.dtype(dtype).type]


def _as_program(obj) -> Program:
    return obj if isinstance(obj, Program) else flatten(obj)


def _grad_mode(grad):
    if grad in (None, False, "none"):
        return cabi.AB_GRAD_NONE, 0
    if grad in (True, "spatial", "xyz"):
        return cabi.AB_GRAD_SPATIAL, 3
    if grad == "param":
        return cabi.AB_GRAD_PARAM, 1
    raise ValueError(f"unknown grad mode {grad!r} (use None, 'spatial' or 'param')")


def _is_2d(spec) -> bool:
    """The grids the kernels walk as (1, nx, ny) (make_gridk in csrc/ab_capi.cu)."""
    return spec.res[2] == 1 and spec.res[1] > 1 and float(spec.size[2]) == 0.0


def compile_program(obj, *, dtype="f32", grad=None, is2d=False, **opts):
    """Blocks until the straight-line kernel for this program's structure is built (nvcc, a few seconds, cached under
    aegolius_b200/jit/) and registered. create() / create_torch() do the same in the background on first use; this is
    for callers who want the first evaluation to run on it already."""
    prog = _as_program(obj)
    code, _ = _dtype(dtype)
    return codegen.ensure(prog, "f32" if code == cabi.AB_F32 else "f64", grad, is2d=is2d, how="sync", **opts)


def wait_for_compilations(timeout=None):
    """Blocks until every background kernel build started so far is registered."""
    codegen.wait(timeout)


def slab_ranges(n_planes: int, parts: int):
    """np.array_split(range(n_planes), parts) as (begin, end) pairs: contiguous x-slabs (SURVEY §8e)."""
    base, extra = divmod(n_planes, parts)
    out, s = [], 0
    for r in range(parts):
        e = s + base + (1 if r < extra else 0)
        out.append((s, e))
        s = e
    return out


_SPEC_LIBS = {}


def specialize(obj, *, dtype="f32", grad=None, verbose=False):
    """Optional: compiles (once, cached under aegolius_b200/spec/) a build of the interpreter that contains only the ops
    of this program and registers it with the library; every later evaluation of a program whose ops are covered, with
    the same dtype and gradient mode, runs on it. Results are identical (same op bodies); the kernel is a fraction of the
    general one's size, which matters because the deep trees are instruction-cache-bound (C3 + gradient: -13 %).
    Needs nvcc at run time; costs one compilation (about ten seconds) per distinct (op set, dtype, grad). Programs of the
    lite tier are left alone (returns None): their general kernel is already small and runs wider."""
    from . import build as _build
    prog = _as_program(obj)
    code, _ = _dtype(dtype)
    gmode, _ = _grad_mode(grad)
    if gmode == cabi.AB_GRAD_PARAM:
        kind = 4 if code == cabi.AB_F32 else 5
    else:
        kind = (0 if code == cabi.AB_F32 else 2) + (1 if gmode == cabi.AB_GRAD_SPATIAL else 0)
    if gmode != cabi.AB_GRAD_PARAM and max(cabi.lib().ab_op_tier(int(o)) for o in prog.ops["opcode"]) == 0:
        # lite programs already run on a 23 KB kernel with twice the points per thread; a specialised build at the
        # standard width is slower (C1 at 1025^3: 3.0 -> 3.9 ms)
        return None
    used = sorted({oc.NAMES[int(o)] for o in prog.ops["opcode"]})
    path = _build.build_specialized(used, kind, verbose=verbose)
    if path not in _SPEC_LIBS:
        lib = C.CDLL(path)
        lib.ab_spec_kparams_size.restype = C.c_uint64
        if lib.ab_spec_kind() != kind:
            raise RuntimeError(f"{path}: wrong kind")
        mask = (C.c_uint8 * oc.OP_COUNT)()
        for name in used + ["END"]:
            mask[{v: k for k, v in oc.NAMES.items()}[name]] = 1
        cabi.check(cabi.lib().ab_spec_register(code, gmode, mask, oc.OP_COUNT, C.cast(lib.ab_spec_launch, C.c_void_p),
                                               lib.ab_spec_kparams_size()))
        _SPEC_LIBS[path] = lib  # keeps the shared object loaded
    return path


_AUTO_SPEC = {"on": False, "pending": {}, "lock": None}


def set_auto_specialize(enable=True):
    """Opt-in: every evaluation of a program that has no specialised kernel yet starts ONE background compilation for its
    (op set, dtype, gradient mode); evaluations keep running on the general kernels until the build is registered, then
    switch to it. Off by default (it launches nvcc on the host)."""
    import threading
    _AUTO_SPEC["on"] = bool(enable)
    if _AUTO_SPEC["lock"] is None:
        _AUTO_SPEC["lock"] = threading.Lock()


def wait_for_specializations(timeout=None):
    """Blocks until the background builds started so far are registered (tests, benchmarks)."""
    for th in list(_AUTO_SPEC["pending"].values()):
        th.join(timeout)


def _auto_specialize(prog, dtype, grad):
    if not _AUTO_SPEC["on"] or prog.stages:
        return
    import threading
    key = (tuple(sorted({int(o) for o in prog.ops["opcode"]})), str(dtype), str(grad))
    with _AUTO_SPEC["lock"]:
        if key in _AUTO_SPEC["pending"]:
            return

        def work():
            try:
                specialize(prog, dtype=dtype, grad=grad)
            except Exception:  # no nvcc / compile error: stay on the general kernels
                pass

        th = threading.Thread(target=work, name="aegolius-specialize", daemon=True)
        _AUTO_SPEC["pending"][key] = th
        th.start()


def bind_to_device_numa(device=0):
    """Pins the calling process to the CPUs NVML reports as local to `device` (same PCIe root / NUMA node), so that
    page-locked buffers allocated afterwards land in memory next to the GPU and the D2H leg does not cross sockets.
    Returns the CPU set, or None when NVML / affinity control is unavailable (nothing is changed then)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        # honour CUDA_VISIBLE_DEVICES: NVML enumerates physical devices
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[device]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else device
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


class PinnedArray:
    """Page-locked host buffer exposed as a numpy array (for the D2H leg of create())."""

    def __init__(self, shape, dtype, portable=False, write_combined=False):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        cabi.check(cabi.lib().ab_host_alloc_pinned_flags(nbytes, (1 if portable else 0) | (2 if write_combined else 0),
                                                         C.byref(p)))
        self._ptr = p
        buf = (C.c_char * max(1, nbytes)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._ptr is not None:
            self.array = None
            cabi.lib().ab_host_free_pinned(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_STAGED_ONLY = ("programs with grid stencils (conv_averaging / conv_edge_detection / signed modifications) are evaluated on "
                "grids only, without gradients in x, y, z (a stencil's output depends on the whole grid, so it has no "
                "pointwise spatial derivative); parameter tangents (grad='param') are supported")


def create(obj, co, *, dtype="f32", grad=None, device=0, out=None, out_grad=None, slab=None):
    """Evaluates the SDF of `obj` on `co`.

    obj   : SPOMSO GenericGeometry (any subclass), aegolius_b200 frontend object, or a flattened Program.
    co    : GridSpec / GridCoords / plain (3,N) float64 array. Arrays produced by SPOMSO's generate_grid are
            recognised (grid mode: coordinates are regenerated in-kernel); anything else is uploaded (points mode).
    dtype : "f32" (default) or "f64" (bit-compatible output type with the reference, tighter parity).
    grad  : None or "spatial" -> returns (field, gradient (3,N)).
    slab  : (x0, x1) plane range of a grid to evaluate (multi-GPU sharding along the slowest axis).
    Returns a numpy array (N,) of `dtype` (and the (3,N) gradient).
    """
    prog = _as_program(obj)
    code, npdt = _dtype(dtype)
    gmode, rows = _grad_mode(grad)
    spec = detect_grid(co)
    if prog.stages:
        if spec is None or gmode == cabi.AB_GRAD_SPATIAL:
            raise NotImplementedError(_STAGED_ONLY)
        x0, x1 = (0, spec.res[0]) if slab is None else slab
        n = (x1 - x0) * spec.res[1] * spec.res[2]
        field = out if out is not None else np.empty(n, dtype=npdt)
        if field.dtype != npdt or field.size != n or not field.flags.c_contiguous:
            raise ValueError("out= must be a C-contiguous array of the evaluation dtype with N elements")
        if not rows:
            field[...] = _staged_torch(prog, spec, code, slab, None, device).cpu().numpy()
            return field
        g_arr = out_grad if out_grad is not None else np.empty((rows, n), dtype=npdt)
        if g_arr.dtype != npdt or g_arr.shape != (rows, n) or not g_arr.flags.c_contiguous:
            raise ValueError("out_grad= must be a C-contiguous (1, N) array of the evaluation dtype")
        f_dev, g_dev = _staged_torch(prog, spec, code, slab, None, device, param=True)
        field[...] = f_dev.cpu().numpy()
        g_arr[...] = g_dev.cpu().numpy()
        return field, g_arr
    _auto_specialize(prog, dtype, grad)
    if (spec is not None and not rows and out is None and prog.n_ops == 2
            and int(prog.ops[0]["opcode"]) == oc.P_POINT_CLOUD):
        # a bare, untransformed cloud on a grid (PointCloud3D(points).create(coor)): the dedicated nearest-neighbour
        # path walks its octree once per warp of samples instead of once per sample
        dim = int(prog.ops[0]["a"])
        return point_cloud_sdf(spec, prog.blobs[int(prog.ops[0]["b"])][:dim], dim=dim, dtype=dtype, device=device, slab=slab)
    # default path: the straight-line kernel compiled for this program's structure (built in the background on first
    # use and cached on disk; the interpreter serves the calls made meanwhile — identical results either way)
    codegen.ensure(prog, "f32" if code == cabi.AB_F32 else "f64", grad, is2d=spec is not None and _is_2d(spec))
    cp = cabi.CProgram(prog)
    lib = cabi.lib()
    if spec is not None:
        x0, x1 = (0, spec.res[0]) if slab is None else slab
        n = (x1 - x0) * spec.res[1] * spec.res[2]
        g = cabi.make_grid(spec.size, spec.res, (x0, x1))
    else:
        if slab is not None:
            raise ValueError("slab= needs grid coordinates")
        co = np.ascontiguousarray(np.asarray(co, dtype=np.float64))
        if co.ndim != 2 or co.shape[0] not in (2, 3):
            raise ValueError(f"coordinates must have shape (3, N) or (2, N), got {co.shape}")
        if co.shape[0] == 2:
            co = np.concatenate([co, np.zeros((1, co.shape[1]))], axis=0)
        n = co.shape[1]
    field = out if out is not None else np.empty(n, dtype=npdt)
    if field.dtype != npdt or field.size != n or not field.flags.c_contiguous:
        raise ValueError("out= must be a C-contiguous array of the evaluation dtype with N elements")
    gptr, gstride, g_arr = None, 0, None
    if rows:
        g_arr = out_grad if out_grad is not None else np.empty((rows, n), dtype=npdt)
        if g_arr.dtype != npdt or g_arr.shape != (rows, n) or not g_arr.flags.c_contiguous:
            raise ValueError("out_grad= must be a C-contiguous (3, N) array of the evaluation dtype")
        gptr, gstride = g_arr.ctypes.data, n
    if n == 0:
        return (field, g_arr) if rows else field
    if spec is not None:
        cabi.check(lib.ab_eval_grid_host(cp.ref(), C.byref(g), code, gmode, field.ctypes.data, gptr, gstride, device))
    else:
        cabi.check(lib.ab_eval_points_host(cp.ref(), co.ctypes.data, n, n, code, gmode, field.ctypes.data, gptr,
                                           gstride, device))
    return (field, g_arr) if rows else field


def grid_min_step(spec):
    """min over the axes of |co[i, 1] - co[i, 0]| on generate_grid coordinates (modifications.py:239-240): the threshold
    below which `signed` calls a sample "boundary". Evaluated like np.linspace does (start + 1 * step)."""
    seps = []
    for size, n in zip(spec.size, spec.res):
        x = np.linspace(-float(size) / 2, float(size) / 2, int(n))
        seps.append(abs(x[1] - x[0]))
    return float(min(seps))


def _check_stage_grid(prog, spec):
    for st in prog.stages:
        want = tuple(resolution_conversion(int(r)) for r in st["res"] if r)
        if want != tuple(spec.res[:len(want)]) or (len(want) == 2 and spec.res[2] != 1):
            raise ValueError(f"Cannot reshape the pattern with shape ({spec.n_points},)")  # what smarter_reshape raises
        if st["kind"] == 2 and min(spec.res) < 3:
            raise ValueError("can't extend empty axis using modes other than 'constant' or 'empty'")  # np.pad


def _staged_torch(prog, spec, code, slab, out, device, mask_gather=None, *, param=False, out_grad=None, loss=None):
    """Programs with grid-stencil stages on the x-slab `slab` of a grid, into the torch tensor `out` (or a new one), on the
    current torch stream. Program.stage_plan says on which planes each stage is needed: in program order, the pruned
    prefix program ops[:k] is evaluated on the stage's planned range (with the fields of earlier stages bound), filtered by
    ab_box_filter / ab_edge_filter as if that range were the whole field (reflection at a cut only corrupts the halo, which
    the plan keeps out of the planes read later; at a grid face it reflects as the whole field does), or signed from the
    boundary mask of the whole field (ab_signed_mask / ab_signed_field_slab); the result is bound to the P_FIELD op that
    replaced the modification, slab-local, and the pruned program runs on the slab. Intermediate fields come from the torch
    allocator; nothing is synchronised.

    The mask of a signed stage covers every plane. Without `mask_gather` this process evaluates the stage's prefix on the
    whole axis to pack it (the cost of one whole-grid prefix evaluation per signed stage, even for a thin slab). A sharded
    evaluation passes a distributed.MaskGather: this process packs the mask of `mask_gather.planes` only, and
    mask_gather(local_words, words_per_plane, flags) returns the whole mask (and max-reduces the two flags in place).

    param=True carries the parameter tangent prog.dargs through the same pipeline: every stencil is linear in its field, so
    d(stage)/d theta is the same stencil on the tangent of its input. Each prefix runs in AB_GRAD_PARAM mode into a value
    and a tangent row, the box / edge filter runs on both rows, `signed` applies the sign pattern of the value (mask from the
    value only) to both (ab_signed_field_slab_tangent), and each tangent row is bound to its P_FIELD op beside the field.
    Returns (field, (1, n) tangent) into `out` / `out_grad` (a (1, >= n) tensor), or, with loss=(target, accum), runs the
    final program through ab_eval_grid_loss (accum[0] = sum r^2, accum[1] = sum 2 r dF/dtheta over the slab) and returns
    None."""
    import torch
    _check_stage_grid(prog, spec)
    if param and prog.dargs is None:
        raise ValueError("grad='param' needs Program.dargs (engine.program_tangent)")
    gmode = cabi.AB_GRAD_PARAM if param else cabi.AB_GRAD_NONE
    dev = torch.device("cuda", device)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    tdt = torch.float32 if code == cabi.AB_F32 else torch.float64
    jdt = "f32" if code == cabi.AB_F32 else "f64"
    item = 4 if code == cabi.AB_F32 else 8
    lib = cabi.lib()
    n0, pp = spec.res[0], spec.res[1] * spec.res[2]
    x0, x1 = (0, n0) if slab is None else (int(slab[0]), int(slab[1]))
    plan, _ = prog.stage_plan(spec.res, (x0, x1), None if mask_gather is None else mask_gather.planes)
    fields = {}  # blob -> (device tensor, its tangent row or None, their first plane)
    res3 = lambda m: (C.c_uint32 * 3)(m, spec.res[1], spec.res[2])

    def run(p, lo, hi, dst, ddst=None, target=None):
        bound, dbound = [None] * len(prog.blobs), [None] * len(prog.blobs)
        for blob, (t, dt, p0) in fields.items():
            if p0 <= lo and hi - p0 <= t.numel() // pp:  # the plan makes every field a program reads cover its range
                bound[blob] = (t.data_ptr() + (lo - p0) * pp * item, (hi - lo) * pp)
                if dt is not None:
                    dbound[blob] = (dt.data_ptr() + (lo - p0) * pp * item, (hi - lo) * pp)
        cp = cabi.CProgram(p, device_blobs=bound, device_dblobs=dbound if param else None)
        codegen.ensure(p, jdt, "param" if param else None, is2d=_is_2d(spec))
        g = cabi.make_grid(spec.size, spec.res, (lo, hi))
        if target is not None:
            cabi.check(lib.ab_eval_grid_loss(cp.ref(), C.byref(g), code, C.c_void_p(target.data_ptr()),
                                             C.c_void_p(loss[1].data_ptr()), device, stream))
            return
        cabi.check(lib.ab_eval_grid(cp.ref(), C.byref(g), code, gmode, C.c_void_p(dst.data_ptr()),
                                    C.c_void_p(ddst.data_ptr()) if param else None, ddst.stride(0) if param else 0,
                                    device, stream))

    def rows(m):  # value row and (param) tangent row of m samples
        return (torch.empty(m, dtype=tdt, device=dev),
                torch.empty((1, m), dtype=tdt, device=dev) if param else None)

    for st, ev, valid in plan:
        if ev is None:
            continue  # no later program reads this stage
        lo, hi = ev
        pre = prog.prefix(prog.stage_op_index(st)).pruned()  # without the subtrees an earlier stage's field replaced
        src, dsrc = rows((hi - lo) * pp)
        run(pre, lo, hi, src, dsrc)
        srcs = [src] + ([dsrc] if param else [])
        if st["kind"] in (0, 1):  # box / edge filter: linear, the tangent row takes the same stencil
            dsts = [torch.empty_like(x) for x in srcs]
            for a, b in zip(srcs, dsts):
                if st["kind"] == 0:
                    cabi.check(lib.ab_box_filter(C.c_void_p(a.data_ptr()), res3(hi - lo), (C.c_uint32 * 3)(*st["ksize"]),
                                                 st["iterations"], code, C.c_void_p(b.data_ptr()), device, stream))
                else:
                    cabi.check(lib.ab_edge_filter(C.c_void_p(a.data_ptr()), res3(hi - lo), code, C.c_void_p(b.data_ptr()),
                                                  device, stream))
            fields[st["blob"]] = (dsts[0], dsts[1] if param else None, lo)
        else:
            words = (spec.res[2] + 31) // 32
            wpp = spec.res[1] * words  # mask words per plane
            flags = torch.zeros(2, dtype=torch.int32, device=dev)
            m0, m1 = (0, n0) if mask_gather is None else mask_gather.planes
            mask = torch.empty((m1 - m0) * wpp, dtype=torch.int32, device=dev)
            cabi.check(lib.ab_signed_mask(C.c_void_p(src.data_ptr() + (m0 - lo) * pp * item), res3(m1 - m0),
                                          grid_min_step(spec), code, C.c_void_p(mask.data_ptr()),
                                          C.c_void_p(flags.data_ptr()), device, stream))
            if mask_gather is not None:
                mask = mask_gather(mask, wpp, flags)
            dst, ddst = rows((valid[1] - valid[0]) * pp)
            if param:  # the value's sign pattern on both rows (the mask depends on theta only piecewise constantly)
                cabi.check(lib.ab_signed_field_slab_tangent(
                    C.c_void_p(mask.data_ptr()), C.c_void_p(flags.data_ptr()), C.c_void_p(src.data_ptr()),
                    C.c_void_p(dsrc.data_ptr()), lo, (C.c_uint32 * 3)(*spec.res), valid[0], valid[1], code,
                    C.c_void_p(dst.data_ptr()), C.c_void_p(ddst.data_ptr()), device, stream))
            else:
                cabi.check(lib.ab_signed_field_slab(C.c_void_p(mask.data_ptr()), C.c_void_p(flags.data_ptr()),
                                                    C.c_void_p(src.data_ptr()), lo, (C.c_uint32 * 3)(*spec.res), valid[0],
                                                    valid[1], code, C.c_void_p(dst.data_ptr()), device, stream))
            fields[st["blob"]] = (dst, ddst, valid[0])
        del src, dsrc, srcs
    n = (x1 - x0) * pp
    # the subtrees that fed the stages are dead code now: P_FIELD overwrites their value
    if loss is not None:
        if loss[0].numel() != n or loss[0].dtype != tdt or not loss[0].is_contiguous():
            raise ValueError("the target must be a contiguous tensor of the evaluation dtype with one value per slab sample")
        run(prog.pruned(), x0, x1, None, target=loss[0])
        return None
    if out is None:
        out = torch.empty(n, dtype=tdt, device=dev)
    elif out.numel() != n or out.dtype != tdt or not out.is_contiguous() or out.device != dev:
        raise ValueError("out= must be a contiguous CUDA tensor of the evaluation dtype with one value per slab sample")
    if not param:
        run(prog.pruned(), x0, x1, out)
        return out
    gbuf = out_grad if out_grad is not None else torch.empty((1, (n + 7) // 8 * 8), dtype=tdt, device=dev)
    if gbuf.dim() != 2 or gbuf.shape[1] < n or gbuf.dtype != tdt or gbuf.stride(1) != 1 or gbuf.device != dev:
        raise ValueError("out_grad= must be a (1, >= N) CUDA tensor of the evaluation dtype with unit column stride")
    run(prog.pruned(), x0, x1, out, gbuf)
    return out, gbuf[:, :n]


def create_with_gradient(obj, co, **kw):
    return create(obj, co, grad="spatial", **kw)


# ---- parameter sensitivities (stand-in for jacfwd(geometry, argnums=k), Code/examples/autodiff/gradient_map_3D.py:84) ----


def program_tangent(geometry, params, argnum, rel_step=1e-6):
    """Flattens geometry(*params) and attaches Program.dargs = d args / d params[argnum].

    The host-side folding (rotation matrices, frames, sin/cos of constant angles ...) is differentiated numerically in
    fp64 by a central difference of the flattened argument pools (structure must not change with the parameter); the
    kernel then propagates the tangent analytically (forward-mode dual numbers) through every op."""
    params = list(params)
    theta = float(params[argnum])
    h = rel_step * max(1.0, abs(theta))
    lo, hi = list(params), list(params)
    lo[argnum], hi[argnum] = theta - h, theta + h
    p0, p_lo, p_hi = (flatten(geometry(*q), fold_frames=False) for q in (params, lo, hi))
    if not (np.array_equal(p0.ops, p_lo.ops) and np.array_equal(p0.ops, p_hi.ops)):
        raise ValueError("the program structure changes with the parameter; cannot differentiate through it")
    if not p0.stages == p_lo.stages == p_hi.stages:  # e.g. a kernel size or iteration count derived from the parameter
        raise ValueError("a grid-stencil stage changes with the parameter; cannot differentiate through it")
    # arguments the parameter does not reach are bit-identical at theta - h and theta + h: exactly zero tangent, nothing
    # is thresholded away (a genuinely small derivative stays). The remaining tangents carry the central difference's
    # ~h^2 truncation error of the HOST-side folding (rotation matrices, frames, sin / cos of constant angles); the kernel
    # propagates them analytically.
    p0.dargs = np.where(p_hi.args == p_lo.args, 0.0, (p_hi.args - p_lo.args) / (2.0 * h))
    return p0


def jacfwd(geometry, argnums=0, *, mode="dual", dtype="f64", rel_step=1e-6, device=0):
    """Returns g(co, *params) -> d field / d params[argnums] for a builder `geometry(*params) -> geometry object`:
    the counterpart of jacfwd(geometry, argnums=k)(*p) in Code/examples/autodiff/gradient_map_3D.py:84.

    mode="dual" (default): forward-mode dual numbers inside the interpreter (AB_GRAD_PARAM): every op reads its
        arguments as (value, d/d theta) pairs. Parameters that reach a table argument (curve-instance records,
        polyline / polygon / triangle vertices, sector tables) are not supported there.
    mode="fd": both programs at params[k] +- h evaluated in fp64 on the GPU, central difference (~1e-9 relative);
        works for every op.
    Trees with grid-stencil stages take both modes on grids: in dual mode the tangent goes through the same stencils
    (_staged_torch)."""

    def grad_map_dual(co, *params):
        prog = program_tangent(geometry, params, argnums, rel_step)
        return create(prog, co, dtype=dtype, grad="param", device=device)[1][0]

    def grad_map(co, *params):
        params = list(params)
        theta = float(params[argnums])
        h = rel_step * max(1.0, abs(theta))
        lo, hi = list(params), list(params)
        lo[argnums], hi[argnums] = theta - h, theta + h
        f_hi = create(geometry(*hi), co, dtype="f64", device=device)
        f_lo = create(geometry(*lo), co, dtype="f64", device=device)
        f_hi -= f_lo
        f_hi *= 1.0 / (2.0 * h)
        return f_hi

    if mode == "dual":
        return grad_map_dual
    if mode == "fd":
        return grad_map
    raise ValueError("mode must be 'dual' or 'fd'")


def value_and_grad(geometry, spec, target, *, dtype="f32", device=0, post=None, specialized=False):
    """Counterpart of jax.value_and_grad(worker)(params) in Code/examples/autodiff/position_optimization.py:101-179 for the
    least-squares objective used there: loss(params) = sum((F(params) - target)^2), F = field of geometry(*params) on the
    grid `spec`. Returns f(params) -> (loss, d loss / d params).

    One AB_GRAD_PARAM launch per parameter (K forward-mode passes; K is a handful of shape parameters). Without `post`
    the sums  sum(r^2), sum(2 r dF/dtheta_k)  are reduced inside the kernel (ab_eval_grid_loss: no per-point stores, two
    doubles come back); with `post` the launch returns (F, dF/dtheta_k) as torch tensors and the sums are torch reductions.
    `target` is a torch CUDA tensor or array of N values; `post(F, dF)` may map the field before the residual (e.g. a
    falloff) and must return the transformed pair. specialized=True runs the loop on a program-specialised build of the
    tangent kernel (engine.specialize, needs nvcc once)."""
    import torch
    dev = torch.device("cuda", device)
    tdt = torch.float32 if _dtype(dtype)[0] == cabi.AB_F32 else torch.float64
    tgt = torch.as_tensor(np.asarray(target) if not torch.is_tensor(target) else target, dtype=tdt, device=dev)

    code = _dtype(dtype)[0]
    accum = torch.zeros(2, dtype=torch.float64, device=dev)

    def f(params):
        params = [float(v) for v in params]
        grads, loss = [], None
        for k in range(len(params)):
            prog = program_tangent(geometry, params, k)
            if specialized and prog.stages:
                raise NotImplementedError("specialized=True does not cover trees with grid stencils (their prefix programs "
                                          "run on the general or program-compiled kernels); call without it")
            if specialized:  # one compilation per op set (cached); later steps of the optimisation loop reuse it
                specialize(prog, dtype=dtype, grad="param")
            if post is None:
                # fused: the kernel reduces sum r^2 and sum 2 r dF/dtheta_k itself (ab_eval_grid_loss), nothing is stored
                if prog.stages:  # the staged pipeline, with the reduction in the final program's kernel
                    _staged_torch(prog, spec, code, None, None, device, param=True, loss=(tgt, accum))
                else:
                    cp = cabi.CProgram(prog)
                    codegen.ensure(prog, "f32" if code == cabi.AB_F32 else "f64", "param", is2d=_is_2d(spec))
                    g = cabi.make_grid(spec.size, spec.res)
                    stream = torch.cuda.current_stream(dev).cuda_stream
                    cabi.check(cabi.lib().ab_eval_grid_loss(cp.ref(), C.byref(g), code, tgt.data_ptr(), accum.data_ptr(),
                                                            device, C.c_void_p(stream)))
                both = accum.cpu()
                if loss is None:
                    loss = float(both[0])
                grads.append(float(both[1]))
                continue
            field, dfield = create_torch(prog, spec, dtype=dtype, grad="param", device=device)
            dfield = dfield[0]
            field, dfield = post(field, dfield)
            r = field - tgt
            if loss is None:
                loss = float(torch.sum(r * r))
            grads.append(float(torch.sum(2.0 * r * dfield)))
        return loss, np.asarray(grads)

    return f


# ---- device-resident evaluation (torch owns the memory and the stream) ------------------------------------------------------


def create_torch(obj, spec: GridSpec, *, dtype="f32", grad=None, device=0, slab=None, out=None, out_grad=None,
                 mask_gather=None):
    """Grid evaluation into torch CUDA tensors on the current torch stream (no host copy). Returns field
    (and gradient (3,N) view of a row-padded buffer). Programs with grid-stencil stages evaluate their stages on the
    slab plus the halo they need (_staged_torch, where `mask_gather` is described); they take grad='param' (the tangent
    goes through the same stencils) but no spatial gradient."""
    import torch
    prog = _as_program(obj)
    code, npdt = _dtype(dtype)
    if prog.stages:
        gmode, _ = _grad_mode(grad)
        if gmode == cabi.AB_GRAD_SPATIAL:
            raise NotImplementedError(_STAGED_ONLY)
        return _staged_torch(prog, spec, code, slab, out, device, mask_gather, param=gmode == cabi.AB_GRAD_PARAM,
                             out_grad=out_grad)
    _auto_specialize(prog, dtype, grad)
    codegen.ensure(prog, "f32" if code == cabi.AB_F32 else "f64", grad, is2d=_is_2d(spec))
    tdt = torch.float32 if code == cabi.AB_F32 else torch.float64
    gmode, rows = _grad_mode(grad)
    x0, x1 = (0, spec.res[0]) if slab is None else slab
    n = (x1 - x0) * spec.res[1] * spec.res[2]
    dev = torch.device("cuda", device)
    field = out if out is not None else torch.empty(n, dtype=tdt, device=dev)
    gbuf, gptr, stride = None, None, 0
    if rows:
        stride = (n + 7) // 8 * 8
        gbuf = out_grad if out_grad is not None else torch.empty((rows, stride), dtype=tdt, device=dev)
        gptr, stride = gbuf.data_ptr(), gbuf.stride(0)
    cp = cabi.CProgram(prog)
    g = cabi.make_grid(spec.size, spec.res, (x0, x1))
    stream = torch.cuda.current_stream(dev).cuda_stream
    cabi.check(cabi.lib().ab_eval_grid(cp.ref(), C.byref(g), code, gmode, field.data_ptr(), gptr, stride, device,
                                       C.c_void_p(stream)))
    return (field, gbuf[:, :n]) if rows else field


def from_sdf_torch(field, co_resolution, *, slab=None, field_plane0=0, normalize=True, device=0, out=None):
    """from_sdf (vector_functions.py:130-139) on a torch CUDA tensor, on the current torch stream, for a slab of ix planes
    (multi-GPU: distributed.from_sdf_sharded). `field` holds planes [field_plane0, ...) of the grid and must cover the
    slab plus one halo plane on each side that exists in the grid (np.gradient's central stencil); returns the
    (dims, n_slab) view of a row-padded buffer. Concatenating the slabs' results along axis 1 equals the whole-grid call."""
    import torch
    res = tuple(int(r) for r in np.asarray(co_resolution).reshape(-1))
    dims = len(res)
    if dims not in (2, 3):
        raise ValueError("co_resolution must have 2 or 3 entries")
    code = cabi.AB_F32 if field.dtype == torch.float32 else cabi.AB_F64
    x0, x1 = (0, res[0]) if slab is None else (int(slab[0]), int(slab[1]))
    per_plane = int(np.prod(res[1:]))
    lo, hi = max(x0 - 1, 0), min(x1 + 1, res[0])
    if field_plane0 > lo or field.numel() < (hi - field_plane0) * per_plane:
        raise ValueError(f"the field must cover planes [{lo}, {hi}) (slab plus halo); it starts at plane {field_plane0} "
                         f"and holds {field.numel() // per_plane}")
    n = (x1 - x0) * per_plane
    stride = (n + 7) // 8 * 8
    buf = out if out is not None else torch.empty((dims, stride), dtype=field.dtype, device=field.device)
    g = cabi.make_grid((0.0, 0.0, 0.0), res + ((1,) if dims == 2 else ()), (x0, x1))
    stream = torch.cuda.current_stream(field.device).cuda_stream
    cabi.check(cabi.lib().ab_fd_gradient(field.data_ptr(), int(field_plane0), C.byref(g), dims, code, 1 if normalize else 0,
                                         buf.data_ptr(), buf.stride(0), device, C.c_void_p(stream)))
    return buf[:, :n]


def cloud_records(points, dim=3, dtype="f32", device=0):
    """(x, y, z, 0) records of the evaluation dtype on the device, as a torch tensor (M, 4): the layout ab_nn_grid /
    ab_nn_points read. Built once and reused across calls (or broadcast to the other ranks, distributed.py)."""
    import torch
    _, npdt = _dtype(dtype)
    pts = np.asarray(points, dtype=np.float64)
    if pts.ndim != 2 or pts.shape[0] < dim:
        raise ValueError(f"points must have shape ({dim}, M)")
    rec = np.zeros((pts.shape[1], 4), dtype=npdt)
    rec[:, :dim] = pts[:dim].T
    return torch.from_numpy(rec).to(torch.device("cuda", device))


def point_cloud_sdf_torch(spec, records, *, dim=3, slab=None, device=0, out=None):
    """sdf_point_cloud_3d / _2d on grid samples, device-resident: `records` from cloud_records(); returns a torch tensor
    of the slab's unsigned distances (current torch stream)."""
    import torch
    code = cabi.AB_F32 if records.dtype == torch.float32 else cabi.AB_F64
    x0, x1 = (0, spec.res[0]) if slab is None else slab
    n = (x1 - x0) * spec.res[1] * spec.res[2]
    buf = out if out is not None else torch.empty(n, dtype=records.dtype, device=records.device)
    if n == 0:
        return buf
    g = cabi.make_grid(spec.size, spec.res, (x0, x1))
    stream = torch.cuda.current_stream(records.device).cuda_stream
    cabi.check(cabi.lib().ab_nn_grid(records.data_ptr(), records.shape[0], dim, C.byref(g), code, buf.data_ptr(), device,
                                     C.c_void_p(stream)))
    return buf


# ---- from_sdf ------------------------------------------------------------------------------------------------------------------


def from_sdf(sdf_, co_resolution, *, dtype=None, device=0, normalize=True):
    """vector_functions.py:130-139: unit-spacing np.gradient of the reshaped field + batch_normalize, on the GPU.
    `sdf_` is a host array of N = prod(co_resolution) values; returns (dims, N)."""
    res = tuple(int(r) for r in np.asarray(co_resolution).reshape(-1))
    dims = len(res)
    if dims not in (2, 3):
        raise ValueError("co_resolution must have 2 or 3 entries")
    f = np.asarray(sdf_)
    if dtype is None:
        dtype = "f32" if f.dtype == np.float32 else "f64"
    code, npdt = _dtype(dtype)
    f = np.ascontiguousarray(f.reshape(-1), dtype=npdt)
    n = int(np.prod(res))
    if f.size != n:
        raise ValueError(f"Cannot reshape the pattern with shape {f.shape}")
    if any(r < 2 for r in res):
        raise ValueError("Shape of array too small to calculate a numerical gradient, at least 2 elements are "
                         "required.")
    lib = cabi.lib()
    d_f, d_o = C.c_void_p(), C.c_void_p()
    stride = (n + 7) // 8 * 8
    cabi.check(lib.ab_device_alloc(n * f.itemsize, device, C.byref(d_f)))
    try:
        cabi.check(lib.ab_device_alloc(dims * stride * f.itemsize, device, C.byref(d_o)))
        try:
            cabi.check(lib.ab_memcpy_h2d(d_f, f.ctypes.data, n * f.itemsize, device, None))
            g = cabi.make_grid((0.0, 0.0, 0.0), res + ((1,) if dims == 2 else ()))
            cabi.check(lib.ab_fd_gradient(d_f, 0, C.byref(g), dims, code, 1 if normalize else 0, d_o, stride, device,
                                          None))
            out = np.empty((dims, n), dtype=npdt)
            for r in range(dims):
                cabi.check(lib.ab_memcpy_d2h(out[r].ctypes.data, d_o.value + r * stride * f.itemsize, n * f.itemsize,
                                             device, None))
            cabi.check(lib.ab_stream_sync(device, None))
        finally:
            lib.ab_device_free(d_o, device)
    finally:
        lib.ab_device_free(d_f, device)
    return out


class _DevBuf:
    """A device allocation through the C ABI (freed on close / garbage collection)."""

    def __init__(self, nbytes, device):
        self.ptr = C.c_void_p()
        self.device = device
        cabi.check(cabi.lib().ab_device_alloc(int(nbytes), device, C.byref(self.ptr)))

    @classmethod
    def upload(cls, arr, device):
        arr = np.ascontiguousarray(arr)
        buf = cls(arr.nbytes, device)
        cabi.check(cabi.lib().ab_memcpy_h2d(buf.ptr, arr.ctypes.data, arr.nbytes, device, None))
        return buf

    def download(self, out, offset=0):
        cabi.check(cabi.lib().ab_memcpy_d2h(out.ctypes.data, C.c_void_p(self.ptr.value + offset), out.nbytes, self.device,
                                            None))

    def close(self):
        if self.ptr.value:
            cabi.lib().ab_device_free(self.ptr, self.device)
            self.ptr = C.c_void_p()

    __del__ = close


def _field_args(u, dtype):
    u = np.asarray(u)
    if u.ndim not in (2, 3):
        raise ValueError("the field must be a 2D or 3D array")
    if dtype is None:
        dtype = "f32" if u.dtype == np.float32 else "f64"
    code, npdt = _dtype(dtype)
    res = tuple(u.shape) + ((1,) if u.ndim == 2 else ())
    return np.ascontiguousarray(u, dtype=npdt), (C.c_uint32 * 3)(*res), code, npdt


def conv_averaging(u, kernel_size, iterations, *, dtype=None, device=0):
    """post_processing.py:552-599 on the GPU: `iterations` passes of a box filter (scipy.ndimage.convolve placement,
    mode 'reflect'). `u` is the field reshaped to the grid (smarter_reshape), `kernel_size` an int or one per axis."""
    if iterations == 0:
        return u
    f, res, code, npdt = _field_args(u, dtype)
    if isinstance(kernel_size, (int, np.integer)):
        kernel_size = (int(kernel_size),) * f.ndim
    kernel_size = tuple(int(k) for k in np.asarray(kernel_size).reshape(-1))
    if len(kernel_size) != f.ndim:
        raise ValueError("Dimension of the kernel and the field must match!")
    ks = (C.c_uint32 * 3)(*(kernel_size + ((1,) if f.ndim == 2 else ())))
    d_in, d_out = _DevBuf.upload(f, device), _DevBuf(f.nbytes, device)
    try:
        cabi.check(cabi.lib().ab_box_filter(d_in.ptr, res, ks, int(iterations), code, d_out.ptr, device, None))
        out = np.empty(f.shape, dtype=npdt)
        d_out.download(out)
        cabi.check(cabi.lib().ab_stream_sync(device, None))
    finally:
        d_in.close()
        d_out.close()
    return out


def conv_edge_detection(u, *, dtype=None, device=0):
    """post_processing.py:602-623 on the GPU: the 3x3 edge kernel over the first two axes."""
    f, res, code, npdt = _field_args(u, dtype)
    d_in, d_out = _DevBuf.upload(f, device), _DevBuf(f.nbytes, device)
    try:
        cabi.check(cabi.lib().ab_edge_filter(d_in.ptr, res, code, d_out.ptr, device, None))
        out = np.empty(f.shape, dtype=npdt)
        d_out.download(out)
        cabi.check(cabi.lib().ab_stream_sync(device, None))
    finally:
        d_in.close()
        d_out.close()
    return out


class VectorFieldFromSDF:
    """geom_vector.py:188-198 + the modifiers of ModifyVectorObject (modifications.py:1712-1971): the gradient field of
    an SDF (from_sdf) followed by the recorded elementwise modifiers, evaluated in two launches on the device
    (ab_fd_gradient, ab_vec_apply) without the (3, N) field visiting the host in between."""

    def __init__(self, co_resolution):
        self.co_resolution = co_resolution
        self._ops = []
        self._mod = []

    @property
    def modifications(self):
        return self._mod

    def _record(self, name, opcode, *operands):
        if len(self._ops) >= cabi.AB_MAX_VEC_OPS:
            raise ValueError(f"at most {cabi.AB_MAX_VEC_OPS} vector modifiers per field")
        self._mod.append(name)
        self._ops.append((opcode, operands))
        return self

    def add(self, second_field):
        return self._record("add", cabi.AB_VOP_ADD, ("any", second_field))

    def subtract(self, second_field):
        return self._record("subtract", cabi.AB_VOP_SUB, ("any", second_field))

    def rescale(self, second_field):
        return self._record("rescale", cabi.AB_VOP_RESCALE, ("scale", second_field))

    def rotate_phi(self, phi):
        return self._record("rotate_phi", cabi.AB_VOP_ROT_Z, ("angle", phi))

    def rotate_theta(self, theta):
        return self._record("rotate_theta", cabi.AB_VOP_ROT_THETA, ("angle", theta))

    def rotate_x(self, alpha):
        return self._record("rotate_x", cabi.AB_VOP_ROT_X, ("angle", alpha))

    def rotate_y(self, alpha):
        return self._record("rotate_y", cabi.AB_VOP_ROT_Y, ("angle", alpha))

    def rotate_z(self, alpha):
        return self._record("rotate_z", cabi.AB_VOP_ROT_Z, ("angle", alpha))

    def rotate_axis(self, axis, alpha):
        return self._record("rotate_axis", cabi.AB_VOP_ROT_AXIS, ("axis", axis), ("angle", alpha))

    def revolution_x(self, co):
        return self._record("revolution_x", cabi.AB_VOP_REVOLVE_X, ("coords", co))

    def revolution_y(self, co):
        return self._record("revolution_y", cabi.AB_VOP_REVOLVE_Y, ("coords", co))

    def revolution_z(self, co):
        return self._record("revolution_z", cabi.AB_VOP_REVOLVE_Z, ("coords", co))

    def normalize(self):
        return self._record("normalize", cabi.AB_VOP_NORMALIZE)

    # ---- evaluation ----
    @staticmethod
    def _operand(role, value, n, npdt, device, keep):
        """-> (kind, vec3, scalar, device pointer, stride) of one operand; arrays are uploaded as `npdt`."""
        v = np.asarray(value, dtype=np.float64)
        if role == "coords" or (role in ("any", "scale", "axis") and v.ndim == 2):
            if v.shape != (3, n):
                raise ValueError(f"a per-point vector operand must have shape (3, {n}), got {v.shape}")
            buf = _DevBuf.upload(v.astype(npdt), device)
            keep.append(buf)
            return cabi.AB_VK_VEC_ARRAY, (0.0, 0.0, 0.0), 0.0, buf.ptr.value, n
        if role in ("any", "axis") and v.size == 3 and n != 3:
            return cabi.AB_VK_VEC3, tuple(float(x) for x in v.reshape(3)), 0.0, None, 0
        if v.size == 1 and role != "axis":
            return cabi.AB_VK_SCALAR, (0.0, 0.0, 0.0), float(v.reshape(())), None, 0
        if v.shape == (n,) and role != "axis":
            buf = _DevBuf.upload(v.astype(npdt), device)
            keep.append(buf)
            return cabi.AB_VK_ARRAY, (0.0, 0.0, 0.0), 0.0, buf.ptr.value, n
        raise ValueError(f"operand of shape {v.shape} is not accepted here (field of {n} points)")

    def _run(self, sdf_, dtype, device, components=()):
        res = tuple(int(r) for r in np.asarray(self.co_resolution).reshape(-1))
        dims = len(res)
        f = np.asarray(sdf_)
        if dtype is None:
            dtype = "f32" if f.dtype == np.float32 else "f64"
        code, npdt = _dtype(dtype)
        n = int(np.prod(res))
        if self._ops and dims != 3:
            raise ValueError("vector modifiers need a 3D field")
        f = np.ascontiguousarray(f.reshape(-1), dtype=npdt)
        if f.size != n:
            raise ValueError(f"Cannot reshape the pattern with shape {f.shape}")
        if any(r < 2 for r in res):
            raise ValueError("Shape of array too small to calculate a numerical gradient, at least 2 elements are "
                             "required.")
        lib = cabi.lib()
        stride = (n + 7) // 8 * 8
        keep = []
        d_f, d_v = _DevBuf.upload(f, device), _DevBuf(3 * stride * f.itemsize, device)
        keep += [d_f, d_v]
        try:
            g = cabi.make_grid((0.0, 0.0, 0.0), res + ((1,) if dims == 2 else ()))
            cabi.check(lib.ab_fd_gradient(d_f.ptr, 0, C.byref(g), dims, code, 1, d_v.ptr, stride, device, None))
            if self._ops:
                ops = (cabi.ab_vec_op * len(self._ops))()
                for k, (opcode, operands) in enumerate(self._ops):
                    ops[k].opcode = opcode
                    for j, (role, value) in enumerate(operands):
                        kind, c, s, ptr, st = self._operand(role, value, n, npdt, device, keep)
                        if j == 0:
                            ops[k].kind0, ops[k].s0, ops[k].a0, ops[k].stride0 = kind, s, ptr, st
                            ops[k].c = (C.c_double * 3)(*c)
                        else:
                            ops[k].kind1, ops[k].s1, ops[k].a1, ops[k].stride1 = kind, s, ptr, st
                cabi.check(lib.ab_vec_apply(d_v.ptr, stride, n, ops, len(self._ops), code, device, None))
            out = {}
            if components:
                d_c = _DevBuf(n * f.itemsize, device)
                keep.append(d_c)
                ids = {"x": cabi.AB_VC_X, "y": cabi.AB_VC_Y, "z": cabi.AB_VC_Z, "phi": cabi.AB_VC_PHI,
                       "theta": cabi.AB_VC_THETA, "length": cabi.AB_VC_LENGTH}
                for name in components:
                    cabi.check(lib.ab_vec_component(d_v.ptr, stride, n, ids[name], code, d_c.ptr, device, None))
                    out[name] = np.empty(n, dtype=npdt)
                    d_c.download(out[name])
            else:
                vec = np.empty((dims, n), dtype=npdt)
                for r in range(dims):
                    d_v.download(vec[r], r * stride * f.itemsize)
                out["vec"] = vec
            cabi.check(lib.ab_stream_sync(device, None))
        finally:
            for b in keep:
                b.close()
        return out

    def create(self, sdf_, *, dtype=None, device=0):
        return self._run(sdf_, dtype, device)["vec"]

    propagate = create

    def x(self, sdf_, **kw):
        return self._component("x", sdf_, **kw)

    def y(self, sdf_, **kw):
        return self._component("y", sdf_, **kw)

    def z(self, sdf_, **kw):
        return self._component("z", sdf_, **kw)

    def phi(self, sdf_, **kw):
        return self._component("phi", sdf_, **kw)

    def theta(self, sdf_, **kw):
        return self._component("theta", sdf_, **kw)

    def length(self, sdf_, **kw):
        return self._component("length", sdf_, **kw)

    def _component(self, name, sdf_, *, dtype=None, device=0):
        return self._run(sdf_, dtype, device, components=(name,))[name]

    def components(self, sdf_, names=("x", "y", "z", "phi", "theta", "length"), *, dtype=None, device=0):
        """Several scalar maps from ONE evaluation of the pipeline (the reference re-evaluates it per call)."""
        return self._run(sdf_, dtype, device, components=tuple(names))


# ---- point clouds ----------------------------------------------------------------------------------------------------------------


def point_cloud_sdf(co, points, *, dim=3, dtype="f32", device=0, slab=None):
    """sdf_point_cloud_3d / sdf_point_cloud_2d (sdf_3D.py:283-286, sdf_2D.py:221-224): unsigned distance to the
    nearest cloud point with the dedicated tiled brute-force kernel."""
    code, npdt = _dtype(dtype)
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
    if pts.ndim != 2 or pts.shape[0] < dim:
        raise ValueError(f"points must have shape ({dim}, M)")
    m = pts.shape[1]
    lib = cabi.lib()
    spec = detect_grid(co)
    d_cloud, d_out, d_co = C.c_void_p(), C.c_void_p(), C.c_void_p()
    cabi.check(lib.ab_cloud_upload(pts.ctypes.data, m, dim, pts.shape[1], code, device, C.byref(d_cloud)))
    try:
        if spec is not None:
            x0, x1 = (0, spec.res[0]) if slab is None else slab
            n = (x1 - x0) * spec.res[1] * spec.res[2]
        else:
            co = np.ascontiguousarray(np.asarray(co, dtype=np.float64))
            n = co.shape[1]
        out = np.empty(n, dtype=npdt)
        if n == 0:
            return out
        cabi.check(lib.ab_device_alloc(n * out.itemsize, device, C.byref(d_out)))
        try:
            if spec is not None:
                g = cabi.make_grid(spec.size, spec.res, (x0, x1))
                cabi.check(lib.ab_nn_grid(d_cloud, m, dim, C.byref(g), code, d_out, device, None))
            else:
                rows = co.shape[0]
                cabi.check(lib.ab_device_alloc(rows * n * 8, device, C.byref(d_co)))
                cabi.check(lib.ab_memcpy_h2d(d_co, co.ctypes.data, rows * n * 8, device, None))
                cabi.check(lib.ab_nn_points(d_cloud, m, dim, d_co, cabi.AB_F64, n, n, code, d_out, device, None))
            cabi.check(lib.ab_memcpy_d2h(out.ctypes.data, d_out, n * out.itemsize, device, None))
            cabi.check(lib.ab_stream_sync(device, None))
        finally:
            lib.ab_device_free(d_out, device)
            if d_co.value:
                lib.ab_device_free(d_co, device)
    finally:
        lib.ab_device_free(d_cloud, device)
    return out


# ---- drop-in patch of an installed SPOMSO ---------------------------------------------------------------------------------------

_PATCHED = {}


def patch(dtype="f64", device=0):
    """Rebinds spomso.cores.geom.GenericGeometry.create/propagate to the GPU path. Trees that cannot be flattened
    raise NotImplementedError (there is no silent fallback)."""
    from spomso.cores import geom

    if "create" in _PATCHED:
        return
    _PATCHED["create"] = geom.GenericGeometry.create
    _PATCHED["propagate"] = geom.GenericGeometry.propagate

    def _create(self, co):
        return create(self, co, dtype=dtype, device=device)

    def _propagate(self, co, *parameters_):
        return create(self, co, dtype=dtype, device=device)

    _propagate.__name__ = "propagate"  # introspect.py recognises nested nodes by this name
    _create.__name__ = "create"
    geom.GenericGeometry.create = _create
    geom.GenericGeometry.propagate = _propagate


def unpatch():
    if "create" in _PATCHED:
        from spomso.cores import geom
        geom.GenericGeometry.create = _PATCHED.pop("create")
        geom.GenericGeometry.propagate = _PATCHED.pop("propagate")
