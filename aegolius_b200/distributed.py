"""Multi-GPU plumbing: one process per GPU (torch.distributed, NCCL over NVLink/NVSwitch; gloo on CPU for tests).

The path shards with NO data-path collective: every grid point depends only on its own coordinates and the (tiny,
replicated) program, so each rank evaluates one contiguous slab of ix planes — contiguous in SPOMSO's memory layout,
where x is the slowest axis (helper_functions.py:72-75, SURVEY §8e). What this module adds around that:

  * evaluate_sharded        the slab of a geometry tree (field, optionally the analytic gradient);
  * point_cloud_sharded     point cloud -> distance: the cloud is replicated with ONE broadcast (16 B per point), the query
                            grid is sharded like any other field (sdf_3D.py:283-286);
  * from_sdf_sharded        from_sdf (vector_functions.py:130-139) per slab: the two halo planes np.gradient's central
                            stencil needs are RECOMPUTED locally (2 extra planes per rank) instead of exchanged;
  * gather_field / gather_rows   OPTIONAL assembly of the full field on every rank, written in place: one
                            all_gather_into_tensor straight into the result when the slabs are equal, a group of
                            broadcasts into views of the result when they are not (1025 planes over 8 ranks = 129, 128 ...);
                            no staging buffers, no re-copy;
  * evaluate_multicast      the B200-native assembly: the result lives in a symmetric allocation mapped by all ranks, and
                            the evaluation kernel itself stores through the NVLS multicast address (multimem.st), so every
                            value lands in every GPU's copy while it is being computed — no gather pass at all.

Assembly is timed separately from the throughput (bench.py, tools/check_multi_gpu.py).
"""
from __future__ import annotations

import os

import numpy as np

from .engine import slab_ranges


def rank_slab(n_planes: int, rank: int, world: int):
    """(x0, x1) of `rank`: np.array_split(range(n_planes), world)[rank] as a half-open range."""
    return slab_ranges(n_planes, world)[rank]


def padded_slab_points(spec, world: int) -> int:
    """Points of the largest slab (1025 planes over 8 ranks = 129, 128, ...)."""
    per_plane = spec.res[1] * spec.res[2]
    return max(x1 - x0 for x0, x1 in slab_ranges(spec.res[0], world)) * per_plane


def aligned_slab_ranges(spec, world: int, itemsize: int = 4):
    """slab_ranges with every slab START moved down to a plane whose first sample is 16-byte aligned in the assembled field
    (1025^2 samples per plane are odd, so only every 4th plane of an fp32 field is): the slabs then keep their 128-bit
    stores when they are written into one shared buffer (evaluate_multicast)."""
    import math
    per_plane = spec.res[1] * spec.res[2]
    q = 16 // math.gcd(16, per_plane * itemsize)  # planes between aligned starts
    starts = [x0 - x0 % q for x0, _ in slab_ranges(spec.res[0], world)]
    return [(s, e) for s, e in zip(starts, starts[1:] + [spec.res[0]])]


def _world(group=None):
    import torch.distributed as dist
    if not dist.is_initialized():
        return 1, 0
    return dist.get_world_size(group), dist.get_rank(group)


def gather_field(local, spec, group=None, out=None):
    """The per-rank slabs -> the full flat field (N,) on every rank, assembled IN PLACE.

    `local` is this rank's slab as a 1-D torch tensor (CUDA with NCCL, CPU with gloo). Equal slabs: one
    all_gather_into_tensor whose output IS the result. Unequal slabs on NCCL: all_gather into views of the result
    (ProcessGroupNCCL runs it as one group of broadcasts, each landing in its view). gloo needs equal sizes, so the CPU
    path pads (tests only)."""
    import torch
    import torch.distributed as dist
    world, rank = _world(group)
    per_plane = spec.res[1] * spec.res[2]
    ranges = slab_ranges(spec.res[0], world)
    n_local = (ranges[rank][1] - ranges[rank][0]) * per_plane
    if local.numel() != n_local:
        raise ValueError(f"rank {rank}: slab has {local.numel()} points, expected {n_local}")
    if out is None:
        out = torch.empty(spec.n_points, dtype=local.dtype, device=local.device)
    elif out.numel() != spec.n_points or out.dtype != local.dtype or not out.is_contiguous():
        raise ValueError("out= must be a contiguous tensor of the whole field")
    if world == 1:
        out.copy_(local)
        return out
    local = local.contiguous()
    if len({x1 - x0 for x0, x1 in ranges}) == 1:
        dist.all_gather_into_tensor(out, local, group=group)
        return out
    views = [out[x0 * per_plane:x1 * per_plane] for x0, x1 in ranges]
    if local.is_cuda:
        dist.all_gather(views, local, group=group)
        return out
    pad = padded_slab_points(spec, world)
    send = torch.zeros(pad, dtype=local.dtype)
    send[:n_local] = local
    recv = torch.empty(pad * world, dtype=local.dtype)
    dist.all_gather_into_tensor(recv, send, group=group)
    for r, v in enumerate(views):
        v.copy_(recv[r * pad:r * pad + v.numel()])
    return out


def gather_rows(local_rows, spec, group=None):
    """(K, n_local) per-rank rows (a gradient slab) -> (K, N) on every rank, row by row in place."""
    import torch
    out = torch.empty((local_rows.shape[0], spec.n_points), dtype=local_rows.dtype, device=local_rows.device)
    for k in range(local_rows.shape[0]):
        gather_field(local_rows[k], spec, group, out=out[k])
    return out


class _MaskLayout:
    """The plane layout gather_field assembles: n0 planes of `per_plane` values."""

    def __init__(self, n0, per_plane):
        self.res = (n0, per_plane, 1)
        self.n_points = n0 * per_plane


class MaskGather:
    """The boundary mask of a `signed` stage covers whole columns along x, so a rank cannot sign its slab from its own
    planes alone. With this passed as engine.create_torch(mask_gather=), each rank packs the mask of its own slab
    (`planes`, 1 bit per sample), the slabs are all-gathered in place (gather_field) and the negative / NaN flags are
    max-reduced: 1/32 of a fp32 field crosses the ranks instead of every rank evaluating the whole grid."""

    def __init__(self, spec, group=None):
        world, rank = _world(group)
        self.group = group
        self.n0 = spec.res[0]
        self.planes = rank_slab(self.n0, rank, world)

    def __call__(self, local_words, words_per_plane, flags):
        import torch.distributed as dist
        dist.all_reduce(flags, op=dist.ReduceOp.MAX, group=self.group)
        return gather_field(local_words, _MaskLayout(self.n0, words_per_plane), self.group)


def _mask_gather(obj, spec, group):
    from . import engine
    world, _ = _world(group)
    return MaskGather(spec, group) if world > 1 and engine._as_program(obj).stages else None


def evaluate_sharded(obj, spec, *, dtype="f32", grad=None, group=None, gather=False):
    """Evaluates this rank's slab on its GPU (device = LOCAL_RANK). gather=True assembles the full field — and, with
    grad=, the full (K, N) gradient — on every rank. Trees with grid-stencil stages recompute the halo their stencils need
    on every rank (Program.stage_plan); their `signed` masks are all-gathered (MaskGather)."""
    from . import engine
    world, rank = _world(group)
    device = int(os.environ.get("LOCAL_RANK", "0"))
    slab = rank_slab(spec.res[0], rank, world)
    obj = engine._as_program(obj)
    res = engine.create_torch(obj, spec, dtype=dtype, grad=grad, device=device, slab=slab,
                              mask_gather=_mask_gather(obj, spec, group))
    if not gather or world == 1:
        return res
    if grad:
        return gather_field(res[0], spec, group), gather_rows(res[1], spec, group)
    return gather_field(res, spec, group)


def broadcast_cloud(points, *, dim=3, dtype="f32", src=0, group=None):
    """The cloud as (M, 4) device records on every rank: rank `src` packs and uploads its (dim, M) array, the others
    receive it with one broadcast (the count first). `points` may be None on the other ranks."""
    import torch
    import torch.distributed as dist
    from . import engine
    world, rank = _world(group)
    device = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1:
        return engine.cloud_records(points, dim, dtype, device)
    dev = torch.device("cuda", device)
    tdt = torch.float32 if engine._dtype(dtype)[0] == 0 else torch.float64
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    rec = None
    if rank == src:
        rec = engine.cloud_records(points, dim, dtype, device)
        count[0] = rec.shape[0]
    dist.broadcast(count, src, group=group)
    if rank != src:
        rec = torch.empty((int(count[0]), 4), dtype=tdt, device=dev)
    dist.broadcast(rec, src, group=group)
    return rec


def point_cloud_sharded(spec, points, *, dim=3, dtype="f32", src=0, group=None, gather=False, records=None):
    """sdf_point_cloud_3d / _2d on this rank's slab of the query grid; the cloud is replicated (broadcast_cloud), nothing
    else crosses the ranks. Pass `records` to reuse an already replicated cloud."""
    from . import engine
    world, rank = _world(group)
    device = int(os.environ.get("LOCAL_RANK", "0"))
    if records is None:
        records = broadcast_cloud(points, dim=dim, dtype=dtype, src=src, group=group)
    local = engine.point_cloud_sdf_torch(spec, records, dim=dim, slab=rank_slab(spec.res[0], rank, world), device=device)
    return gather_field(local, spec, group) if gather and world > 1 else local


def from_sdf_sharded(obj, spec, *, dtype="f32", group=None, normalize=True, smooth=None):
    """from_sdf of the field of `obj` on this rank's slab: the field is evaluated on the slab plus one halo plane on each
    side that exists in the grid (recomputed, not exchanged), then np.gradient's stencil runs on the slab. Returns
    (field slab, (dims, n_slab) vectors); the slabs' vectors concatenate bit-identically to the whole-grid from_sdf."""
    from . import engine
    world, rank = _world(group)
    device = int(os.environ.get("LOCAL_RANK", "0"))
    x0, x1 = rank_slab(spec.res[0], rank, world)
    lo, hi = max(x0 - 1, 0), min(x1 + 1, spec.res[0])
    per_plane = spec.res[1] * spec.res[2]
    obj = engine._as_program(obj)
    halo = engine.create_torch(obj, spec, dtype=dtype, device=device, slab=(lo, hi), mask_gather=_mask_gather(obj, spec, group))
    res = spec.res if spec.res[2] > 1 or float(spec.size[2]) != 0.0 else spec.res[:2]
    vec = engine.from_sdf_torch(halo, res, slab=(x0, x1), field_plane0=lo, normalize=normalize, device=device)
    return halo[(x0 - lo) * per_plane:(x1 - lo) * per_plane], vec


# ---- assembly by the evaluation kernel itself: NVLS multicast stores ---------------------------------------------------------------

class MulticastField:
    """A field (N,) [+ gradient (3, stride)] in a symmetric allocation mapped by every rank of the node, with its NVLS
    multicast address. evaluate_multicast() fills it on ALL ranks at once: each rank's kernel stores its slab with
    multimem.st. `.field` / `.grad` are this rank's ordinary tensors over its own copy."""

    def __init__(self, spec, dtype="f32", grad=False, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        from . import engine
        self.spec = spec
        self.group = group if group is not None else dist.group.WORLD
        device = int(os.environ.get("LOCAL_RANK", "0"))
        tdt = torch.float32 if engine._dtype(dtype)[0] == 0 else torch.float64
        n = spec.n_points
        self.stride = (n + 7) // 8 * 8
        total = self.stride * (4 if grad else 1)
        self.buf = symm.empty(total, dtype=tdt, device=torch.device("cuda", device))
        self.handle = symm.rendezvous(self.buf, self.group.group_name)
        self.mc_ptr = int(getattr(self.handle, "multicast_ptr", 0) or 0)
        if not self.mc_ptr:
            raise RuntimeError("this node offers no NVLS multicast mapping for symmetric memory (needs NVSwitch and a "
                               "driver with multicast support); use gather_field instead")
        self.field = self.buf[:n]
        self.grad = self.buf[self.stride:].view(3, self.stride)[:, :n] if grad else None
        self.itemsize = self.buf.element_size()

    def barrier(self):
        """All ranks' stores are complete and visible."""
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize(self.buf.device)
        dist.barrier(self.group)


def evaluate_multicast(obj, mc: MulticastField, *, grad=None):
    """Evaluates this rank's slab and stores it through the multicast address: when every rank has returned from
    mc.barrier(), mc.field (and mc.grad) hold the WHOLE grid on every GPU. No gather pass, no staging: the NVSwitch
    replicates each 16-byte store. Needs the program-compiled kernel with the multicast store path (built on first use)."""
    import ctypes as C
    import torch
    from . import cabi, codegen, engine
    prog = engine._as_program(obj)
    spec = mc.spec
    world, rank = _world(mc.group)
    device = mc.buf.device.index
    x0, x1 = aligned_slab_ranges(spec, world, mc.itemsize)[rank]
    per_plane = spec.res[1] * spec.res[2]
    dt = "f32" if mc.buf.dtype == torch.float32 else "f64"
    if x1 <= x0:
        return
    gmode, rows = engine._grad_mode(grad)
    if rows and mc.grad is None:
        raise ValueError("the MulticastField was created without a gradient")
    if not codegen.ensure(prog, dt, grad, is2d=engine._is_2d(spec), how="sync", multicast=True):
        raise RuntimeError("could not build the multicast-store kernel for this program")
    off = x0 * per_plane * mc.itemsize
    g = cabi.make_grid(spec.size, spec.res, (x0, x1))
    cp = cabi.CProgram(prog)
    stream = torch.cuda.current_stream(mc.buf.device).cuda_stream
    gptr = mc.mc_ptr + mc.stride * mc.itemsize + off if rows else None
    cabi.check(cabi.lib().ab_eval_grid_multicast(cp.ref(), C.byref(g), cabi.AB_F32 if dt == "f32" else cabi.AB_F64, gmode,
                                                 C.c_void_p(mc.mc_ptr + off), C.c_void_p(gptr) if gptr else None, mc.stride,
                                                 device, C.c_void_p(stream)))
