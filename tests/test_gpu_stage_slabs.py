"""Trees with grid-stencil stages (conv_averaging / conv_edge_detection / signed used as modifications) on x-slabs: the
slabs of create(slab=) and create_torch(slab=) concatenate bit for bit to the whole-grid field, for the golden staged
scenarios and for seeded random staged trees; the signed mask and flags work slab by slab; the sharded paths on two GPUs
(tools/check_stage_slabs_multi_gpu.py). Both sides of every comparison run in this process under the same AB_JIT mode
(program-compiled fp32 kernels may differ from the interpreter in the last bits)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import golden_names, load_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED = [n for n in golden_names() if n.startswith("stencil_")]


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _splits(n0):
    from aegolius_b200.engine import slab_ranges
    out = [[(0, n0)], [(0, 1), (1, n0)], [(0, n0 - 1), (n0 - 1, n0)]]
    out += [slab_ranges(n0, p) for p in (2, 3, 5) if p <= n0]
    return out


def _check_slabs(prog, spec, dtype):
    import torch
    import aegolius_b200 as ab
    whole = ab.create(prog, spec, dtype=dtype)
    side = torch.cuda.Stream()
    for parts in _splits(spec.res[0]):
        got = np.concatenate([ab.create(prog, spec, dtype=dtype, slab=s) for s in parts])
        assert np.array_equal(_bits(got), _bits(whole)), (parts, np.nanmax(np.abs(got - whole)))
        with torch.cuda.stream(side):
            dev = [ab.create_torch(prog, spec, dtype=dtype, slab=s) for s in parts]
        side.synchronize()
        got = torch.cat(dev).cpu().numpy()
        assert np.array_equal(_bits(got), _bits(whole)), ("create_torch", parts)
    return whole


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("name", STAGED)
def test_golden_staged_scenarios_on_slabs(golden, name, dtype):
    import aegolius_b200 as ab
    c = load_case(golden, name)
    spec = ab.GridSpec(c["size"], c["res"])
    _check_slabs(c["prog"], spec, dtype)


def _random_tree(rng, ab):
    """A seeded staged tree on an odd-sized 2D or 3D grid: box stages (k 1..6 per axis, 1..3 iterations), edge stages,
    signed (3D), a stage of a stage, a stage on one branch of a union."""
    dims = 3 if rng.random() < 0.6 else 2
    res = tuple(int(r) for r in (rng.integers(2, 12, 3) * 2 + 1 if dims == 3 else rng.integers(4, 30, 2) * 2 + 1))
    size = (4.0,) * dims

    def leaf():
        if dims == 3:
            o = ab.Sphere(rng.uniform(0.6, 1.3)) if rng.random() < 0.5 else ab.Box(*rng.uniform(0.8, 2.0, 3))
            o.move(tuple(rng.uniform(-0.6, 0.6, 3)))
        else:
            o = ab.Circle(rng.uniform(0.6, 1.3)) if rng.random() < 0.5 else ab.Rectangle(*rng.uniform(0.8, 2.0, 2))
            o.move(tuple(rng.uniform(-0.6, 0.6, 2)) + (0.0,))
        return o

    def stage(o):
        r = rng.random()
        if dims == 3 and r < 0.25:
            o.boundary()
            o.signed(res)
        elif r < 0.4:
            o.conv_edge_detection(res)
        else:
            o.conv_averaging(tuple(int(k) for k in rng.integers(1, 7, dims)), int(rng.integers(1, 4)), res)

    a = leaf()
    stage(a)
    if rng.random() < 0.4:
        stage(a)  # a stage of a stage
    if rng.random() < 0.6:
        if rng.random() < 0.5:
            a = ab.CombineGeometry("UNION2").combine(a, leaf())
        else:
            a = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(a, leaf(), parameters=0.2)
        if rng.random() < 0.5:
            stage(a)
    a.onion(0.1)
    return a, ab.GridSpec(size, res)


@pytest.mark.parametrize("seed", range(30))
def test_random_staged_trees_on_slabs(seed):
    import aegolius_b200 as ab
    rng = np.random.default_rng(1000 + seed)
    tree, spec = _random_tree(rng, ab)
    prog = ab.flatten(tree)
    assert prog.stages
    for dtype in ("f32", "f64"):
        _check_slabs(prog, spec, dtype)


def _lib():
    from aegolius_b200 import cabi
    return cabi.lib()


def _u32(*v):
    return (C.c_uint32 * len(v))(*v)


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _pack(field, res, thr):
    n0, n1, n2 = res
    words = (n2 + 31) // 32
    b = np.zeros((n0, n1, words * 32), dtype=np.uint64)
    b[..., :n2] = field.reshape(res) < thr
    return (b.reshape(n0, n1, words, 32) << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32).reshape(-1)


def test_slab_masks_concatenate_to_the_whole_mask():
    import torch
    from aegolius_b200 import cabi
    from aegolius_b200.engine import slab_ranges
    res = (23, 17, 45)  # 45 z samples: two mask words per row, the second padded
    n0, pp, words = res[0], res[1] * res[2], (res[2] + 31) // 32
    f = torch.rand(n0 * pp, dtype=torch.float32, device="cuda")
    thr = 0.3
    whole = torch.empty(n0 * res[1] * words, dtype=torch.int32, device="cuda")
    flags = torch.zeros(2, dtype=torch.int32, device="cuda")
    cabi.check(_lib().ab_signed_mask(_ptr(f), _u32(*res), thr, cabi.AB_F32, _ptr(whole), _ptr(flags), 0, None))
    assert np.array_equal(whole.cpu().numpy().view(np.uint32), _pack(f.cpu().numpy(), res, np.float32(thr)))
    parts = []
    for x0, x1 in slab_ranges(n0, 4):
        m = torch.empty((x1 - x0) * res[1] * words, dtype=torch.int32, device="cuda")
        cabi.check(_lib().ab_signed_mask(C.c_void_p(f.data_ptr() + x0 * pp * 4), _u32(x1 - x0, *res[1:]), thr, cabi.AB_F32,
                                         _ptr(m), _ptr(flags), 0, None))
        parts.append(m)
    assert torch.equal(torch.cat(parts), whole)
    assert flags.tolist() == [0, 0]


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("poison", ["none", "negative", "negative+nan"])
def test_one_slab_flags_change_every_slab(dtype, poison):
    """A negative sample (pass-through) or a NaN (cancels the pass-through) in one slab only acts on every slab as on the
    whole field: slab-wise masks with shared flags, then ab_signed_field_slab, against ab_signed_field."""
    import torch
    from aegolius_b200 import cabi
    from aegolius_b200.engine import slab_ranges
    tdt, code, item = (torch.float32, cabi.AB_F32, 4) if dtype == "f32" else (torch.float64, cabi.AB_F64, 8)
    res = (19, 15, 37)
    n0, pp, words = res[0], res[1] * res[2], (res[2] + 31) // 32
    g = torch.Generator().manual_seed(7)
    x = torch.linspace(-1, 1, n0)[:, None, None]
    y = torch.linspace(-1, 1, res[1])[None, :, None]
    z = torch.linspace(-1, 1, res[2])[None, None, :]
    shell = ((x * x + y * y + z * z).sqrt() - 0.6).abs() + 0.02 * torch.rand(res, generator=g)
    f = shell.to(tdt).reshape(-1).cuda()
    if "negative" in poison:
        f[1 * pp + 3] = -0.5  # plane 1: first slab only
    if "nan" in poison:
        f[(n0 - 1) * pp + 5] = float("nan")  # last plane: last slab only
    thr = 2.0 / (res[2] - 1)
    whole = torch.empty_like(f)
    cabi.check(_lib().ab_signed_field(_ptr(f), _u32(*res), thr, code, _ptr(whole), 0, None))
    if poison == "negative":
        assert torch.equal(whole, f)
    else:
        assert (whole < 0).any()
    ranges = slab_ranges(n0, 3)
    mask = torch.empty(n0 * res[1] * words, dtype=torch.int32, device="cuda")
    flags = torch.zeros(2, dtype=torch.int32, device="cuda")
    for x0, x1 in ranges:
        cabi.check(_lib().ab_signed_mask(C.c_void_p(f.data_ptr() + x0 * pp * item), _u32(x1 - x0, *res[1:]), thr, code,
                                         C.c_void_p(mask.data_ptr() + x0 * res[1] * words * 4), _ptr(flags), 0, None))
    outs = []
    for x0, x1 in ranges:
        own = f[x0 * pp:x1 * pp].clone()  # only the slab's own planes of the field
        o = torch.empty_like(own)
        cabi.check(_lib().ab_signed_field_slab(_ptr(mask), _ptr(flags), _ptr(own), x0, _u32(*res), x0, x1, code, _ptr(o), 0,
                                               None))
        outs.append(o)
    got = torch.cat(outs)
    assert np.array_equal(_bits(got.cpu().numpy()), _bits(whole.cpu().numpy()))


def test_signed_tree_with_negative_samples_in_one_slab_passes_through_everywhere():
    import aegolius_b200 as ab
    s = ab.Sphere(0.3)
    s.move((-1.7, 0.0, 0.0))  # negative samples only near the x = -2 face
    s.signed((16, 12, 20))
    s0 = ab.Sphere(0.3)
    s0.move((-1.7, 0.0, 0.0))
    spec = ab.GridSpec((4, 4, 4), (16, 12, 20))
    prog = ab.flatten(s)
    whole = _check_slabs(prog, spec, "f64")
    assert np.array_equal(whole, ab.create(s0, spec, dtype="f64"))
    assert np.array_equal(ab.create(prog, spec, dtype="f64", slab=(10, 17)), whole[10 * 13 * 21:])


def test_staged_trees_still_reject_gradients_and_point_lists():
    import aegolius_b200 as ab
    s = ab.Sphere(1.0)
    s.conv_averaging(3, 1, (16, 12, 20))
    spec = ab.GridSpec((4, 4, 4), (16, 12, 20))
    with pytest.raises(NotImplementedError, match="without gradients"):
        ab.create(s, spec, grad="spatial")
    with pytest.raises(NotImplementedError, match="without gradients"):
        ab.create(s, spec, grad="spatial", slab=(0, 3))
    with pytest.raises(NotImplementedError, match="without gradients"):
        ab.create_torch(s, spec, grad="spatial")
    with pytest.raises(NotImplementedError, match="without gradients"):
        ab.create(s, np.random.default_rng(0).uniform(-1, 1, (3, 100)))


def test_sharded_staged_trees_on_two_devices():
    """tools/check_stage_slabs_multi_gpu.py under torch.distributed.run on 2 GPUs: evaluate_sharded(gather=True) of a
    box-stage tree and of a signed tree, and from_sdf_sharded of a staged tree, bit-identical to one GPU."""
    from aegolius_b200 import cabi
    if cabi.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tools", "check_stage_slabs_multi_gpu.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert '"ok": true' in r.stdout and '"ok": false' not in r.stdout, r.stdout[-3000:]
