"""Parameter tangents (grad="param", jacfwd(mode="dual"), value_and_grad) of trees with grid-stencil stages: every stage is
linear in its field, so the tangent goes through the same stencil and, for `signed`, the same sign pattern. Checked against
central differences of the fp64 oracle, against differences along random argument directions on the GPU, slab by slab bit
for bit, through the fused loss, compiled against interpreter, and sharded on two GPUs
(tools/check_stage_tangents_multi_gpu.py)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import interp_np

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAVE_NVCC = shutil.which("nvcc") is not None or os.path.exists("/usr/local/cuda/bin/nvcc")
R3 = (24, 20, 22)  # GridSpec -> 25 x 21 x 23 samples
R2 = (40, 36)      # -> 41 x 37
EDGE_TAPS = 16.0   # sum |taps| of the edge filter: centre 8, eight neighbours -1 (box filter and signed: 1)


def _sphere_box_stage(r, x):
    import aegolius_b200 as ab
    s = ab.Sphere(r)
    s.move((x, 0.113, -0.171))
    s.conv_averaging((3, 3, 3), 2, R3)
    s.onion(0.1)
    return s


def _circle_edge(x, y):
    import aegolius_b200 as ab
    c = ab.Circle(1.17)  # (its radius would be a constant shift: the edge filter of a constant is 0)
    c.move((x, y, 0.0))
    c.conv_edge_detection(R2)
    return c


def _box_signed(a, x):
    import aegolius_b200 as ab
    b = ab.Box(a, 1.23, 0.97)
    b.move((x, 0.071, -0.093))
    b.boundary()
    b.signed(R3)
    return b


def _stage_of_stage_union(r, w):
    import aegolius_b200 as ab
    s = ab.Sphere(r)
    s.move((-0.41, 0.13, 0.07))
    s.conv_averaging(3, 1, R3)
    s.conv_averaging((2, 3, 2), 1, R3)  # a stage of a stage
    b = ab.Box(1.1, 0.83, 1.37)
    b.move((0.37, -0.11, 0.05))
    u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=w)
    u.onion(0.05)
    return u


# name -> (builder, parameters, grid size, grid resolution, sum |taps| of its stencils)
BUILDERS = {
    "sphere_box_onion": (_sphere_box_stage, (1.05, 0.231), (4.0, 4.0, 4.0), R3, 1.0),
    "circle_edge_2d": (_circle_edge, (0.193, -0.137), (4.0, 4.0), R2, EDGE_TAPS),
    "box_boundary_signed": (_box_signed, (1.61, 0.157), (4.0, 4.0, 4.0), R3, 1.0),
    "stage_of_stage_smooth_union": (_stage_of_stage_union, (0.93, 0.31), (4.0, 4.0, 4.0), R3, 1.0),
}


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _spec(name):
    import aegolius_b200 as ab
    _, _, size, res, _ = BUILDERS[name]
    return ab.GridSpec(size, res)


@pytest.mark.parametrize("name", list(BUILDERS))
def test_staged_jacfwd_matches_oracle_differences(name):
    import aegolius_b200 as ab
    builder, p, _, _, taps = BUILDERS[name]
    spec = _spec(name)
    for k in range(len(p)):
        dual64 = ab.jacfwd(builder, argnums=k, mode="dual", dtype="f64")(spec, *p)
        dual32 = ab.jacfwd(builder, argnums=k, mode="dual", dtype="f32")(spec, *p)
        fd = ab.jacfwd(builder, argnums=k, mode="fd")(spec, *p)
        h = 1e-5
        lo, hi = list(p), list(p)
        lo[k] -= h
        hi[k] += h
        exp = (interp_np.run_grid(ab.flatten(builder(*hi)), spec.size, spec.res)
               - interp_np.run_grid(ab.flatten(builder(*lo)), spec.size, spec.res)) / (2 * h)
        assert np.abs(exp).max() > 1e-2  # the parameter reaches the field
        kd = np.abs(exp - dual64) > 1e-3 * taps  # samples whose stencil holds a branch flip inside the difference step
        assert kd.mean() < 0.02, (name, k, kd.mean())
        assert np.max(np.abs(exp - dual64)[~kd]) < 1e-5 * taps, (name, k)
        assert np.max(np.abs(dual32 - dual64)[~kd]) < 2e-3 * taps, (name, k)
        kf = np.abs(exp - fd) > 1e-3 * taps
        assert kf.mean() < 0.02
        assert np.max(np.abs(exp - fd)[~kf]) < 1e-5 * taps


def _random_tree(seed):
    import aegolius_b200 as ab
    from test_gpu_stage_slabs import _random_tree as make
    rng = np.random.default_rng(1000 + seed)
    tree, spec = make(rng, ab)
    prog = ab.flatten(tree)
    assert prog.stages
    prog.dargs = 0.1 * np.random.default_rng(seed).normal(size=prog.args.shape)  # no table arguments in these trees
    return prog, spec


def _taps(prog):
    return EDGE_TAPS ** sum(st["kind"] == 1 for st in prog.stages)


@pytest.mark.parametrize("seed", range(30))
def test_random_direction_tangent_matches_gpu_differences(seed):
    import aegolius_b200 as ab
    from aegolius_b200.program import Program
    prog, spec = _random_tree(seed)
    _, tangent = ab.create(prog, spec, dtype="f64", grad="param")
    h = 1e-6

    def at(t):
        return ab.create(Program(prog.ops, prog.args + t * prog.dargs, prog.blobs, prog.n_pslots, prog.n_vslots,
                                 prog.stages), spec, dtype="f64")
    exp = (at(h) - at(-h)) / (2 * h)
    taps = _taps(prog)
    kd = np.abs(exp - tangent[0]) > 1e-3 * taps
    assert kd.mean() < 0.02, kd.mean()
    assert np.max(np.abs(exp - tangent[0])[~kd]) < 1e-5 * taps


def _splits(n0):
    from aegolius_b200.engine import slab_ranges
    out = [[(0, n0)], [(0, 1), (1, n0)], [(0, n0 - 1), (n0 - 1, n0)]]
    out += [slab_ranges(n0, p) for p in (2, 3, 5) if p <= n0]
    return out


def _check_tangent_slabs(prog, spec, dtype):
    import torch
    import aegolius_b200 as ab
    field, tangent = ab.create(prog, spec, dtype=dtype, grad="param")
    side = torch.cuda.Stream()
    for parts in _splits(spec.res[0]):
        got = [ab.create(prog, spec, dtype=dtype, grad="param", slab=s) for s in parts]
        assert np.array_equal(_bits(np.concatenate([f for f, _ in got])), _bits(field)), parts
        assert np.array_equal(_bits(np.concatenate([t[0] for _, t in got])), _bits(tangent[0])), parts
        with torch.cuda.stream(side):
            dev = [ab.create_torch(prog, spec, dtype=dtype, grad="param", slab=s) for s in parts]
        side.synchronize()
        assert np.array_equal(_bits(torch.cat([f for f, _ in dev]).cpu().numpy()), _bits(field)), ("create_torch", parts)
        assert np.array_equal(_bits(torch.cat([t[0] for _, t in dev]).cpu().numpy()), _bits(tangent[0])), ("torch", parts)
    return field, tangent


@pytest.mark.parametrize("seed", range(30))
def test_random_staged_tangents_on_slabs(seed):
    prog, spec = _random_tree(seed)
    for dtype in ("f32", "f64"):
        _check_tangent_slabs(prog, spec, dtype)


def test_signed_pass_through_carries_the_tangent_unchanged():
    """A sphere whose negative samples lie only near the x = -2 face: `signed` passes field and tangent through, on
    every slab, so the tangent equals that of the tree without `signed`."""
    import aegolius_b200 as ab
    from aegolius_b200.engine import program_tangent
    res = (16, 12, 20)

    def tree(r, x, signed):
        s = ab.Sphere(r)
        s.move((x, 0.0, 0.0))
        if signed:
            s.signed(res)
        return s

    spec = ab.GridSpec((4, 4, 4), res)
    for k in range(2):
        prog = program_tangent(lambda r, x: tree(r, x, True), (0.3, -1.7), k)
        plain = program_tangent(lambda r, x: tree(r, x, False), (0.3, -1.7), k)
        field, tangent = _check_tangent_slabs(prog, spec, "f64")
        f0, t0 = ab.create(plain, spec, dtype="f64", grad="param")
        assert np.array_equal(_bits(field), _bits(f0)) and np.array_equal(_bits(tangent), _bits(t0))
        assert np.abs(t0).max() > 0.5


def test_staged_value_and_grad_fused_unfused_differences_and_adam():
    import aegolius_b200 as ab
    builder, p, _, _, _ = BUILDERS["stage_of_stage_smooth_union"]
    spec = _spec("stage_of_stage_smooth_union")
    rng = np.random.default_rng(4)
    target64 = interp_np.run_grid(ab.flatten(builder(1.1, 0.22)), spec.size, spec.res) + 0.01 * rng.normal(size=spec.n_points)
    exp_loss = float(np.sum((interp_np.run_grid(ab.flatten(builder(*p)), spec.size, spec.res) - target64) ** 2))
    for dt, rtol in (("f64", 1e-11), ("f32", 2e-5)):
        loss, grads = ab.value_and_grad(builder, spec, target64, dtype=dt)(p)
        assert abs(loss - exp_loss) <= rtol * exp_loss
        loss_u, grads_u = ab.value_and_grad(builder, spec, target64, dtype=dt, post=lambda f, d: (f, d))(p)
        assert abs(loss - loss_u) <= 10 * rtol * abs(loss_u)
        assert np.allclose(grads, grads_u, rtol=50 * rtol, atol=50 * rtol * np.max(np.abs(grads_u)))
    vg = ab.value_and_grad(builder, spec, target64, dtype="f64")
    loss0, g0 = vg(p)
    h = 1e-5
    fd = np.array([(vg(np.add(p, h * e))[0] - vg(np.add(p, -h * e))[0]) / (2 * h) for e in np.eye(len(p))])
    assert np.allclose(g0, fd, rtol=1e-3, atol=1e-3 * np.abs(fd).max()), (g0, fd)
    params, m, v, lr = np.array(p, dtype=np.float64), np.zeros(len(p)), np.zeros(len(p)), 0.02
    for it in range(1, 9):
        loss, g = vg(params)
        m = 0.9 * m + 0.1 * g
        v = 0.999 * v + 0.001 * g * g
        params = params - lr * (m / (1 - 0.9 ** it)) / (np.sqrt(v / (1 - 0.999 ** it)) + 1e-8)
    assert vg(params)[0] < 0.8 * loss0
    with pytest.raises(NotImplementedError, match="specialized"):
        ab.value_and_grad(builder, spec, target64, specialized=True)(p)


def test_staged_trees_reject_spatial_gradients_with_the_new_message():
    import aegolius_b200 as ab
    builder, p, _, _, _ = BUILDERS["sphere_box_onion"]
    spec = _spec("sphere_box_onion")
    for call in (lambda: ab.create(builder(*p), spec, grad="spatial"),
                 lambda: ab.create_torch(builder(*p), spec, grad="spatial"),
                 lambda: ab.create(builder(*p), np.zeros((3, 10)), grad="param")):
        with pytest.raises(NotImplementedError, match="without gradients in x, y, z.*grad='param'"):
            call()


def test_compiled_staged_tangent_matches_the_interpreter():
    import torch
    import aegolius_b200 as ab
    from aegolius_b200 import cabi, codegen as cg
    from aegolius_b200.engine import program_tangent
    builder, p, _, _, _ = BUILDERS["stage_of_stage_smooth_union"]
    spec = _spec("stage_of_stage_smooth_union")
    prog = program_tangent(builder, p, 1)
    final = prog.pruned()
    assert cg.ensure(final, "f64", "param", how="sync" if HAVE_NVCC else None) or not HAVE_NVCC
    lib = cabi.lib()
    h0 = lib.ab_prog_hits()
    fa, da = ab.create(prog, spec, dtype="f64", grad="param")
    if HAVE_NVCC:
        assert lib.ab_prog_hits() > h0
    old = lib.ab_prog_enable(0)
    try:
        fb, db = ab.create(prog, spec, dtype="f64", grad="param")
    finally:
        lib.ab_prog_enable(old)
    assert np.array_equal(_bits(fa), _bits(fb)) and np.array_equal(_bits(da), _bits(db))
    target = torch.as_tensor(fa + 0.01, device="cuda")
    f = ab.value_and_grad(builder, spec, target, dtype="f64")
    la, ga = f(p)
    old = lib.ab_prog_enable(0)
    try:
        lb, gb = f(p)
    finally:
        lib.ab_prog_enable(old)
    assert abs(la - lb) <= 1e-12 * abs(lb) and np.allclose(ga, gb, rtol=1e-12, atol=1e-14)


def test_sharded_staged_tangents_on_two_devices():
    """tools/check_stage_tangents_multi_gpu.py under torch.distributed.run on 2 GPUs: evaluate_sharded(grad="param",
    gather=True) of a box-stage tree and of a signed tree, bit-identical to one GPU."""
    from aegolius_b200 import cabi
    if cabi.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tools", "check_stage_tangents_multi_gpu.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert '"ok": true' in r.stdout and '"ok": false' not in r.stdout, r.stdout[-3000:]
