#!/usr/bin/env python
"""Builds, ahead of time, the program-compiled kernels (aegolius_b200/codegen.py) of every golden scenario, of the
BASELINE configurations and of the smoke / bench programs into aegolius_b200/jit/. Run by __graft_entry__.build() in the
build container (nvcc, no GPU); the binaries travel to the GPU box with the tree, so tests, smoke() and bench.py find
their kernels on disk (AB_JIT=cache never runs nvcc)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def items():
    import numpy as np
    import aegolius_b200 as ab
    from aegolius_b200 import workloads
    from aegolius_b200.program import Program
    out = []
    path = os.path.join(ROOT, "tests", "golden", "scenarios.npz")
    from conftest import GRADIENT_CASES
    grad_cases = set(GRADIENT_CASES)
    with np.load(path, allow_pickle=False) as d:
        for name in [str(n) for n in d["__names__"]]:
            keys = {k[len(name) + 1:]: d[k] for k in d.files if k.startswith(name + "/")}
            prog = Program.from_arrays(keys, prefix="prog_")
            res = tuple(int(r) for r in keys["res"])
            is2d = not res[2] > 1
            progs = [prog.pruned() if prog.stages else prog]
            for st in prog.stages:  # staged programs run their (pruned) prefixes too
                progs.append(prog.prefix(prog.stage_op_index(st)).pruned())
            for p in progs:
                for dt in ("f32", "f64"):
                    out.append((p, dt, None, is2d))
            if name in grad_cases:  # evaluated on point lists (flavour 0) with gradients
                for dt in ("f32", "f64"):
                    out.append((prog, dt, None, False))
                    out.append((prog, dt, "spatial", False))
                    if is2d:  # and on its own 2D grid (tests/test_gpu_jit.py::test_compiled_gradient_kernels_on_2d_grids)
                        out.append((prog, dt, "spatial", True))
    for build, is2d in ((workloads.build_c1, False), (workloads.build_c2, True), (workloads.build_c3, False)):
        prog = ab.flatten(build())
        for dt in ("f32", "f64"):
            for g in (None, "spatial"):
                out.append((prog, dt, g, is2d))
                out.append((prog, dt, g, False))
    # smoke() and the shallow-tree probes of bench.py
    s = ab.Sphere(1.0)
    s.move((0.5, 0, 0))
    b = ab.Box(1.5, 1.0, 0.8)
    b.rotate(np.pi / 5, (0, 0, 1))
    b.move((-0.4, 0.2, 0.1))
    u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=0.3)
    u.twist(0.5)
    sph = ab.Sphere(1.0)
    sph.move((0.3, 0.1, -0.2))
    for obj in (u, sph, ab.Sphere(1.0)):
        prog = ab.flatten(obj)
        for dt in ("f32", "f64"):
            for g in (None, "spatial"):
                out.append((prog, dt, g, False))
    # parameter tangents through grid-stencil stages (tests/test_gpu_stage_tangents.py, tools/stage_tangent_probe.py): the
    # pruned prefixes and the final program of each tangent program, in parameter mode and in value mode (differences)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import stage_tangent_probe
    import test_gpu_stage_tangents
    from aegolius_b200.engine import program_tangent
    staged = [(program_tangent(builder, p, k), len(res) == 2)
              for builder, p, _, res, _ in test_gpu_stage_tangents.BUILDERS.values() for k in range(len(p))]
    staged += [(prog, False) for _, prog, _ in stage_tangent_probe.programs()]
    for prog, is2d in staged:
        for q in [prog.pruned()] + [prog.prefix(prog.stage_op_index(st)).pruned() for st in prog.stages]:
            for dt in ("f32", "f64"):
                for g in (None, "param"):
                    out.append((q, dt, g, is2d))
    return out


FORWARD_TANGENT_CASES = ("c3_deep_tree", "c1_sphere_box_smooth_union")


def forward_tangent_sources():
    """fp64 field + gradient kernels built WITHOUT the pull-backs (adjoint=False) for two goldens: tests/test_gpu_jit.py
    checks that this build returns the interpreter's gradient to the bit (INTEGRATION.md: AB_JIT_ADJOINT=0)."""
    import numpy as np
    from aegolius_b200 import codegen
    from aegolius_b200.program import Program
    out = []
    with np.load(os.path.join(ROOT, "tests", "golden", "scenarios.npz"), allow_pickle=False) as d:
        for name in FORWARD_TANGENT_CASES:
            keys = {k[len(name) + 1:]: d[k] for k in d.files if k.startswith(name + "/")}
            prog = Program.from_arrays(keys, prefix="prog_")
            out.append(codegen.generate(codegen.signature(prog), "f64", "spatial", adjoint=False))
    return out


def main(verbose=True):
    from aegolius_b200 import codegen
    res = codegen.prebuild(items(), verbose=verbose)
    for src in forward_tangent_sources():
        codegen.build_source(src)
    return res


if __name__ == "__main__":
    main()
