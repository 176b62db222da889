"""Measures parameter tangents through grid-stencil stages on the GPU, in one call, fp32 at 513^3, for a tree shaped like
tests/scenarios.py's stencil_conv_averaging_tree3d (two box stages, one a stage of a stage under a smooth union) and for a
boundary-then-signed tree:

  1. the value-only staged evaluation (create_torch);
  2. one parameter's forward tangent (create_torch(grad="param"), what jacfwd(mode="dual") runs);
  3. one value_and_grad parameter step (the staged pipeline in parameter mode with the fused loss reduction);
  4. jacfwd(mode="fd") for one parameter: two fp64 staged evaluations and their difference.

Times are CUDA-event times of the device work on the current stream (median of --reps after a warm-up). Prints the
card's name and power limit first and one JSON line per measurement, and writes them to --out.

    python tools/stage_tangent_probe.py [--reps 10] [--out profiles/r04_stage_tangent_probe.jsonl]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

RES = 513
PARAMS = {"stencil_conv_averaging_tree3d": (1.1, 0.3), "boundary_signed": (0.9, -0.52)}


def averaged(r, w):
    import aegolius_b200 as ab
    s = ab.Sphere(r)
    s.move((0.4, -0.2, 0.3))
    s.conv_averaging((2, 3, 4), 2, (RES,) * 3)
    s.rounding(0.05)
    b = ab.Box(1.6, 1.0, 2.0)
    b.rotate(0.5, (0, 1, 0))
    u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=w)
    u.conv_averaging(3, 1, (RES,) * 3)
    return u


def signed(r, x):
    import aegolius_b200 as ab
    a = ab.Sphere(r)
    a.move((x, 0.13, 0.07))
    t = ab.Torus(1.0, 0.35)
    t.move((0.4, -0.2, 0.1))
    u = ab.CombineGeometry("UNION2").combine(a, t)
    u.boundary()
    u.signed((RES,) * 3)
    return u


BUILDERS = {"stencil_conv_averaging_tree3d": averaged, "boundary_signed": signed}


def programs():
    """(builder name, tangent program of parameter 0, the fp64 programs at theta -+ h) for prebuild_jit and the probe."""
    from aegolius_b200 import engine, flatten
    out = []
    for name, builder in BUILDERS.items():
        p = PARAMS[name]
        out.append((name, engine.program_tangent(builder, p, 0), flatten(builder(*p))))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_stage_tangent_probe.jsonl"))
    args = ap.parse_args()
    os.environ.setdefault("AB_JIT", "cache")  # kernels already on disk, no nvcc while timing
    import torch
    import aegolius_b200 as ab
    from aegolius_b200 import cabi, codegen, engine
    from stage_slab_probe import _time, card
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)
    emit({"card": card()})
    spec = ab.GridSpec((4.0, 4.0, 4.0), (RES,) * 3)
    for name, prog, value_prog in programs():
        builder, p = BUILDERS[name], PARAMS[name]
        target = engine.create_torch(value_prog, spec, dtype="f32") + 0.01
        accum = torch.zeros(2, dtype=torch.float64, device="cuda")
        h = 1e-6 * max(1.0, abs(p[0]))
        lo, hi = ab.flatten(builder(p[0] - h, *p[1:])), ab.flatten(builder(p[0] + h, *p[1:]))

        def fd():
            d = engine.create_torch(hi, spec, dtype="f64")
            d -= engine.create_torch(lo, spec, dtype="f64")
            d *= 1.0 / (2.0 * h)
        ms = {
            "value_only": _time(lambda: engine.create_torch(value_prog, spec, dtype="f32"), args.reps),
            "param_tangent": _time(lambda: engine.create_torch(prog, spec, dtype="f32", grad="param"), args.reps),
            "value_and_grad_step": _time(lambda: engine._staged_torch(prog, spec, cabi.AB_F32, None, None, 0, param=True,
                                                                      loss=(target, accum)), args.reps),
            "jacfwd_fd_f64": _time(fd, args.reps),
        }
        emit({"measure": "staged parameter tangent, device time of one parameter", "tree": name, "res": list(spec.res),
              "dtype": "f32 (fd: f64)", "jit": codegen.mode(), "stages": len(prog.stages),
              "ms": {k: round(v, 3) for k, v in ms.items()},
              "param_over_value": round(ms["param_tangent"] / ms["value_only"], 3),
              "vg_step_over_value": round(ms["value_and_grad_step"] / ms["value_only"], 3)})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.writelines(json.dumps(d) + "\n" for d in lines)


if __name__ == "__main__":
    main()
