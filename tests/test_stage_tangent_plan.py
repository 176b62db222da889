"""Parameter tangents of trees with grid-stencil stages, host side: the prefix and pruned programs the staged pipeline runs
carry the tangent of the argument pool, engine.program_tangent keeps the stages, and a parameter that changes a stage is
refused. No GPU needed."""
import numpy as np
import pytest

import aegolius_b200 as ab
from aegolius_b200 import opcodes as oc
from aegolius_b200.engine import program_tangent

R3 = (16, 12, 20)  # GridSpec -> 17 x 13 x 21


def _sphere_box_stage(r, x):
    """A sphere (radius r, moved by x) under a 3-box filter, smooth-united with a plain box: pruned() drops the subtree the
    stage replaced."""
    s = ab.Sphere(r)
    s.move((x, 0.1, -0.2))
    s.conv_averaging((3, 3, 3), 2, R3)
    b = ab.Box(1.0, 0.8, 0.6)
    u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=0.2)
    u.onion(0.1)
    return u


def _arg_of(prog, opcode):
    hit = np.nonzero(prog.ops["opcode"] == opcode)[0]
    assert hit.size == 1
    return int(prog.ops["arg"][hit[0]])


def test_prefix_and_pruned_keep_dargs():
    prog = ab.flatten(_sphere_box_stage(1.0, 0.3))
    assert prog.stages
    prog.dargs = np.random.default_rng(0).normal(size=prog.args.shape)
    k = prog.stage_op_index(prog.stages[0])
    pre = prog.prefix(k)
    assert pre.dargs is prog.dargs
    assert pre.pruned().dargs is prog.dargs
    pruned = prog.pruned()
    assert pruned.n_ops < prog.n_ops  # the sphere subtree under the stage is dead code in the final program
    assert pruned.dargs is prog.dargs
    assert np.array_equal(pruned.args, prog.args)  # offsets stay absolute: the same tangent vector applies


def test_program_tangent_of_a_staged_builder_keeps_stages_and_tangent():
    plain = ab.flatten(_sphere_box_stage(1.0, 0.3), fold_frames=False)
    for argnum, opcode in ((0, oc.P_SPHERE), (1, oc.TRANSLATE)):
        prog = program_tangent(_sphere_box_stage, (1.0, 0.3), argnum)
        assert prog.stages == plain.stages
        assert np.array_equal(prog.ops, plain.ops)
        off = _arg_of(prog, opcode)
        # d radius / d r = 1, d shift_x / d x = -1 (the point is moved, not the shape)
        assert abs(prog.dargs[off]) == pytest.approx(1.0, abs=1e-8)
        others = np.delete(prog.dargs, off)
        assert not others.any()  # nothing else depends on the parameter: exactly zero
        pre = prog.prefix(prog.stage_op_index(prog.stages[0])).pruned()
        assert pre.dargs is prog.dargs and pre.stages == []


def test_program_tangent_refuses_a_parameter_that_changes_a_stage():
    def builder(r, k):
        s = ab.Sphere(r)
        s.conv_averaging(3, int(round(k)), R3)
        return s

    # round(2.5 - h) = 2, round(2.5 + h) = 3: same op list, a different iteration count
    with pytest.raises(ValueError, match="stage changes"):
        program_tangent(builder, (1.0, 2.5), 1)
    prog = program_tangent(builder, (1.0, 2.5), 0)  # the radius leaves the stage alone
    assert prog.stages[0]["iterations"] == 2 and prog.dargs.any()
