"""Program.stage_plan: the plane ranges on which each grid-stencil stage is evaluated and must be exact when a tree with
stages is evaluated on an x-slab. Every expected range below is derived by hand in the comment next to it."""
import numpy as np
import pytest

import aegolius_b200 as ab
from aegolius_b200 import opcodes as oc
from aegolius_b200.program import OP_DTYPE, Program

R3 = (16, 12, 20)          # GridSpec -> 17 x 13 x 21
RES3 = (17, 13, 21)
R2 = (64, 48)              # -> 65 x 49
RES2 = (65, 49, 1)


def _box(k, it, res=R3):
    s = ab.Sphere(1.0)
    s.conv_averaging(k, it, res)
    return ab.flatten(s)


def _ranges(plan):
    return [(ev, valid) for _, ev, valid in plan]


@pytest.mark.parametrize("k,it,expected", [
    (5, 2, (2, 13)),   # odd: 2 * 2 planes below 6, 2 * 2 above 9
    (3, 3, (3, 12)),   # odd: 3 * 1 below, 3 * 1 above
    (4, 3, (3, 15)),   # even: 3 * ((4 - 1) // 2) = 3 below, 3 * (4 // 2) = 6 above
    (2, 1, (6, 10)),   # even: 0 below, 1 above
    (6, 1, (4, 12)),   # even: 2 below, 3 above
    (1, 3, (6, 9)),    # k = 1: no halo
])
def test_box_halo_follows_the_tap_placement(k, it, expected):
    plan, final = _box(k, it).stage_plan(RES3, (6, 9))
    assert final == (6, 9)
    assert _ranges(plan) == [(expected, (6, 9))]


@pytest.mark.parametrize("slab,expected", [
    ((0, 3), (0, 7)),     # 0 - 4 clips to the face, 3 + 4 = 7
    ((14, 17), (10, 17)),  # 14 - 4 = 10, 17 + 4 clips
    ((0, 1), (0, 5)),     # one plane at the lower face
    ((16, 17), (12, 17)),  # one plane at the upper face
    ((8, 9), (4, 13)),    # one plane inside
    ((0, 17), (0, 17)),   # the whole grid
])
def test_box_ranges_clip_at_the_faces(slab, expected):
    plan, _ = _box(5, 2).stage_plan(RES3, slab)  # 2 iterations of k = 5: 4 planes each side
    assert _ranges(plan) == [(expected, slab)]


def test_kernel_wider_than_the_axis_uses_the_whole_axis():
    res = (9, 13, 21)
    wide = _box(10, 1, (8, 12, 20))   # k = 10 > 9 planes: reflection can wrap past both faces
    fits = _box(9, 1, (8, 12, 20))    # k = 9: 4 planes each side, clipped at 0
    assert _ranges(wide.stage_plan(res, (0, 1))[0]) == [((0, 9), (0, 1))]
    assert _ranges(fits.stage_plan(res, (0, 1))[0]) == [((0, 5), (0, 1))]


def test_edge_filter_reads_one_plane_each_side_in_2d_and_3d():
    c = ab.Circle(1.0)
    c.conv_edge_detection(R2)
    plan, _ = ab.flatten(c).stage_plan(RES2, (10, 20))
    assert _ranges(plan) == [((9, 21), (10, 20))]
    plan, _ = ab.flatten(c).stage_plan(RES2, (0, 1))
    assert _ranges(plan) == [((0, 2), (0, 1))]
    s = ab.Sphere(1.0)
    s.conv_edge_detection(R3)
    plan, _ = ab.flatten(s).stage_plan(RES3, (16, 17))
    assert _ranges(plan) == [((15, 17), (16, 17))]


def test_box_on_a_2d_grid_uses_the_x_kernel_size():
    c = ab.Circle(1.0)
    c.conv_averaging((5, 2), 4, R2)  # x kernel 5, 4 iterations: 8 planes each side; the y kernel does not matter
    plan, _ = ab.flatten(c).stage_plan(RES2, (30, 35))
    assert _ranges(plan) == [((22, 43), (30, 35))]


def test_a_stage_feeding_a_later_prefix_composes_the_halos():
    s = ab.Sphere(1.0)
    s.conv_averaging(3, 1, R3)   # stage A: 1 plane each side
    s.conv_averaging(5, 1, R3)   # stage B reads A: 2 planes each side
    plan, _ = ab.flatten(s).stage_plan(RES3, (6, 9))
    # B is read by the final program on (6, 9) -> evaluated on (4, 11); A must be exact there -> evaluated on (3, 12)
    assert _ranges(plan) == [((3, 12), (4, 11)), ((4, 11), (6, 9))]


def _synthetic(middle):
    """SPHERE; P_FIELD A; <middle>; P_FIELD B; END with A a 3-box and B a 5-box stage (one iteration each)."""
    ops = np.array([(oc.P_SPHERE, 0, 0, 0), (oc.P_FIELD, 0, 0, 0), (middle, 0, 0, 0), (oc.P_FIELD, 0, 1, 0),
                    (oc.END, 0, 0, 0)], dtype=OP_DTYPE)
    stages = [dict(blob=0, kind=0, ksize=(3, 3, 3), iterations=1, res=R3),
              dict(blob=1, kind=0, ksize=(5, 5, 5), iterations=1, res=R3)]
    return Program(ops, np.array([1.0]), [np.zeros((1, 0)), np.zeros((1, 0))], 1, 1, stages)


def test_a_stage_that_pruning_drops_is_not_planned():
    # NEG keeps A's value alive into B's prefix: A exact on B's eval range (4, 11), evaluated on (3, 12)
    kept = _synthetic(oc.NEG).stage_plan(RES3, (6, 9))[0]
    assert _ranges(kept) == [((3, 12), (4, 11)), ((4, 11), (6, 9))]
    # a second leaf overwrites A's value: B's pruned prefix no longer reads A, so A is not computed at all
    dropped = _synthetic(oc.P_SPHERE).stage_plan(RES3, (6, 9))[0]
    assert _ranges(dropped) == [(None, None), ((4, 11), (6, 9))]


def test_a_stage_on_one_branch_of_a_union():
    a = ab.Sphere(0.8)
    a.conv_averaging(4, 2, R3)   # 2 * 1 below, 2 * 2 above
    b = ab.Box(1.0, 1.0, 1.0)
    u = ab.CombineGeometry("UNION2").combine(a, b)
    plan, _ = ab.flatten(u).stage_plan(RES3, (6, 9))
    assert _ranges(plan) == [((4, 13), (6, 9))]


def test_signed_then_box():
    s = ab.Sphere(1.0)
    s.signed(R3)
    s.conv_averaging(3, 1, R3)
    prog = ab.flatten(s)
    # box: exact on (6, 9), evaluated on (5, 10); signed exact on (5, 10). Its mask needs every plane's field, so its
    # prefix runs on the whole axis when this process packs the whole mask ...
    assert _ranges(prog.stage_plan(RES3, (6, 9))[0]) == [((0, 17), (5, 10)), ((5, 10), (6, 9))]
    # ... and on its own planes when the mask of the other slabs comes from elsewhere (sharded: all-gathered)
    assert _ranges(prog.stage_plan(RES3, (6, 9), mask_planes=(6, 9))[0]) == [((5, 10), (5, 10)), ((5, 10), (6, 9))]


def test_signed_alone_and_bad_slabs():
    s = ab.Sphere(1.0)
    s.signed(R3)
    prog = ab.flatten(s)
    assert _ranges(prog.stage_plan(RES3, (0, 1))[0]) == [((0, 17), (0, 1))]
    assert _ranges(prog.stage_plan(RES3, (16, 17), mask_planes=(12, 17))[0]) == [((12, 17), (16, 17))]
    assert _ranges(prog.stage_plan(RES3)[0]) == [((0, 17), (0, 17))]
    for bad in ((3, 3), (-1, 2), (10, 18)):
        with pytest.raises(ValueError):
            prog.stage_plan(RES3, bad)
