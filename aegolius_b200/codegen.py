"""Program compiler: one straight-line sm_100a kernel per program STRUCTURE.

The interpreter (csrc/ab_interp.cuh) pays, per op and per thread, a shared-memory op fetch, a ~7-level dispatch tree,
argument loads from shared memory and a shared-memory round trip for every saved coordinate / value. All of that is
known on the host: control flow is identical for every grid point. This module emits the kernel BODY for one flattened
program — the call sequence over the same hand-written op bodies (csrc/ab_ops.cuh) with

  * compile-time slot numbers: P / V slots become local variables (registers) instead of shared-memory columns,
  * compile-time argument offsets: arguments are still passed at every launch (KParams.args, constant bank 0), so a
    parameter sweep or an optimisation loop reuses ONE binary, but each a[i] is a direct constant-bank operand instead
    of a shared-memory load. Tables (instance records, sector tables, polylines: dynamically indexed) are staged in
    shared memory and addressed through the run-time offset the launcher wrote, so their size is not part of the key,
  * compile-time immediates (axis, instancing mode, fused-PUSH flags) and points per thread chosen per program.

The binary is cached under aegolius_b200/jit/ by a digest of (signature, dtype, gradient mode, options, sources) and
registered with the library (ab_prog_register) under the structure's signature; run_program then prefers it over the
interpreter tiers. Same op bodies, explicitly rounded arithmetic (no cross-op FMA contraction): results are
bit-identical to the interpreter (tests/test_gpu_jit.py).

Reference semantics of the evaluation order being compiled: Code/spomso/spomso/cores/geom.py:29-60,
transformations.py:232-242, modifications.py:88-98 (closure chain), combine.py:115-163.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import threading

import numpy as np

from . import opcodes as oc

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
JIT_DIR = os.path.join(HERE, "jit")
CODEGEN_VERSION = 1

TABLE_OPS = (oc.ROTSYM, oc.CURVE_INST, oc.P_SEGLINE, oc.P_SEGLINE2D, oc.P_POLYGON2D, oc.POLY_SIGN)  # is_table_op() in ab_interp.cuh

# ops without transcendental functions or tables (is_lite_op() in ab_interp.cuh): cheap per point, so more points per thread
LITE_OPS = frozenset((
    oc.END, oc.SAVE_P, oc.LOAD_P, oc.PUSH_V, oc.AFFINE, oc.TRANSLATE, oc.NEXT_AFFINE, oc.NEXT_TRANSLATE, oc.NEXT_LOAD,
    oc.SCALE_P, oc.ELONGATE, oc.ABSX_SUB, oc.SYMMETRY, oc.REVOLVE, oc.REP_INF, oc.ZERO_Z, oc.ROUND, oc.ABS, oc.NEG, oc.SIGN,
    oc.ONION, oc.CONCENTRIC, oc.SCALE_V, oc.EXTRUDE_BEGIN, oc.EXTRUDE_END, oc.C_UNION, oc.C_INTERSECT, oc.C_SUBTRACT,
    oc.C_SUM, oc.C_DIFF, oc.C_SMIN2, oc.C_SMIN3, oc.C_SMAX3, oc.C_SSUB3, oc.P_SPHERE, oc.P_CYLINDER, oc.P_BOX, oc.P_TORUS,
    oc.P_CHAINLINK, oc.P_PLANE, oc.P_UPLANE, oc.P_SEGMENT, oc.P_AXIS, oc.P_CIRCLE, oc.P_BOX2D, oc.P_SEGMENT2D, oc.P_FIELD))

# programs longer than this stay on the interpreter: straight-line code grows with the program and would outgrow the
# instruction caches (and nvcc's patience)
MAX_COMPILED_OPS = 256

KINDS = {  # (dtype, grad) -> (kind id, T, dual K or 0, param)
    ("f32", "none"): (0, "float", 0, False), ("f32", "spatial"): (1, "float", 3, False),
    ("f64", "none"): (2, "double", 0, False), ("f64", "spatial"): (3, "double", 3, False),
    ("f32", "param"): (4, "float", 1, True), ("f64", "param"): (5, "double", 1, True),
}


def signature(prog) -> np.ndarray:
    """(opcode | a << 16 | b << 24) for every op before the terminator: what ab_prog_register keys on."""
    ops = prog.ops
    n = len(ops)
    while n > 0 and int(ops[n - 1]["opcode"]) == oc.END:
        n -= 1
    o = ops[:n]
    return (o["opcode"].astype(np.uint32) | (o["a"].astype(np.uint32) << 16) | (o["b"].astype(np.uint32) << 24))


def signature_hash(sig, dtype_code, grad_mode) -> int:
    """FNV-1a, identical to sig_hash() in csrc/ab_capi.cu (tests compare the two)."""
    h = 1469598103934665603
    for w in list(np.asarray(sig, dtype=np.uint32)) + [dtype_code, grad_mode]:
        w = int(w)
        for k in range(4):
            h ^= (w >> (8 * k)) & 0xff
            h = (h * 1099511628211) & 0xffffffffffffffff
    return h


def fixed_arg_offsets(sig):
    """Offsets (in the kernel's repacked pool) of the ops with a fixed argument count: run_program packs them first, in
    program order, each on a 16-byte boundary (4 scalars), tables afterwards."""
    offs, cursor = {}, 0
    for i, w in enumerate(sig):
        code = int(w) & 0xffff
        if code in TABLE_OPS:
            continue
        offs[i] = cursor
        cursor = (cursor + oc.ARG_COUNT[code] + 3) & ~3
    return offs


def default_options(sig, dtype, grad):
    """Points per thread, the occupancy the register allocator is asked for and the store path, per program class.
    Measured on B200 (profiles/r02_jit_sweep.md): write-bound programs (a handful of cheap ops) want 8 points per thread
    with the warp-transposed store (every STG.128 of a warp covers 512 contiguous bytes; direct 8-wide stores half-fill
    each sector and run at 52 % of the HBM peak instead of 84 %); issue-bound cheap programs want 8 points and direct
    stores; programs with transcendentals want fewer registers per thread the longer they are. `rowsplit` (the body a second
    time for warps whose threads each stay inside one grid row: x and y become per-thread scalars and the compiler drops
    the lane-redundant packed work) pays with 8 points per thread: sphere 81 -> 94 %, C1 42 -> 48 % of the HBM peak, a
    36-op union of boxes and spheres 4.58 -> 3.80 ms; nothing at 4 points (C1 field + gradient) and a loss on C2."""
    lite = all((int(w) & 0xffff) in LITE_OPS for w in sig)
    n = len(sig)
    if grad == "param":
        return dict(width=2 if dtype == "f32" else 1, min_ctas=5)
    if dtype == "f32":
        if grad == "none":
            if lite:
                if n <= 4:
                    return dict(width=8, min_ctas=6, stage8=True, store=1, rowsplit=True)
                return dict(width=8, min_ctas=8, rowsplit=n <= 64)
            if any((int(w) & 0xffff) == oc.CURVE_INST for w in sig):
                # flat walk with the warp-cooperative instance search: the fewer points a thread owns, the smaller the
                # warp's needle (C3 513^3: 2 points 1.69 ms, 4 points 1.82, 8 points 1.90, 8 + second body 2.23)
                return dict(width=2, min_ctas=7)
            if n <= 8:
                return dict(width=8, min_ctas=8, rowsplit=True)
            return dict(width=8, min_ctas=5, rowsplit=True) if n <= 32 else dict(width=4, min_ctas=5)
        return dict(width=4, min_ctas=4) if lite else dict(width=2, min_ctas=7)
    if grad == "none":
        return dict(width=2, min_ctas=6)
    return dict(width=1, min_ctas=6)


class _Emitter:
    def __init__(self, sig, param, slots):
        self.sig = [int(w) for w in sig]
        self.param = param
        self.slots = slots
        self.offs = fixed_arg_offsets(self.sig)
        self.lines = []
        self.n_p = 0
        self.n_v = 0
        self.tables = any((w & 0xffff) in TABLE_OPS for w in self.sig)
        self.leaf_point = "p"  # the variable a primitive reads its point from (the pull-back emitter seeds a dual copy `q`)

    def arg(self, i):
        code = self.sig[i] & 0xffff
        if code in TABLE_OPS:
            base = f"(s_args + (kp.ops[{i}].y & 0xffffu))"
        else:
            base = f"(kp.args + {self.offs[i]})"
        if self.param:
            return f"ArgD<S>{{{base}, {base} + kParamHalf}}"
        return base

    # slot access ------------------------------------------------------------------------------------------
    def save_p(self, s):
        self.n_p = max(self.n_p, s + 1)
        if self.slots == "smem":
            return (f"SK::st(pstack, {3 * s}, kNT, p.x); SK::st(pstack, {3 * s + 1}, kNT, p.y); "
                    f"SK::st(pstack, {3 * s + 2}, kNT, p.z);")
        return f"P{s} = p;"

    def load_p(self, s):
        self.n_p = max(self.n_p, s + 1)
        if self.slots == "smem":
            return (f"p.x = SK::ld(pstack, {3 * s}, kNT); p.y = SK::ld(pstack, {3 * s + 1}, kNT); "
                    f"p.z = SK::ld(pstack, {3 * s + 2}, kNT);")
        return f"p = P{s};"

    def store_v(self, s, expr="acc"):
        self.n_v = max(self.n_v, s + 1)
        if self.slots == "smem":
            return f"SK::st(vstack, {s}, kNT, {expr});"
        return f"V{s} = {expr};"

    def get_v(self, s):
        self.n_v = max(self.n_v, s + 1)
        if self.slots == "smem":
            return f"SK::ld(vstack, {s}, kNT)"
        return f"V{s}"

    # one op -----------------------------------------------------------------------------------------------
    def op(self, i):
        w = self.sig[i]
        code, a, b = w & 0xffff, (w >> 16) & 0xff, (w >> 24) & 0xff
        A = self.arg(i)
        name = oc.NAMES[code]
        e = self.lines.append
        e(f"    // {i}: {name} a={a} b={b}")
        simple_p = {oc.AFFINE: "op_affine", oc.TRANSLATE: "op_translate", oc.SCALE_P: "op_scale_p", oc.ELONGATE: "op_elongate",
                    oc.TWIST: "op_twist", oc.BEND: "op_bend", oc.ABSX_SUB: "op_absx_sub", oc.ROTSYM: "op_rotsym",
                    oc.REVOLVE: "op_revolve", oc.AXIS_REVOLVE: "op_axis_revolve", oc.REP_INF: "op_rep_inf",
                    oc.REP_FIN: "op_rep_fin"}
        prims = {oc.P_SPHERE: "prim_sphere", oc.P_CYLINDER: "prim_cylinder", oc.P_BOX: "prim_box", oc.P_TORUS: "prim_torus",
                 oc.P_CHAINLINK: "prim_chainlink", oc.P_BRAID: "prim_braid", oc.P_ARC3D: "prim_arc3d", oc.P_PLANE: "prim_plane",
                 oc.P_UPLANE: "prim_uplane", oc.P_SEGMENT: "prim_segment", oc.P_CONE: "prim_cone",
                 oc.P_SOLID_ANGLE: "prim_solid_angle", oc.P_TRIANGLE3D: "prim_triangle3d", oc.P_QUAD3D: "prim_quad3d",
                 oc.P_CIRCLE: "prim_circle", oc.P_NEU_CIRCLE: "prim_neu_circle", oc.P_BOX2D: "prim_box2d",
                 oc.P_SEGMENT2D: "prim_segment2d", oc.P_RBOX2D: "prim_rbox2d", oc.P_TRIANGLE2D: "prim_triangle2d",
                 oc.P_ARC: "prim_arc", oc.P_SECTOR: "prim_sector", oc.P_INF_SECTOR: "prim_inf_sector", oc.P_NGON: "prim_ngon",
                 oc.P_POLYGON2D: "prim_polygon2d"}
        pps = {oc.PP_SIGMOID: "pp_sigmoid", oc.PP_POS_SIGMOID: "pp_pos_sigmoid", oc.PP_CAPPED_EXP: "pp_capped_exp",
               oc.PP_HARD_BIN: "pp_hard_bin", oc.PP_LINEAR: "pp_linear", oc.PP_RELU: "pp_relu",
               oc.PP_SMOOTH_RELU: "pp_smooth_relu", oc.PP_SLOWSTART: "pp_slowstart",
               oc.PP_GAUSS_BOUNDARY: "pp_gauss_boundary", oc.PP_GAUSS_FALLOFF: "pp_gauss_falloff"}
        combines = {oc.C_UNION: "min_({v}, acc)", oc.C_INTERSECT: "max_({v}, acc)", oc.C_SUBTRACT: "max_({v}, -acc)",
                    oc.C_SUM: "{v} + acc", oc.C_DIFF: "{v} - acc", oc.C_SMIN2: "smin_poly2({v}, acc, a[0])",
                    oc.C_SMIN3: "smin_poly3({v}, acc, a[0])", oc.C_SMAX3: "-smin_poly3(-{v}, -acc, a[0])",
                    oc.C_SSUB3: "-smin_poly3(-{v}, acc, a[0])", oc.C_BOLTZ_INT: "smax_boltz({v}, acc, a[0])",
                    oc.C_BOLTZ_SUB: "smax_boltz({v}, -acc, a[0])"}
        xyz = "xyz"
        if code == oc.SAVE_P:
            e("    " + self.save_p(a))
        elif code == oc.LOAD_P:
            e("    " + self.load_p(a))
        elif code == oc.PUSH_V:
            e("    " + self.store_v(a))
        elif code in (oc.NEXT_AFFINE, oc.NEXT_TRANSLATE, oc.NEXT_LOAD):
            if b:
                e("    " + self.store_v(b - 1))
            e("    " + self.load_p(a))
            if code == oc.NEXT_AFFINE:
                e(f"    op_affine(p, {A});")
            elif code == oc.NEXT_TRANSLATE:
                e(f"    op_translate(p, {A});")
        elif code in simple_p:
            e(f"    {simple_p[code]}(p, {A});")
        elif code == oc.SYMMETRY:
            e(f"    p.{xyz[a]} = abs_(p.{xyz[a]});")
        elif code == oc.LIN_INST:
            e(f"    op_lin_inst(p, {A}, {a});")
        elif code == oc.CURVE_INST:
            e(f"    op_curve_inst(p, {A}, {a});")
        elif code == oc.ZERO_Z:
            e("    p.z = constant_like(p.z, T(0));")
        elif code == oc.ROUND:
            e(f"    {{ auto a = {A}; acc = acc - a[0]; }}")
        elif code == oc.ABS:
            e("    acc = abs_(acc);")
        elif code == oc.NEG:
            e("    acc = -acc;")
        elif code == oc.SIGN:
            e("    acc = sign_(acc);")
        elif code == oc.ONION:
            e(f"    {{ auto a = {A}; acc = abs_(acc) - a[0]; }}")
        elif code == oc.CONCENTRIC:
            e(f"    {{ auto a = {A}; acc = abs_(acc - a[0]); }}")
        elif code == oc.SCALE_V:
            e(f"    {{ auto a = {A}; acc = acc * a[0]; }}")
        elif code == oc.EXTRUDE_BEGIN:
            e(f"    {{ auto a = {A}; {self.store_v(a, 'abs_(p.z) - a[0]')} p.z = constant_like(p.z, T(0)); }}")
        elif code == oc.EXTRUDE_END:
            e(f"    acc = op_extrude_end<S, T>(acc, {self.get_v(a)});")
        elif code == oc.POLY_SIGN:
            self.n_p = max(self.n_p, a + 1)
            if self.slots == "smem":
                e(f"    acc = op_poly_sign(acc, SK::ld(pstack, {3 * a}, kNT), SK::ld(pstack, {3 * a + 1}, kNT), {A}, {b});")
            else:
                e(f"    acc = op_poly_sign(acc, P{a}.x, P{a}.y, {A}, {b});")
        elif code in pps:
            e(f"    acc = {pps[code]}(acc, {A});")
        elif code in combines:
            e(f"    {{ auto a = {A}; (void)a; acc = {combines[code].format(v=self.get_v(a))}; }}")
            if b:
                e("    " + self.store_v(b - 1))
        elif code in prims:
            e(f"    acc = {prims[code]}({self.leaf_point}, {A});")
        elif code in (oc.P_OINF_CONE, oc.P_INF_CONE):
            e(f"    acc = prim_inf_cone({self.leaf_point}, {A}, {'true' if code == oc.P_OINF_CONE else 'false'});")
        elif code in (oc.P_SEGLINE, oc.P_SEGLINE2D):
            e(f"    acc = prim_segline({self.leaf_point}, {A}, {3 if code == oc.P_SEGLINE else 2});")
        elif code == oc.P_AXIS:
            e(f"    {{ auto a = {A}; acc = {self.leaf_point}.{xyz[a]} - a[0]; }}")
        elif code == oc.P_FIELD:
            if self.param:  # the stencil's tangent row rides along (ab_program.dblobs)
                e(f"    load_field(kp.blob[{b}], kp.dblob[{b}], idx, kp.n, acc);")
            else:
                e(f"    load_field(kp.blob[{b}], idx, kp.n, acc);")
        elif code == oc.P_POINT_CLOUD:
            e(f"    acc = prim_point_cloud<S, T>({self.leaf_point}, kp.blob[{b}], kp.blob_count[{b}], {a}, kp.blob_tree[{b}]);")
        else:
            raise NotImplementedError(f"codegen: opcode {code} ({name})")



class _NoAdjoint(Exception):
    """The program holds an op without a pull-back: the forward-mode build serves it."""


class _AdjointEmitter(_Emitter):
    """Field + spatial gradient with the chain rule applied backwards through the coordinate ops (csrc/ab_adjoint.cuh):
    coordinate ops run on plain points and leave their Jacobian's ingredients in registers, primitives are evaluated on an
    identity-seeded dual point (value + gradient in local coordinates), and a gradient is pulled back to the frame it is
    needed in — the common frame of two values at a combine, the grid's at the end. Frames form a tree (SAVE_P / LOAD_P
    branch it); a node = (parent, pull-back statement)."""

    def __init__(self, sig):
        super().__init__(sig, False, "reg")
        self.nodes = [(None, None)]
        self.cur = 0          # frame of `p`
        self.acc_node = 0     # frame of `acc`
        self.slot_node = {}   # P slot -> frame
        self.v_node = {}      # V slot -> frame

    def node(self, pb):
        self.nodes.append((self.cur, pb))
        self.cur = len(self.nodes) - 1

    def _chain(self, n):
        out = []
        while n is not None:
            out.append(n)
            n = self.nodes[n][0]
        return out

    def lca(self, a, b):
        ca = self._chain(a)
        sb = set(self._chain(b))
        return next(n for n in ca if n in sb)

    def pull(self, var, n, to):
        while n != to:
            parent, pb = self.nodes[n]
            self.lines.append("    " + pb.format(v=var))
            n = parent

    def save_p(self, s):
        self.slot_node[s] = self.cur
        return super().save_p(s)

    def load_p(self, s):
        self.cur = self.slot_node[s]
        return super().load_p(s)

    def store_v(self, s, expr="acc"):
        self.v_node[s] = self.acc_node
        return super().store_v(s, expr)

    def finish(self):
        self.lines.append("    // gradient back to grid coordinates")
        self.pull("acc", self.acc_node, 0)

    def op(self, i):
        w = self.sig[i]
        code, a, b = w & 0xffff, (w >> 16) & 0xff, (w >> 24) & 0xff
        A = self.arg(i)
        e = self.lines.append
        head = f"    // {i}: {oc.NAMES[code]} a={a} b={b}"
        identity_jacobian = {oc.TRANSLATE: "op_translate", oc.REP_INF: "op_rep_inf", oc.REP_FIN: "op_rep_fin"}
        taped = {oc.ELONGATE: ("TapeElongate<P>", "fwd_elongate(p, {A}, {t});", "pb_elongate({{v}}, {t});"),
                 oc.TWIST: ("TapeTwist<P>", "fwd_twist(p, {A}, {t});", "pb_twist({{v}}, {A}, {t});"),
                 oc.BEND: ("TapeBend<P>", "fwd_bend(p, {A}, {t});", "pb_bend({{v}}, {A}, {t});"),
                 oc.ROTSYM: ("TapeRot<P>", "fwd_rotsym(p, {A}, {t});", "pb_rot({{v}}, {t});"),
                 oc.REVOLVE: ("TapeRevolve<P>", "fwd_revolve(p, {A}, {t});", "pb_revolve({{v}}, {t});"),
                 oc.AXIS_REVOLVE: ("TapeRevolve<P>", "fwd_axis_revolve(p, {A}, {t});", "pb_axis_revolve({{v}}, {A}, {t});")}
        local_gradient = {oc.P_SPHERE: "grad_sphere", oc.P_TORUS: "grad_torus", oc.P_BOX: "grad_box", oc.P_CYLINDER: "grad_cylinder"}
        t = f"t{i}"
        if code in (oc.SAVE_P, oc.LOAD_P, oc.PUSH_V):
            super().op(i)
        elif code in (oc.NEXT_AFFINE, oc.NEXT_TRANSLATE, oc.NEXT_LOAD):
            e(head)
            if b:
                e("    " + self.store_v(b - 1))
            e("    " + self.load_p(a))
            if code == oc.NEXT_AFFINE:
                e(f"    op_affine(p, {A});")
                self.node(f"pb_affine({{v}}, {A});")
            elif code == oc.NEXT_TRANSLATE:
                e(f"    op_translate(p, {A});")
        elif code == oc.AFFINE:
            e(head)
            e(f"    op_affine(p, {A});")
            self.node(f"pb_affine({{v}}, {A});")
        elif code in identity_jacobian:
            e(head)
            e(f"    {identity_jacobian[code]}(p, {A});")
        elif code == oc.LIN_INST:
            e(head)
            e(f"    op_lin_inst(p, {A}, {a});")
        elif code == oc.SCALE_P:
            e(head)
            e(f"    op_scale_p(p, {A});")
            self.node(f"pb_scale({{v}}, ({A})[0]);")
        elif code in taped:
            ty, fwd, pb = taped[code]
            e(head)
            e(f"    {ty} {t};")
            e("    " + fwd.format(A=A, t=t))
            self.node(pb.format(A=A, t=t))
        elif code in (oc.ABSX_SUB, oc.SYMMETRY):
            ax = 0 if code == oc.ABSX_SUB else a
            c = "xyz"[ax]
            e(head)
            e(f"    const Mask<W> {t} = lt_(p.{c}, T(0));")
            e(f"    op_absx_sub(p, {A});" if code == oc.ABSX_SUB else f"    p.{c} = abs_(p.{c});")
            self.node(f"pb_flip<{ax}>({{v}}, {t});")
        elif code == oc.CURVE_INST:
            e(head)
            e(f"    int {t}[W];")
            e(f"    fwd_curve_inst(p, {A}, {a}, {t});")
            if a:  # aligned variants rotate into the instance's frame; the plain one only translates
                self.node(f"pb_curve_inst({{v}}, {A}, {t});")
        elif code == oc.ZERO_Z:
            e(head)
            e("    p.z = P(T(0));")
            self.node("pb_zero_z({v});")
        elif code == oc.EXTRUDE_BEGIN:
            e(head)
            self.n_v = max(self.n_v, a + 1)
            self.v_node[a] = self.cur
            e(f"    {{ auto a = {A}; Pt<S> q; seed_local(q, p); V{a} = abs_(q.z) - a[0]; }}")
            e("    p.z = P(T(0));")
            self.node("pb_zero_z({v});")
        elif code == oc.EXTRUDE_END:
            e(head)
            to = self.lca(self.acc_node, self.v_node[a])
            self.pull(f"V{a}", self.v_node[a], to)
            self.v_node[a] = to
            self.pull("acc", self.acc_node, to)
            e(f"    acc = op_extrude_end<S, T>(acc, V{a});")
            self.acc_node = to
        elif code in (oc.ROUND, oc.ABS, oc.NEG, oc.SIGN, oc.ONION, oc.CONCENTRIC, oc.SCALE_V) or oc.PP_SIGMOID <= code <= oc.PP_GAUSS_FALLOFF:
            super().op(i)  # value ops: the dual number keeps its frame
        elif oc.C_UNION <= code <= oc.C_BOLTZ_SUB:
            to = self.lca(self.acc_node, self.v_node[a])
            e(f"    // {i}: operands of the combine into their common frame")
            self.pull(f"V{a}", self.v_node[a], to)
            self.v_node[a] = to  # (the slot now holds the pulled-back gradient, should it be read again)
            self.pull("acc", self.acc_node, to)
            self.acc_node = to
            super().op(i)
        elif code == oc.POLY_SIGN:  # the interior sign at the coordinates saved in slot a: a factor -1 / +1, the frame stays
            self.n_p = max(self.n_p, a + 1)
            e(head)
            e(f"    acc = op_poly_sign(acc, S(P{a}.x), S(P{a}.y), {A}, {b});")
        elif code in local_gradient:
            e(head)
            e(f"    acc = {local_gradient[code]}(p, {A});")
            self.acc_node = self.cur
        elif oc.P_SPHERE <= code <= oc.P_POINT_CLOUD or oc.P_CIRCLE <= code <= oc.P_POLYGON2D:  # (not P_FIELD: no derivative)
            # the primitive on an identity-seeded dual point: value + gradient in local coordinates
            n0 = len(self.lines)
            self.leaf_point = "q"
            try:
                super().op(i)
            finally:
                self.leaf_point = "p"
            body = self.lines[n0 + 1:]
            del self.lines[n0 + 1:]
            e("    {")
            e("      Pt<S> q;")
            e("      seed_local(q, p);")
            for ln in body:
                e("  " + ln)
            e("    }")
            self.acc_node = self.cur
        else:
            raise _NoAdjoint(oc.NAMES.get(code, str(code)))


_TEMPLATE = r'''// generated by aegolius_b200/codegen.py (version @VERSION@) — do not edit.
// program signature hash @HASH@, @NOPS@ ops; @KINDNAME@; @WIDTH@ points per thread, slots in @SLOTS@, 2D-grid flavour @IS2D@.
#define AB_TIER_FULL 2
#define AB_STORE_POLICY @STOREPOLICY@
#include "ab_interp.cuh"
#include "ab_adjoint.cuh"

namespace ab {
typedef @T@ ProgT;
typedef @S@ ProgS;
constexpr bool kParam = @PARAM@;
constexpr int kNT = @NT@;
constexpr bool kTables = @TABLES@;
constexpr int kIs2D = @IS2D@;  // grid flavour this binary serves: 0 = 3D grids and point lists, 1 = 2D grids
constexpr int kNP = @NP@, kNV = @NV@;  // shared-memory slot columns (0 when the slots live in registers)
constexpr bool kCompact = @COMPACT@;  // compact 16 x 16 tiles (3D grids) instead of the flat walk
constexpr bool kStage8 = @STAGE8@;    // Pack<float, 8> results leave through the per-warp transposition (store_pack_w8_transposed)

__global__ void __launch_bounds__(kNT, @MINCTAS@) ab_prog_kernel(const __grid_constant__ KParams<ProgT> kp) {
  typedef ProgT T;
  typedef ProgS S;
  constexpr int W = S::width;
  typedef Pack<T, W> P;
  typedef StackOf<S> SK;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* s_args = reinterpret_cast<T*>(smem_raw);
  P* pstack = reinterpret_cast<P*>(smem_raw + kp.off_pstack);
  P* vstack = reinterpret_cast<P*>(smem_raw + kp.off_vstack);
  if (kTables) {  // tables are indexed per point: staged once per persistent CTA (the scalar arguments are not read from here)
    for (uint32_t i = threadIdx.x; i < kp.n_args; i += kNT) s_args[i] = kp.args[i];
    __syncthreads();
  }
  double loss_sum = 0.0, dloss_sum = 0.0;  // loss mode only (parameter-tangent kernels)
@LOOPHEAD@
@BODYALL@
  }
  if constexpr (kParam) {
    if (kp.loss_accum) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        loss_sum += __shfl_xor_sync(0xffffffffu, loss_sum, off);
        dloss_sum += __shfl_xor_sync(0xffffffffu, dloss_sum, off);
      }
      if ((threadIdx.x & 31) == 0) {
        atomicAdd(kp.loss_accum, loss_sum);
        atomicAdd(kp.loss_accum + 1, dloss_sum);
      }
    }
  }
}
}  // namespace ab

#define AB_PROG_EXPORT extern "C" __attribute__((visibility("default")))

// same contract as ab_spec_launch (csrc/ab_interp_spec.cu): returns the cudaError_t of the launch, *status = AB_OK / AB_ETOOLARGE
AB_PROG_EXPORT int ab_prog_launch(const void* kparams, int sms, unsigned long long smem_optin, void* stream, int* status) {
  using namespace ab;
  const KParams<ProgT>& kp = *reinterpret_cast<const KParams<ProgT>*>(kparams);
  typedef StackOf<ProgS> SK;
  *status = AB_OK;
  const size_t args_bytes = kTables ? prog_args_bytes<ProgT>(kp.n_args) : 0;
  const size_t stack_bytes = (size_t)sizeof(typename SK::P) * SK::cols * ((size_t)kNP * 3 + kNV) * kNT;
  const size_t smem = args_bytes + stack_bytes + (kStage8 ? (size_t)kNT * 32 : 0);
  if (smem > (size_t)smem_optin) {
    *status = AB_ETOOLARGE;
    return (int)cudaSuccess;
  }
  cudaError_t e;
  static size_t attr_smem = 0;
  if (smem > 48 * 1024 && smem > attr_smem) {
    e = cudaFuncSetAttribute(ab_prog_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    attr_smem = smem;
  }
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ab_prog_kernel, kNT, smem);
  if (e != cudaSuccess) return (int)e;
  if (occ < 1) {
    *status = AB_ETOOLARGE;
    return (int)cudaSuccess;
  }
  const uint64_t tile_pts = (uint64_t)kNT * ProgS::width;
  const uint32_t nb1 = (kp.g.n1 + compact_tile_rows(ProgS::width) - 1) / compact_tile_rows(ProgS::width), nb2 = compact_col_blocks(kp.g.n2);
  if (kCompact && (!kp.grid_mode || kp.g.is2d || kp.n % kp.g.plane)) {
    *status = AB_EINVAL;  // (run_program only sends whole planes of 3D grids here)
    return (int)cudaSuccess;
  }
  const uint64_t n_tiles = kCompact ? (kp.n / kp.g.plane) * nb1 * nb2 : (kp.n + tile_pts - 1) / tile_pts;
  const uint64_t resident = (uint64_t)sms * occ;  // persistent CTAs: a whole number of resident waves
  const unsigned grid = (unsigned)(n_tiles < resident ? n_tiles : resident);
  KParams<ProgT>& k = const_cast<KParams<ProgT>&>(kp);
  k.off_args = (uint32_t)(args_bytes + stack_bytes);  // the staged arguments sit at offset 0; this field carries the store stage
  k.off_pstack = (uint32_t)args_bytes;
  k.off_vstack = (uint32_t)(args_bytes + (size_t)sizeof(typename SK::P) * SK::cols * kNP * 3 * kNT);
  if (kCompact) {  // gridDim.x tiles decomposed over (planes, row blocks, column blocks)
    k.tile_stride[0] = grid / (nb1 * nb2);
    const uint32_t rem = grid % (nb1 * nb2);
    k.tile_stride[1] = rem / nb2;
    k.tile_stride[2] = rem % nb2;
  } else if (kp.grid_mode) {
    const uint64_t d = (uint64_t)grid * tile_pts;
    k.tile_stride[0] = (uint32_t)(d / kp.g.plane);
    const uint64_t rem = d % kp.g.plane;
    k.tile_stride[1] = (uint32_t)(rem / kp.g.n2);
    k.tile_stride[2] = (uint32_t)(rem % kp.g.n2);
  }
  ab_prog_kernel<<<grid, kNT, smem, (cudaStream_t)stream>>>(kp);
  return (int)cudaGetLastError();
}
AB_PROG_EXPORT unsigned long long ab_prog_kparams_size(void) { return sizeof(ab::KParams<ab::ProgT>); }
AB_PROG_EXPORT int ab_prog_kind(void) { return @KIND@; }
AB_PROG_EXPORT int ab_prog_flavor(void) { return @FLAVOR@; }
AB_PROG_EXPORT unsigned long long ab_prog_hash(void) { return @HASH@ull; }
'''


def generate(sig, dtype="f32", grad="none", **opts) -> str:
    """CUDA source of the straight-line kernel for the program structure `sig` (see signature())."""
    sig = np.asarray(sig, dtype=np.uint32)
    if len(sig) == 0:
        raise ValueError("empty program")
    grad = grad or "none"
    kind, T, K, param = KINDS[(dtype, grad)]
    o = dict(slots="reg", nt=128, is2d=0, store=0, stage8=False, multicast=False, compact=False, rowsplit=False,
             adjoint=os.environ.get("AB_JIT_ADJOINT", "1") != "0")
    o.update(default_options(sig, dtype, grad))
    if opts.get("compact"):  # measured (profiles/r02_jit_sweep.md): C5 field + gradient 19.7 -> 18.8 ms, C3 value 1.82 -> 1.44 ms
        o.update(width=2, min_ctas=8, stage8=False)
        if dtype == "f32" and grad == "none":  # 4 points per thread halve the per-thread share of the search: 1.54 -> 1.36 ms
            o.update(width=4, min_ctas=7)
    o.update({k: v for k, v in opts.items() if v is not None})
    em = None
    adjoint = bool(o["adjoint"]) and grad == "spatial" and o["slots"] == "reg"
    if adjoint:  # gradient by pull-backs (ab_adjoint.cuh) when every op of the program has one
        try:
            em = _AdjointEmitter(sig)
            for i in range(len(sig)):
                em.op(i)
            em.finish()
        except _NoAdjoint:
            em, adjoint = None, False
    if adjoint and dtype == "f32":  # fewer live registers than three tangents per coordinate: one more CTA per SM fits
        lite = all((int(w) & 0xffff) in LITE_OPS for w in sig)
        # (C5 field + gradient on compact tiles: 2 points per thread 15.4 ms, 4 points 13.8 ms at 6 CTAs / SM, 79 registers)
        has_search = any((int(w) & 0xffff) == oc.CURVE_INST for w in sig)
        if opts.get("compact"):
            tuned = dict(width=4, min_ctas=6)
        elif lite:  # (a 36-op union: 6.05 ms with the second body, 5.87 without)
            tuned = dict(width=4, min_ctas=5, rowsplit=len(sig) <= 12)
        elif not has_search and len(sig) <= 48:  # twisted torus 769^3: 2 points 1.47 ms, 4 points 1.30 ms (87 % of the HBM peak)
            tuned = dict(width=4, min_ctas=6 if len(sig) <= 16 else 5)
        else:  # flat walk with the instance search: 2 points per thread (C3 513^3: 2.19 ms against 2.26)
            tuned = {}
        o.update({k: v for k, v in tuned.items() if opts.get(k) is None})
    elif adjoint and opts.get("min_ctas") is None:  # fp64: 64 registers are enough now (C3 256^3: 0.918 -> 0.900 ms)
        o.update(min_ctas=8)
    if o["multicast"]:
        o["store"] = 4  # multimem.st: `out` is a multicast address (ab_eval_grid_multicast)
        if dtype == "f32" and grad == "none" and opts.get("width") is None and int(o["width"]) < 4:
            o.update(width=4, min_ctas=5)  # 128-bit multimem stores, a warp's store = 512 contiguous bytes
    W = int(o["width"])
    if (T, W) not in (("float", 1), ("float", 2), ("float", 4), ("float", 8), ("double", 1), ("double", 2)):
        raise ValueError(f"no {W}-wide store for {T}")
    S = f"Pack<{T}, {W}>" if K == 0 else f"Dual<Pack<{T}, {W}>, {K}>"
    if em is None:
        em = _Emitter(sig, param, o["slots"])
        for i in range(len(sig)):
            em.op(i)
    decls = []
    if o["slots"] == "reg":
        if em.n_p:
            decls.append(f"    Pt<{'P' if adjoint else 'S'}> " + ", ".join(f"P{i}" for i in range(em.n_p)) + ";")
        if em.n_v:
            decls.append("    S " + ", ".join(f"V{i}" for i in range(em.n_v)) + ";")
    dcode = {"f32": 0, "f64": 1}[dtype]  # AB_F32 / AB_F64
    gcode = {"none": 0, "spatial": 1, "param": 2}[grad]
    rep = {"VERSION": CODEGEN_VERSION, "HASH": signature_hash(sig, dcode, gcode), "NOPS": len(sig),
           "KINDNAME": f"{dtype}, grad={grad}" + (" (gradient by pull-backs, ab_adjoint.cuh)" if adjoint else ""), "WIDTH": W, "SLOTS": "registers" if o["slots"] == "reg" else "shared memory",
           "T": T, "S": S, "PARAM": "true" if param else "false", "NT": int(o["nt"]),
           "TABLES": "true" if em.tables else "false", "NP": em.n_p if o["slots"] == "smem" else 0,
           "NV": em.n_v if o["slots"] == "smem" else 0, "MINCTAS": int(o["min_ctas"]), "IS2D": int(bool(o["is2d"])), "STOREPOLICY": int(o["store"]),
           "FLAVOR": int(bool(o["is2d"])) | (2 if o["multicast"] else 0) | (4 if o["compact"] else 0),
           "STAGE8": "true" if (o["stage8"] and W == 8 and K == 0 and T == "float") else "false", "DECLS": "\n".join(decls),
           "BODY": "\n".join(em.lines), "KIND": kind}
    flat_head = """  const uint32_t tile_pts = (uint32_t)kNT * W;
  const uint32_t n32 = (uint32_t)kp.n;
  const uint32_t n_tiles = (n32 + tile_pts - 1) / tile_pts;
  TileWalk walk;
  tile_walk_begin(kp, tile_pts, (uint32_t)W, walk);
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const uint32_t idx = tile * tile_pts + threadIdx.x * W;
    P cx, cy, cz;
    tile_coords<kIs2D>(kp, walk, idx, n32, cx, cy, cz);"""
    compact_head = """  // compact tiles: compact_tile_rows(W) x 16 points of one i0 plane per CTA (ab_interp.cuh), 3D grids only
  const uint32_t nb1 = (kp.g.n1 + compact_tile_rows(ProgS::width) - 1) / compact_tile_rows(ProgS::width), nb2 = compact_col_blocks(kp.g.n2);
  const uint32_t n_tiles = (uint32_t)(kp.n / kp.g.plane) * nb1 * nb2;
  CompactWalk walk;
  compact_walk_begin(kp, nb1, nb2, walk);
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    uint32_t idx;
    uint32_t valid;
    P cx, cy, cz;
    compact_coords(kp, walk, nb1, nb2, cx, cy, cz, idx, valid);"""
    split_head = """  const uint32_t tile_pts = (uint32_t)kNT * W;
  const uint32_t n32 = (uint32_t)kp.n;
  const uint32_t n_tiles = (n32 + tile_pts - 1) / tile_pts;
  TileWalk walk;
  tile_walk_begin(kp, tile_pts, (uint32_t)W, walk);
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const uint32_t idx = tile * tile_pts + threadIdx.x * W;
    P cx, cy, cz;"""
    rep["LOOPHEAD"] = compact_head if o["compact"] else (split_head if o["rowsplit"] else flat_head)
    rep["COMPACT"] = "true" if o["compact"] else "false"
    if o["compact"]:
        rep["EMIT"] = "    emit_compact(kp, acc, idx, valid);"
    elif rep["STAGE8"] == "true":
        rep["EMIT"] = ("    float4* stage = reinterpret_cast<float4*>(smem_raw + kp.off_args) + (threadIdx.x >> 5) * 64;\n"
                       "    store_pack_w8_transposed(kp.out, acc, tile * tile_pts + (threadIdx.x & ~31u) * W, kp.n, aligned, stage);")
    else:
        rep["EMIT"] = "    emit(kp, acc, idx, aligned);"
    if o["compact"] and not ((W == 2 or (W == 4 and T == "float")) and not param and int(o["nt"]) == 128 and not o["is2d"]):
        raise ValueError("compact tiles: 2 (or, fp32, 4) points per thread, 128 threads, 3D grids, value / spatial-gradient kernels")
    body_one = ("""    Pt<P> p;  // plain coordinates: the gradient is pulled back through the coordinate ops afterwards (ab_adjoint.cuh)
    seed(p, cx, cy, cz);
    S acc(T(0));
""" if adjoint else """    Pt<S> p;
    seed(p, cx, cy, cz);
    S acc = constant_like(p.x, T(0));
""") + """@DECLS@
@BODY@
    if constexpr (kParam) {
      if (kp.loss_accum) {
        accumulate_loss(kp, acc, idx, loss_sum, dloss_sum);
        continue;
      }
    }
    const bool aligned = ((reinterpret_cast<uintptr_t>(kp.out) & 15) == 0);
@EMIT@"""
    if o["rowsplit"] and not o["compact"]:
        # the body twice: behind the warp-wide "every run stays in its row" test the slow coordinates are broadcasts
        indent = lambda t: "\n".join(("  " + ln if ln else ln) for ln in t.split("\n"))
        rep["BODYALL"] = ("    if (__all_sync(0xffffffffu, tile_run_in_one_row<T, W>(kp, walk))) {\n"
                          "      tile_coords_uniform<kIs2D>(kp, walk, cx, cy, cz);\n" + indent(body_one) + "\n"
                          "    } else {\n"
                          "      tile_coords<kIs2D>(kp, walk, idx, n32, cx, cy, cz);\n" + indent(body_one) + "\n"
                          "    }")
    else:
        rep["BODYALL"] = body_one
    src = _TEMPLATE
    for k in ("BODYALL",):  # nested placeholders first
        src = src.replace(f"@{k}@", str(rep.pop(k)))
    for k, v in rep.items():
        src = src.replace(f"@{k}@", str(v))
    return src


# ---- building --------------------------------------------------------------------------------------------------------------------

_NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
               "-Xcompiler", "-fvisibility=hidden", "-diag-suppress", "177,186"]
_header_digest = None
_build_slots = threading.Semaphore(int(os.environ.get("AB_JIT_JOBS", "2")))  # background builds are polite to the host


# what a generated translation unit includes (directly or through ab_interp.cuh): only these decide whether a cached binary
# is still valid, so unrelated edits elsewhere in csrc/ do not throw the cache away
_INCLUDED = (os.path.join(CSRC, "ab_interp.cuh"), os.path.join(CSRC, "ab_ops.cuh"), os.path.join(CSRC, "ab_math.cuh"),
             os.path.join(CSRC, "ab_adjoint.cuh"),
             os.path.join(CSRC, "ab_tree.cuh"), os.path.join(CSRC, "ab_spec_default.h"),
             os.path.join(os.path.dirname(HERE), "include", "aegolius_b200.h"))


def _abi_relevant(text: str) -> str:
    """The public header without comments and without function prototypes: what is left (limits, enums, structs) is all a
    generated kernel depends on, so documenting or adding an entry point does not invalidate the cached binaries."""
    import re
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    text = re.sub(r"\b(?:int|uint64_t|const\s+char\s*\*)\s+ab_\w+\s*\([^;{]*\)\s*;", " ", text)
    return " ".join(text.split())


def _headers_digest():
    global _header_digest
    if _header_digest is None:
        h = hashlib.sha256()
        for f in _INCLUDED:
            with open(f, "rb") as fh:
                data = fh.read()
            if f.endswith("aegolius_b200.h"):
                data = _abi_relevant(data.decode()).encode()
            h.update(os.path.basename(f).encode())
            h.update(data)
        _header_digest = h.hexdigest()
    return _header_digest


def binary_path(src: str) -> str:
    dig = hashlib.sha256((src + _headers_digest() + " ".join(_NVCC_FLAGS)).encode()).hexdigest()[:24]
    return os.path.join(JIT_DIR, f"prog_{dig}.so")


def build_source(src: str, verbose=False, keep_ptxas=False) -> str:
    """nvcc -> aegolius_b200/jit/prog_<digest>.so (cached; atomic rename, so concurrent builders are safe)."""
    from .build import _nvcc
    out = binary_path(src)
    if os.path.exists(out):
        return out
    os.makedirs(JIT_DIR, exist_ok=True)
    cu = out[:-3] + f".{os.getpid()}.{threading.get_ident()}.cu"
    tmp = cu[:-3] + ".so.tmp"
    with open(cu, "w") as fh:
        fh.write(src)
    try:
        cmd = [_nvcc()] + _NVCC_FLAGS + (["-Xptxas", "-v"] if keep_ptxas else []) + [
            "-I", CSRC, "-shared", "-o", tmp, cu, "-lcudart"]
        with _build_slots:
            r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for a compiled program:\n{r.stdout}\n{r.stderr}")
        if keep_ptxas:
            with open(out[:-3] + ".ptxas.txt", "w") as fh:
                fh.write(r.stderr)
        os.replace(tmp, out)
    finally:
        for f in (cu, tmp):
            if os.path.exists(f):
                os.remove(f)
    if verbose:
        print(f"[aegolius_b200.codegen] {out}")
    return out


# ---- run-time management: load, register, build in the background ---------------------------------------------------------------

_loaded = {}        # binary path -> CDLL (keeps the shared object mapped)
_registered = set()  # (signature bytes, dtype, grad, is2d)
_pending = {}       # same key -> Thread
_failed = {}        # same key -> error text (a failed build is not retried)
_lock = threading.Lock()
_GRAD_NAMES = {None: "none", False: "none", "none": "none", True: "spatial", "spatial": "spatial", "xyz": "spatial",
               "param": "param"}


def mode() -> str:
    """AB_JIT = on (default: build in the background, interpreter meanwhile) | sync (block on the first build) |
    cache (use binaries already on disk, never run nvcc) | off."""
    m = os.environ.get("AB_JIT", "on").lower()
    return {"1": "on", "0": "off", "true": "on", "false": "off"}.get(m, m)


def set_mode(m: str):
    if m not in ("on", "sync", "cache", "off"):
        raise ValueError("mode must be 'on', 'sync', 'cache' or 'off'")
    os.environ["AB_JIT"] = m


def _key(sig, dtype, grad, flavor):
    return (np.asarray(sig, dtype=np.uint32).tobytes(), dtype, grad, int(flavor))


def _register(path, sig, dtype, grad, is2d):  # is2d: the flavour bits (bit 0 2D grid, bit 1 multicast stores, bit 2 compact tiles)
    import ctypes as C
    from . import cabi
    _DT = {"f32": (cabi.AB_F32,), "f64": (cabi.AB_F64,)}
    lib = _loaded.get(path)
    if lib is None:
        lib = C.CDLL(path)
        lib.ab_prog_kparams_size.restype = C.c_uint64
        _loaded[path] = lib
    kind = KINDS[(dtype, grad)][0]
    if lib.ab_prog_kind() != kind or lib.ab_prog_flavor() != int(is2d):
        raise RuntimeError(f"{path}: built for another kind / flavour")
    sig = np.ascontiguousarray(sig, dtype=np.uint32)
    gcode = {"none": cabi.AB_GRAD_NONE, "spatial": cabi.AB_GRAD_SPATIAL, "param": cabi.AB_GRAD_PARAM}[grad]
    cabi.check(cabi.lib().ab_prog_register(sig.ctypes.data, len(sig), _DT[dtype][0], gcode, int(is2d),
                                           C.cast(lib.ab_prog_launch, C.c_void_p), lib.ab_prog_kparams_size()))


def compilable(prog) -> bool:
    """Short enough to unroll, and made of ops this generator knows (anything else is the library's to reject)."""
    sig = signature(prog)
    return 0 < len(sig) <= MAX_COMPILED_OPS and all((int(w) & 0xffff) in oc.ARG_COUNT and (int(w) & 0xffff) != oc.END
                                                    for w in sig)


def wants_compact_tiles(sig, dtype, grad, is2d) -> bool:
    """fp32 programs with a warp-cooperative op (nearest curve instance) on a 3D grid: a compact-tile build (2 points per
    thread, 16 x 16 tiles) is registered beside the flat one, which keeps serving point lists."""
    return (os.environ.get("AB_JIT_COMPACT", "1") != "0" and dtype == "f32" and grad in ("none", "spatial") and not is2d and
            any((int(w) & 0xffff) == oc.CURVE_INST for w in sig))


def ensure(prog, dtype="f32", grad=None, is2d=False, how=None, multicast=False, **opts):
    """Makes the compiled kernel(s) of `prog`'s structure available to the library. Returns True when the kernel that will
    serve this (dtype, grad, grid kind) is registered on return, False when the interpreter serves the call (build in
    flight, disabled, too long a program, failed build). how: None = mode(); 'sync' blocks on the build.

    A structure with a warp-cooperative op gets two binaries: compact tiles for 3D grids (wants_compact_tiles) and the flat
    walk, which keeps serving point lists."""
    how = how or mode()
    if how == "off" or not compilable(prog):
        return False
    dtype = {"float32": "f32", "float64": "f64"}.get(str(dtype), dtype) if isinstance(dtype, str) else \
        ("f32" if np.dtype(dtype) == np.float32 else "f64")
    grad = _GRAD_NAMES[grad]
    sig = signature(prog)
    compact = opts.pop("compact", None)
    # (multicast stores: flat walk only — the 64-byte row segments of the compact tiles make poor NVLink packets: C5 field
    # assembly on 8 GPUs 8.1 ms flat, 11.9 ms compact)
    variants = [bool(compact)] if compact is not None else \
        ([True, False] if wants_compact_tiles(sig, dtype, grad, is2d) and not multicast else [False])
    ok = [_ensure_one(sig, dtype, grad, bool(is2d), how, multicast, c, opts) for c in variants]
    return ok[0]


def _ensure_one(sig, dtype, grad, is2d, how, multicast, compact, opts):
    flavor = int(is2d) | (2 if multicast else 0) | (4 if compact else 0)
    key = _key(sig, dtype, grad, flavor)
    if key in _registered:
        return True
    if key in _failed:
        return False
    with _lock:
        if key in _registered:
            return True
        th = _pending.get(key)
        if th is None:
            src = generate(sig, dtype, grad, is2d=is2d, multicast=multicast, compact=compact, **opts)
            path = binary_path(src)
            if os.path.exists(path):  # built earlier (this process, another one, or shipped with the tree): just load it
                _register(path, sig, dtype, grad, flavor)
                _registered.add(key)
                return True
            if how == "cache":
                return False

            def work():
                try:
                    p = build_source(src)
                    with _lock:
                        _register(p, sig, dtype, grad, flavor)
                        _registered.add(key)
                except Exception as exc:  # no nvcc / compile error: this structure stays on the interpreter
                    with _lock:
                        _failed[key] = str(exc)
                finally:
                    with _lock:
                        _pending.pop(key, None)

            th = threading.Thread(target=work, name="aegolius-jit", daemon=True)
            _pending[key] = th
            th.start()
    if how == "sync":
        th.join()
        if key in _failed:
            raise RuntimeError(_failed[key])
        return key in _registered
    return False


def wait(timeout=None):
    """Blocks until the background builds started so far are registered."""
    for th in list(_pending.values()):
        th.join(timeout)


def stats():
    from . import cabi
    return dict(registered=len(_registered), pending=len(_pending), failed=len(_failed),
                compiled_launches=int(cabi.lib().ab_prog_hits()))


def prebuild(items, jobs=None, verbose=False):
    """Ahead-of-time build of the kernels for `items` = iterable of (program, dtype, grad, is2d): fills aegolius_b200/jit/
    (e.g. from __graft_entry__.build(), which has nvcc but no GPU) so that the first evaluation finds its binary on disk.
    Returns (built, cached, failed) counts."""
    from concurrent.futures import ThreadPoolExecutor
    global _build_slots
    jobs = jobs or os.cpu_count() or 4
    todo, seen, cached = [], set(), 0
    for prog, dtype, grad, is2d in items:
        if not compilable(prog):
            continue
        grad = _GRAD_NAMES[grad]
        sig = signature(prog)
        key = _key(sig, dtype, grad, is2d)
        if key in seen:
            continue
        seen.add(key)
        srcs = [generate(sig, dtype, grad, is2d=is2d)]
        if wants_compact_tiles(sig, dtype, grad, is2d):
            srcs.append(generate(sig, dtype, grad, is2d=is2d, compact=True))
        for src in srcs:
            if os.path.exists(binary_path(src)):
                cached += 1
            else:
                todo.append(src)
    old, _build_slots = _build_slots, threading.Semaphore(jobs)
    failed = []

    def one(src):
        try:
            build_source(src)
        except Exception as exc:
            failed.append(str(exc)[-600:])
    try:
        with ThreadPoolExecutor(jobs) as ex:
            list(ex.map(one, todo))
    finally:
        _build_slots = old
    if verbose:
        print(f"[aegolius_b200.codegen] prebuilt {len(todo) - len(failed)} kernels, {cached} cached, {len(failed)} failed")
    if failed:
        raise RuntimeError("compiled-program builds failed:\n" + failed[0])
    return len(todo), cached, len(failed)
