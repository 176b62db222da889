"""Flattener: geometry tree (frontend.GenericGeometry) -> linear interpreter program.

The program is linearised in EVALUATION order. For a node with call-order modifications m1..mk the closure chain
of the reference makes the last-called modification the outermost wrapper (modifications.py:88-98), so the
coordinate parts run mk..m1 on the way down, then the leaf / children, then the value parts m1..mk on the way up,
then the node scale (transformations.py:232-242):

    AFFINE(R^T/s, -R^T t) ; pre(mk) .. pre(m1) ; <leaf | children + combine> ; post(m1) .. post(mk) ; SCALE_V(s)

Stack slots are resolved here (control flow is identical for every grid point), so the kernel only sees absolute
slot numbers. All constant sub-expressions (sin/cos of constant angles, frames, instance tables evaluated from the
user's Python curve callable) are folded on the host in fp64.
"""
from __future__ import annotations

import numpy as np

from . import opcodes as oc

OP_DTYPE = np.dtype([("opcode", "<u2"), ("a", "u1"), ("b", "u1"), ("arg", "<u4")])


class FlattenError(NotImplementedError):
    pass


class Program:
    def __init__(self, ops, args, blobs, n_pslots, n_vslots, stages=()):
        self.ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
        self.args = np.ascontiguousarray(args, dtype=np.float64)
        self.blobs = [np.ascontiguousarray(b, dtype=np.float64) for b in blobs]
        self.n_pslots = int(n_pslots)
        self.n_vslots = int(n_vslots)
        self.dargs = None
        # grid-stencil stages (conv_averaging / conv_edge_detection used as modifications): each entry names the P_FIELD
        # blob it feeds and the stencil to run on the field accumulated by ops[:op_index] (see engine._staged_torch)
        self.stages = [dict(st) for st in stages]

    @property
    def n_ops(self):
        return int(self.ops.shape[0])

    def nbytes(self):
        return int(self.ops.nbytes + self.args.nbytes)

    def disassemble(self) -> str:
        lines = []
        for i, op in enumerate(self.ops):
            code = int(op["opcode"])
            n = oc.ARG_COUNT.get(code, 0)
            off = int(op["arg"])
            if n is None:
                n = min(4, len(self.args) - off)
            a = ", ".join(f"{v:.6g}" for v in self.args[off:off + n])
            lines.append(f"{i:4d} {oc.NAMES.get(code, code):<16} a={int(op['a'])} b={int(op['b'])} [{a}]")
        return "\n".join(lines)

    # serialisation for golden fixtures / transport to the GPU box
    def to_arrays(self, prefix="prog_"):
        d = {prefix + "ops": self.ops.view(np.uint8).reshape(-1, 8).copy(), prefix + "args": self.args,
             prefix + "slots": np.array([self.n_pslots, self.n_vslots, len(self.blobs)], dtype=np.int64)}
        for i, b in enumerate(self.blobs):
            d[f"{prefix}blob{i}"] = b
        if self.stages:
            d[prefix + "stages"] = np.array([[st["blob"], st["kind"], *st["ksize"], st["iterations"], *st["res"]]
                                             for st in self.stages], dtype=np.int64)
        return d

    def stage_op_index(self, st):
        """Position of the P_FIELD op fed by stage `st`."""
        hit = np.nonzero((self.ops["opcode"] == oc.P_FIELD) & (self.ops["b"] == st["blob"]))[0]
        if hit.size != 1:
            raise ValueError("stage without a unique P_FIELD op")
        return int(hit[0])

    def prefix(self, op_index):
        """The program that stops right before ops[op_index]: its result is the field a stencil stage consumes."""
        ops = np.concatenate([self.ops[:op_index], np.array([(oc.END, 0, 0, 0)], dtype=OP_DTYPE)])
        pre = Program(ops, self.args, self.blobs, self.n_pslots, self.n_vslots,
                      [st for st in self.stages if self.stage_op_index(st) < op_index])
        pre.dargs = self.dargs  # the argument pool is shared and its offsets absolute: the same tangent applies
        return pre

    def stage_plan(self, res, slab=None, mask_planes=None):
        """Which planes each stencil stage must be computed on so that the program is exact on the x-slab `slab` of a grid
        of `res` samples (default: the whole grid). Returns (stages, final): for each stage in program order a tuple
        (stage, eval, valid), where `eval` is the plane range on which its pruned prefix program is evaluated and `valid`
        the range on which its filtered field must be exact (both None when no later program reads the stage), and `final`
        the slab itself. Ranges are half-open (lo, hi) and lie in [0, res[0]).

        The halo along x, per stage: a box filter of axis-0 size k and `it` iterations reads it * ((k - 1) // 2) planes
        below and it * (k // 2) above (the even-kernel tap placement of ab_box_filter); when k exceeds the axis, reflection
        can wrap past both faces, and the whole axis is used. The edge filter reads one plane on each side (x is a
        stencil axis in 2D and 3D). `signed` reads its field only on its own planes, but its boundary mask covers whole
        columns: its prefix is also evaluated on `mask_planes`, the planes whose mask this process packs itself (default:
        all; a sharded evaluation packs its own slab and all-gathers the rest). A stage's field must be exact on the union
        of the eval ranges of every later program whose pruned form still reads it."""
        n0 = int(res[0])
        x0, x1 = (0, n0) if slab is None else (int(slab[0]), int(slab[1]))
        if not 0 <= x0 < x1 <= n0:
            raise ValueError(f"slab ({x0}, {x1}) is not a non-empty plane range of [0, {n0})")
        m0, m1 = (0, n0) if mask_planes is None else (int(mask_planes[0]), int(mask_planes[1]))
        order = sorted(self.stages, key=self.stage_op_index)
        need = [None] * len(order)

        def widen(i, rng):
            need[i] = rng if need[i] is None else (min(need[i][0], rng[0]), max(need[i][1], rng[1]))

        def reads(prog, rng):
            live = {int(b) for c, b in zip(prog.ops["opcode"], prog.ops["b"]) if int(c) == oc.P_FIELD}
            for i, st in enumerate(order):
                if st["blob"] in live:
                    widen(i, rng)

        reads(self.pruned(), (x0, x1))
        plan = [None] * len(order)
        for i in range(len(order) - 1, -1, -1):
            st, valid = order[i], need[i]
            if valid is None:
                plan[i] = (st, None, None)
                continue
            lo, hi = valid
            if st["kind"] == 0:
                k, it = int(st["ksize"][0]), int(st["iterations"])
                lo, hi = (0, n0) if k > n0 else (lo - it * ((k - 1) // 2), hi + it * (k // 2))
            elif st["kind"] == 1:
                lo, hi = lo - 1, hi + 1
            else:
                lo, hi = min(lo, m0), max(hi, m1)
            ev = (max(lo, 0), min(hi, n0))
            plan[i] = (st, ev, valid)
            reads(self.prefix(self.stage_op_index(st)).pruned(), ev)
        return plan, (x0, x1)

    def pruned(self):
        """Dead-code elimination by one backward liveness pass over the op list (registers: the point p, the value acc,
        the P / V slots). What it is for: a stencil stage replaces a subtree's value by a P_FIELD op, but the subtree's ops
        stay in the list in front of it; every later prefix program and the final program would evaluate them again although
        P_FIELD overwrites their result. Argument offsets are absolute, so dropping ops needs no repacking."""
        ops = self.ops[:-1]
        n = len(ops)
        keep = np.zeros(n, dtype=bool)
        live_p, live_acc, live_P, live_V = False, True, set(), set()
        coord = {oc.AFFINE, oc.TRANSLATE, oc.SCALE_P, oc.ELONGATE, oc.TWIST, oc.BEND, oc.ABSX_SUB, oc.SYMMETRY, oc.ROTSYM,
                 oc.REVOLVE, oc.AXIS_REVOLVE, oc.REP_INF, oc.REP_FIN, oc.LIN_INST, oc.CURVE_INST, oc.ZERO_Z}
        unary = {oc.ROUND, oc.ABS, oc.NEG, oc.SIGN, oc.ONION, oc.CONCENTRIC, oc.SCALE_V} | set(range(oc.PP_SIGMOID, oc.PP_GAUSS_FALLOFF + 1))
        for i in range(n - 1, -1, -1):
            code, a, b = int(ops["opcode"][i]), int(ops["a"][i]), int(ops["b"][i])
            if code == oc.SAVE_P:
                if a in live_P:
                    keep[i] = True
                    live_P.discard(a)
                    live_p = True
            elif code == oc.LOAD_P:
                if live_p:
                    keep[i] = True
                    live_p = False
                    live_P.add(a)
            elif code == oc.PUSH_V:
                if a in live_V:
                    keep[i] = True
                    live_V.discard(a)
                    live_acc = True
            elif code in (oc.NEXT_AFFINE, oc.NEXT_TRANSLATE, oc.NEXT_LOAD):  # [V[b-1] = acc;] p = P[a] [transformed]
                need_v = b > 0 and (b - 1) in live_V
                if live_p or need_v:
                    keep[i] = True
                    live_p = False
                    live_P.add(a)
                    if need_v:
                        live_V.discard(b - 1)
                        live_acc = True
            elif code in coord:  # p = f(p)
                keep[i] = live_p
            elif code == oc.EXTRUDE_BEGIN:  # V[a] = |p.z| - h; p.z = 0
                if live_p or a in live_V:
                    keep[i] = True
                    live_V.discard(a)
                    live_p = True
            elif code == oc.EXTRUDE_END:  # acc = f(acc, V[a])
                if live_acc:
                    keep[i] = True
                    live_V.add(a)
            elif code == oc.POLY_SIGN:  # acc = acc * sign(P[a])
                if live_acc:
                    keep[i] = True
                    live_P.add(a)
            elif code in unary:  # acc = f(acc)
                keep[i] = live_acc
            elif oc.C_UNION <= code <= oc.C_BOLTZ_SUB:  # acc = f(V[a], acc); [V[b-1] = acc]
                need_v = b > 0 and (b - 1) in live_V
                if live_acc or need_v:
                    keep[i] = True
                    if need_v:
                        live_V.discard(b - 1)
                    live_acc = True
                    live_V.add(a)
            elif code >= oc.P_SPHERE:  # a leaf: acc = f(p) (P_FIELD reads its blob only)
                if live_acc:
                    keep[i] = True
                    live_acc = False
                    if code != oc.P_FIELD:
                        live_p = True
            else:
                raise FlattenError(f"pruned(): opcode {code} not classified")
        if keep.all():
            return self
        out = np.concatenate([ops[keep], self.ops[-1:]])
        kept = Program(out, self.args, self.blobs, self.n_pslots, self.n_vslots, list(self.stages))
        kept.dargs = self.dargs
        return kept

    @classmethod
    def from_arrays(cls, d, prefix="prog_"):
        ops = np.ascontiguousarray(d[prefix + "ops"]).view(OP_DTYPE).reshape(-1)
        slots = d[prefix + "slots"]
        blobs = [d[f"{prefix}blob{i}"] for i in range(int(slots[2]))]
        stages = []
        if prefix + "stages" in d:
            for row in np.asarray(d[prefix + "stages"]).reshape(-1, 9):
                stages.append(dict(blob=int(row[0]), kind=int(row[1]), ksize=tuple(int(v) for v in row[2:5]),
                                   iterations=int(row[5]), res=tuple(int(v) for v in row[6:9])))
        return cls(ops, d[prefix + "args"], blobs, int(slots[0]), int(slots[1]), stages)


def _vec3(v, what):
    a = np.asarray(v, dtype=np.float64).reshape(-1)
    if a.size == 1:
        a = np.repeat(a, 3)
    if a.size != 3:
        raise ValueError(f"{what} must have 3 components, got {a.size}")
    return a


def _rot2(angle):
    """[[cos, sin], [-sin, cos]] — the 2x2 block SPOMSO uses throughout (e.g. modifications.py:1020-1021)."""
    c, s = np.cos(angle), np.sin(angle)
    m = np.eye(3)
    m[0, 0], m[0, 1], m[1, 0], m[1, 1] = c, s, -s, c
    return m


def _segment_frame(a, b, what):
    """Frame of mirror / linear_instancing (modifications.py:978-985, 1058-1065)."""
    a = _vec3(a, what + " a")
    b = _vec3(b, what + " b")
    w = b - a
    c = (b + a) / 2
    l = np.linalg.norm(w)
    x = w / l
    y = np.asarray([-x[1], x[0], 0.0])
    ny = np.linalg.norm(y)
    if not np.isfinite(l) or l == 0 or ny == 0:
        raise ValueError(f"{what}: segment parallel to z (or of zero length) gives a NaN frame in the reference "
                         f"(modifications.py:982-983)")
    y = y / ny
    z = np.cross(x, y)
    rot = np.asarray([x, y, z])
    return rot, c, l


# modifications without a value part (they only warp the coordinates handed to the inner SDF)
_COORD_ONLY_MODS = frozenset((
    "elongation", "twist", "bend", "shear", "shear_xz", "shear_yz", "shear_xy", "shear_zy", "shear_yx", "shear_zx",
    "infinite_repetition", "finite_repetition", "symmetry", "mirror", "rotational_symmetry", "linear_instancing",
    "curve_instancing", "aligned_curve_instancing", "fully_aligned_curve_instancing", "revolution", "axis_revolution",
    "move_sdf", "rotate_sdf"))

_SHEAR = {  # name -> (matrix builder as in modifications.py:579-774, transpose?)
    "shear_xz": ((1, 0), True), "shear_yz": ((1, 0), False),
    "shear_xy": ((2, 0), True), "shear_zy": ((2, 0), False),
    "shear_yx": ((2, 1), True), "shear_zx": ((2, 1), False),
}


def _shear_matrix(name, p):
    t = np.tan(p["angle"])
    if name == "shear":
        sa, fa = p["sheared_axis"], p["fixed_axis"]
        table = {(0, 1): ((2, 0), True), (0, 2): ((1, 0), True), (1, 0): ((2, 1), True), (1, 2): ((1, 0), False),
                 (2, 0): ((2, 1), False), (2, 1): ((2, 0), False)}
        if (sa, fa) not in table:
            raise ValueError("Specify a valid axis index")
        (r, c), tr = table[(sa, fa)]
    else:
        (r, c), tr = _SHEAR[name]
    o = np.eye(3)
    o[r, c] = -t
    return o.T if tr else o


class _Builder:
    def __init__(self):
        self.ops = []
        self.args = []
        self.blobs = []
        self.stages = []
        self.max_p = 0
        self.max_v = 0
        self.p_alias = None  # P-slot known to hold exactly the current coordinates (lets nested combines share it)

    def emit(self, opcode, a=0, b=0, args=()):
        if opcode in (oc.SAVE_P, oc.LOAD_P):
            self.p_alias = a
        elif 8 <= opcode < 32 or opcode == oc.EXTRUDE_BEGIN:
            self.p_alias = None
        args = [float(x) for x in np.asarray(args, dtype=np.float64).reshape(-1)]
        n = oc.ARG_COUNT.get(opcode)
        if n is not None and n != len(args):
            raise AssertionError(f"{oc.NAMES[opcode]} expects {n} args, got {len(args)}")
        off = len(self.args)
        self.args.extend(args)
        self.ops.append((opcode, a, b, off))

    def use_p(self, slot):
        self.max_p = max(self.max_p, slot + 1)
        if slot >= oc.MAX_PSLOTS:
            raise FlattenError(f"combine nesting deeper than {oc.MAX_PSLOTS}")

    def use_v(self, slot):
        self.max_v = max(self.max_v, slot + 1)
        if slot >= oc.MAX_VSLOTS:
            raise FlattenError(f"value stack deeper than {oc.MAX_VSLOTS}")

    # ---- affine helpers ------------------------------------------------------------------------------------
    def affine(self, M, b):
        M = np.asarray(M, dtype=np.float64)
        b = np.asarray(b, dtype=np.float64)
        if M.shape == (3, 3) and _is_identity(M) and not np.any(b != 0):
            return  # identity node transform: emit nothing (keeps p_alias valid)
        self.emit(oc.AFFINE, args=list(M.reshape(-1)) + list(b))

    # ---- node ----------------------------------------------------------------------------------------------
    def node(self, n, pd, vd, stack=()):
        if any(n is s for s in stack):
            raise FlattenError("geometry tree contains a cycle")
        stack = stack + (n,)
        R = np.asarray(n.rotation_matrix, dtype=np.float64)
        t = np.asarray(n.center, dtype=np.float64)
        s = float(n.scale)
        if R.shape != (3, 3):
            raise ValueError(f"shapes {R.T.shape} and (3,N) not aligned")  # what the reference raises in create()
        rm = R.T
        self.affine(rm / s, -rm.dot(t))

        posts = []
        self.cur_pd = pd
        for k in range(len(n._mods) - 1, -1, -1):
            name, p = n._mods[k]
            if name in ("polygon", "shape"):
                # d * interior (geom_2d.py:415-457, 530-555): the reference first returns the field untouched if it has a
                # negative sample (a grid-wide test). The modifications applied BEFORE this one must therefore keep the
                # unsigned curve distance non-negative, i.e. be pure coordinate warps.
                bad = [m for m, _ in n._mods[:k] if m not in _COORD_ONLY_MODS]
                if bad or n.kind != "leaf":
                    raise FlattenError(f"{name}() after {bad or n.kind}: the reference decides by a grid-wide sign test "
                                       f"(np.any(d < 0)) whether to apply it; only coordinate modifications may precede it")
            post, vd = self.mod_pre(name, p, vd)
            posts.append(post)

        if n.kind == "leaf":
            self.cur_vd = vd  # first free V slot, for leaves that need a temporary
            self.leaf(n.leaf, n._geo_parameters)
        elif n.kind == "nested":
            self.node(n.inner, pd, vd, stack)
        elif n.kind == "combine":
            self.combine(n, pd, vd, stack)
        else:
            raise FlattenError(f"unknown node kind {n.kind}")

        for post in reversed(posts):
            for (code, a, args) in post:
                if code == oc.P_FIELD:
                    self.emit(code, b=a)
                elif code == oc.POLY_SIGN:
                    self.emit(code, a=a[0], b=a[1], args=args)
                else:
                    self.emit(code, a=a, args=args)
        if s != 1.0:
            self.emit(oc.SCALE_V, args=[s])

    def combine(self, n, pd, vd, stack):
        op, kids, w = n.combine_op, tuple(n.children), n.combine_parameter
        binary = {"UNION2": oc.C_UNION, "SUBTRACT2": oc.C_SUBTRACT, "INTERSECT2": oc.C_INTERSECT, "SUM": oc.C_SUM,
                  "DIFFERENCE": oc.C_DIFF}
        nary = {"UNION": oc.C_UNION, "INTERSECT": oc.C_INTERSECT}
        param = {"SMOOTH_UNION2_2": oc.C_SMIN2, "SMOOTH_UNION2": oc.C_SMIN3, "SMOOTH_INTERSECT2": oc.C_SMAX3,
                 "SMOOTH_INTERSECT2_BOLTZMANN": oc.C_BOLTZ_INT, "SMOOTH_SUBTRACT2": oc.C_SSUB3,
                 "SMOOTH_SUBTRACT2_BOLTZMANN": oc.C_BOLTZ_SUB}
        args = ()
        if op in binary or op in param:
            if len(kids) != 2:  # the reference's 2-argument lambdas raise TypeError (combine.py:51-78)
                raise TypeError(f"{op} takes exactly 2 objects, {len(kids)} given")
            code = binary.get(op, param.get(op))
            if op in param:
                w = float(np.asarray(w, dtype=np.float64).reshape(-1)[0]) if np.ndim(w) else float(w)
                args = (w,)
                if w == 0.0 and code in (oc.C_SMIN2, oc.C_SMIN3, oc.C_SMAX3, oc.C_SSUB3):
                    # smoothmin_poly*(x, y, 0) returns plain min (combine.py:14,22)
                    code = {oc.C_SMIN2: oc.C_UNION, oc.C_SMIN3: oc.C_UNION, oc.C_SMAX3: oc.C_INTERSECT,
                            oc.C_SSUB3: oc.C_SUBTRACT}[code]
                    args = ()
                elif w == 0.0:
                    raise ZeroDivisionError("smoothmax_boltz with width 0 (combine.py:31)")
        elif op in nary:
            if len(kids) == 0:
                raise TypeError(f"{op} needs at least one object")
            code = nary[op]
        else:
            raise SyntaxError(f"{op} is not an implemented operation.")

        slot, nxt = pd, pd + 1
        if len(kids) > 1:
            if self.p_alias is not None:
                slot, nxt = self.p_alias, pd  # current p already sits in a live slot: share it, save nothing
            else:
                self.use_p(pd)
                self.emit(oc.SAVE_P, a=pd)
        self.node(kids[0], nxt, vd, stack)
        for k in kids[1:]:
            self.use_v(vd)
            self.emit(oc.PUSH_V, a=vd)
            self.emit(oc.LOAD_P, a=slot)
            self.node(k, nxt, vd + 1, stack)
            self.emit(code, a=vd, args=args)

    # ---- modifications -------------------------------------------------------------------------------------
    def mod_pre(self, name, p, vd):
        """Emits the coordinate part of a modification now; returns (value part as [(opcode, a, args)], new vd)."""
        post = []
        if name == "elongation":
            ev = np.asarray(p["ev"], dtype=np.float64).reshape(-1)
            if ev.size < 3:
                raise IndexError("elongation vector needs 3 components (modifications.py:91-93)")
            self.emit(oc.ELONGATE, args=list(-ev[:3] / 2) + list(ev[:3] / 2))
        elif name == "twist":
            self.emit(oc.TWIST, args=[p["pitch"]])
        elif name == "bend":
            r, ang = float(p["radius"]), float(p["angle"])
            c, s = np.cos(ang / 2), np.sin(ang / 2)
            self.emit(oc.BEND, args=[r, ang / 2, c, s, r * ang / 2, r * s, r * (1 - c), r * (ang / 2)])
        elif name in _SHEAR or name == "shear":
            self.affine(_shear_matrix(name, p), np.zeros(3))
        elif name == "infinite_repetition":
            d = _vec3(p["distances"], "distances")
            if np.any(d == 0):
                raise ZeroDivisionError("infinite_repetition distance of 0 (np.mod by zero, modifications.py:820)")
            self.emit(oc.REP_INF, args=list(d) + list(d / 2))
        elif name in ("finite_repetition", "finite_repetition_rescaled"):
            size = _vec3(p["size"], "size")
            rep = _vec3(p["rep"], "repetitions")
            c = size * (1 - 1 / rep) / 2
            d = size * (1 / 2 - 1 / rep)
            s = size / rep
            self.emit(oc.REP_FIN, args=list(c) + list(d) + list(s) + list(s / 2))
            if name == "finite_repetition_rescaled":
                sss = float(np.min(s / (_vec3(p["f"], "instance_size") + _vec3(p["padding"], "padding"))))
                self.emit(oc.SCALE_P, args=[1.0 / sss])
                post.append((oc.SCALE_V, 0, [sss]))
        elif name == "symmetry":
            axis = int(p["axis"])
            if axis == 3 or axis < -3:
                raise IndexError(f"index {axis} is out of bounds for axis 0 with size 3")  # modifications.py:951
            if axis < 3:  # axis > 3 is a no-op in the reference (:948-949)
                self.emit(oc.SYMMETRY, a=axis % 3)
        elif name == "mirror":
            rot, c, l = _segment_frame(p["a"], p["b"], "mirror")
            self.affine(rot, -rot.dot(c))
            self.emit(oc.ABSX_SUB, args=[l / 2])
        elif name == "rotational_symmetry":
            angle = float(p["angle"])
            self.affine(_rot2(angle / 2 - p["phase"]), np.zeros(3))
            # args: angle, radius, number of sectors, pad, then (cos, sin) of every sector's centre direction
            # theta_k = k*angle + angle/2: the kernel picks the sector from atan2 and rotates by the exact table entry
            # instead of going through mod / cos / sin of the reduced angle (same map, fewer roundings)
            nsec = int(np.ceil(2 * np.pi / abs(angle) - 1e-9))
            if nsec < 1 or nsec > 1024 or not angle > 0:
                raise FlattenError(f"rotational_symmetry order {2 * np.pi / angle:g} is outside [1, 1024]")
            th = (np.arange(nsec) + 0.5) * angle
            tab = np.stack([np.cos(th), np.sin(th)], axis=1).reshape(-1)
            self.emit(oc.ROTSYM, args=[angle, p["radius"], float(nsec), 0.0] + list(tab))
        elif name == "linear_instancing":
            rot, c, l = _segment_frame(p["a"], p["b"], "linear_instancing")
            n = int(p["n"])
            if n < 2:
                raise ZeroDivisionError("linear_instancing needs n >= 2 (modifications.py:1069 divides by n-1)")
            s = l / (n - 1)
            d = s / 2
            self.affine(rot, -rot.dot(c))
            self.emit(oc.LIN_INST, a=1 if n > 2 else 0, args=[l / 2, s, d, -l / 2 + d, l / 2 - d, l / 2 - d])
        elif name in ("curve_instancing", "aligned_curve_instancing", "fully_aligned_curve_instancing"):
            self.curve_instancing(name, p)
        elif name == "revolution":
            self.emit(oc.REVOLVE, args=[p["radius"]])
        elif name == "axis_revolution":
            self.emit(oc.AXIS_REVOLVE, args=[p["radius"], np.cos(p["angle"]), np.sin(p["angle"])])
        elif name == "move_sdf":
            self.emit(oc.TRANSLATE, args=list(-_vec3(p["move_vector"], "move_vector")))
        elif name == "scale_sdf":
            k = float(p["scale_factor"])
            self.emit(oc.SCALE_P, args=[1.0 / k])
            post.append((oc.SCALE_V, 0, [k]))
        elif name == "rotate_sdf":
            self.affine(np.asarray(p["rotation_matrix"], dtype=np.float64).T, np.zeros(3))
        elif name == "rounding":
            post.append((oc.ROUND, 0, [p["rounding_radius"]]))
        elif name == "rounding_cs":
            k = max(1 - 2 * p["rounding_radius"] / p["bb_size"] + 1e-8, 1e-8)
            self.emit(oc.SCALE_P, args=[1.0 / k])
            post.append((oc.SCALE_V, 0, [k]))
            post.append((oc.ROUND, 0, [p["rounding_radius"]]))
        elif name == "boundary":
            post.append((oc.ABS, 0, []))
        elif name == "invert":
            post.append((oc.NEG, 0, []))
        elif name == "sign":
            post.append((oc.SIGN, 0, []))
        elif name == "onion":
            post.append((oc.ONION, 0, [p["thickness"]]))
        elif name == "concentric":
            post.append((oc.CONCENTRIC, 0, [p["width"] / 2]))
        elif name == "extrusion":
            self.use_v(vd)
            self.emit(oc.EXTRUDE_BEGIN, a=vd, args=[p["distance"] / 2])
            post.append((oc.EXTRUDE_END, vd, []))
            vd += 1
        elif name == "sigmoid_falloff":
            post.append((oc.PP_SIGMOID, 0, [p["amplitude"], p["width"]]))
        elif name == "positive_sigmoid_falloff":
            post.append((oc.PP_POS_SIGMOID, 0, [p["amplitude"], p["width"]]))
        elif name == "capped_exponential":
            post.append((oc.PP_CAPPED_EXP, 0, [p["amplitude"], p["width"]]))
        elif name == "hard_binarization":
            post.append((oc.PP_HARD_BIN, 0, [p["threshold"]]))
        elif name == "linear_falloff":
            post.append((oc.PP_LINEAR, 0, [p["amplitude"], p["width"]]))
        elif name == "relu":
            post.append((oc.PP_RELU, 0, [p["width"]]))
        elif name == "smooth_relu":
            b = (p["smooth_width"] + p["threshold"]) * 4 * p["threshold"]
            post.append((oc.PP_SMOOTH_RELU, 0, [b, p["width"]]))
        elif name == "slowstart":
            b = (2 * p["smooth_width"] + p["threshold"]) * p["threshold"]
            bw = b / p["width"]
            post.append((oc.PP_SLOWSTART, 0, [p["width"], bw, np.sqrt(bw) * bool(p["ground"])]))
        elif name == "gaussian_boundary":
            post.append((oc.PP_GAUSS_BOUNDARY, 0, [p["amplitude"], p["width"]]))
        elif name == "gaussian_falloff":
            post.append((oc.PP_GAUSS_FALLOFF, 0, [p["amplitude"], p["width"]]))
        elif name in ("polygon", "shape"):
            slot = self.cur_pd
            self.use_p(slot)
            self.emit(oc.SAVE_P, a=slot)  # the coordinates this closure receives (after the outer warps, before the inner ones)
            if name == "polygon":  # interior_polygon(co, self._points): triangulation_functions.py:390-430
                pts = np.asarray(p["points"], dtype=np.float64)
                if pts.ndim != 2 or pts.shape[0] != 3:
                    raise ValueError("operands could not be broadcast together: polygon() subtracts the control points "
                                     "from 3-row coordinates (triangulation_functions.py:385), points must have shape (3, N)")
                pts = pts[:2]
                if pts.shape[1] < 3:
                    raise ValueError("polygon() needs at least 3 points")
                if _polygon_self_intersects(pts):
                    raise FlattenError("self-intersecting polygons (split into loops by the reference, "
                                       "triangulation_functions.py:413-419) are not supported on the GPU path")
                post.append((oc.POLY_SIGN, (slot, 0), [float(pts.shape[1])] + list(pts.T.reshape(-1))))
            else:  # ParametricCurve.shape(): geom_2d.py:435-452, segment by segment
                pts = np.asarray(p["points"], dtype=np.float64)
                rec = []
                for i in range(pts.shape[1] - 1):
                    t = pts[:, i + 1] - pts[:, i]
                    t = t / np.linalg.norm(t)
                    nx, ny = -t[1], abs(t[0])  # n[1] = n[1] - 2 (n[1] < 0) n[1]: only the y component is made positive
                    lx, ux = min(pts[0, i], pts[0, i + 1]), max(pts[0, i], pts[0, i + 1])
                    rec += [pts[0, i], pts[1, i], lx, ux, nx, ny]
                if not np.all(np.isfinite(rec)):
                    raise ValueError("shape(): the sampled curve has a zero-length segment (NaN normal in the reference)")
                post.append((oc.POLY_SIGN, (slot, 1), [float(pts.shape[1] - 1)] + rec))
        elif name == "signed":
            # modifications.py:220-275: a whole-grid post-pass (scans + box filter), staged like the convolutions below
            res = tuple(int(r) for r in np.asarray(p["co_resolution"]).reshape(-1))
            if len(res) != 3:
                raise IndexError("too many indices for array: signed() slices the reshaped field with three indices "
                                 "(modifications.py:244), co_resolution must have 3 entries")
            if len(self.blobs) >= oc.MAX_BLOBS:
                raise FlattenError(f"more than {oc.MAX_BLOBS} blobs (point clouds + stencil stages) in one tree")
            self.blobs.append(np.zeros((1, 0)))
            b = len(self.blobs) - 1
            self.stages.append(dict(blob=b, kind=2, ksize=(2, 2, 1), iterations=1, res=res))
            post.append((oc.P_FIELD, b, []))
        elif name in ("conv_averaging", "conv_edge_detection"):
            # grid stencils (modifications.py:1586-1637): the field accumulated so far is filtered on the grid by
            # a separate kernel and comes back through a P_FIELD op; engine.create runs the stages in order
            res = tuple(int(r) for r in np.asarray(p["co_resolution"]).reshape(-1))
            if len(res) not in (2, 3):
                raise FlattenError(f"{name}: co_resolution must have 2 or 3 entries")
            if name == "conv_averaging":
                ks = p["kernel_size"]
                ks = (int(ks),) * len(res) if isinstance(ks, (int, np.integer)) else tuple(int(k) for k in np.asarray(ks).reshape(-1))
                if len(ks) != len(res):
                    raise ValueError("Dimension of the kernel and the field must match!")
                its = int(p["iterations"])
            else:
                ks, its = (3, 3) + ((1,) if len(res) == 3 else ()), 1
            if len(self.blobs) >= oc.MAX_BLOBS:
                raise FlattenError(f"more than {oc.MAX_BLOBS} blobs (point clouds + stencil stages) in one tree")
            if not (name == "conv_averaging" and its == 0):  # iterations == 0 returns the field untouched
                self.blobs.append(np.zeros((1, 0)))
                b = len(self.blobs) - 1
                self.stages.append(dict(blob=b, kind=0 if name == "conv_averaging" else 1,
                                        ksize=tuple(ks) + (1,) * (3 - len(ks)), iterations=its,
                                        res=tuple(res) + (0,) * (3 - len(res))))
                post.append((oc.P_FIELD, b, []))
        else:
            raise FlattenError(f"modification '{name}' cannot enter the GPU op list")
        return post, vd

    def curve_instancing(self, name, p):
        """Evaluates the user's curve callable on the host and uploads the instance table
        (modifications.py:1110-1118, 1158-1181, 1222-1251)."""
        f, fp, t_range = p["f"], p["f_parameters"], p["t_range"]
        n = int(t_range[-1])
        ts = np.linspace(*t_range)
        fval = np.asarray(f(ts, *fp), dtype=np.float64)
        va = np.zeros((3, n))
        va[:fval.shape[0]] = fval
        if name == "curve_instancing":
            rec = va.T.reshape(-1)
            mode = 0
        else:
            tol = p.get("tol", 0.001)
            fv_min = np.asarray(f(ts - tol, *fp), dtype=np.float64)
            fv_max = np.asarray(f(ts + tol, *fp), dtype=np.float64)
            der = (fv_max - fv_min) / (2 * tol)
            dermag = np.linalg.norm(der, axis=0)
            der = der / dermag
            dx = np.zeros((3, n))
            dx[:fval.shape[0]] = der
            dy = np.zeros((3, n))
            if name == "aligned_curve_instancing":
                dy[0, :] = -dx[1]
                dy[1, :] = dx[0]
            else:
                der2 = (fv_max - 2 * fval + fv_min) / (tol ** 2)
                der2 = der2 / dermag
                der2 = der2 / np.linalg.norm(der2, axis=0)
                dy[:fval.shape[0]] = der2
            dz = np.cross(dx.T, dy.T).T
            rec = np.concatenate([va.T, dx.T, dy.T, dz.T], axis=1).reshape(-1)  # per instance: pos, dx, dy, dz
            mode = 1
        if not np.all(np.isfinite(rec)):
            raise ValueError(f"{name}: the curve frame contains NaN/inf (degenerate tangent or normal)")
        self.emit(oc.CURVE_INST, a=mode, args=[float(n), 0.0, 0.0, 0.0] + list(rec))  # 4-entry header: 16-byte aligned records

    # ---- leaves --------------------------------------------------------------------------------------------
    def leaf(self, name, params):
        e = self.emit
        if name in ("sdf_x", "sdf_y", "sdf_z"):
            e(oc.P_AXIS, a="xyz".index(name[-1]), args=[params[0]])
        elif name == "sdf_sphere":
            e(oc.P_SPHERE, args=[params[0]])
        elif name == "sdf_cylinder":
            e(oc.P_CYLINDER, args=[params[0], params[1] / 2])
        elif name == "sdf_box":
            e(oc.P_BOX, args=_vec3(params[0], "box size") / 2)
        elif name == "sdf_torus":
            e(oc.P_TORUS, args=[params[0], params[1]])
        elif name == "sdf_chainlink":
            e(oc.P_CHAINLINK, args=[params[0], params[1], params[2] / 2])
        elif name == "sdf_braid":
            e(oc.P_BRAID, args=[params[0] / 2, params[1], params[2], params[3]])
        elif name == "sdf_arc_3d":
            R, r, sa, ea = params
            ca = (sa + ea) / 2
            e(oc.P_ARC3D, args=[R, r, np.cos(ca), np.sin(ca), np.abs(ea - ca)])
        elif name in ("sdf_plane", "sudf_plane"):
            nrm = _vec3(params[0], "normal")
            nrm = nrm / np.linalg.norm(nrm)
            if name == "sdf_plane":
                e(oc.P_PLANE, args=list(nrm) + [params[1]])
            else:
                e(oc.P_UPLANE, args=list(nrm) + [params[1] / 2])
        elif name == "sdf_segment_3d":
            a = _vec3(params[0], "a")
            ba = _vec3(params[1], "b") - a
            e(oc.P_SEGMENT, args=list(a) + list(ba) + [np.dot(ba, ba)])
        elif name == "sdf_cone":
            h, ang = params
            q = np.asarray((np.tan(ang), -1.0)) * h
            e(oc.P_CONE, args=[q[0], q[1], h * (0.5 ** (1 / 3)), np.dot(q, q)])
        elif name in ("sdf_oriented_infinite_cone", "sdf_infinite_cone"):
            ang = params[0]
            e(oc.P_OINF_CONE if name == "sdf_oriented_infinite_cone" else oc.P_INF_CONE,
              args=[np.sin(ang), np.cos(ang)])
        elif name in ("sdf_solid_angle", "sdf_sector"):
            radius, a1, a2 = params
            ad = np.abs(a2 - a1) / 2
            ca = (a2 + a1) / 2
            e(oc.P_SOLID_ANGLE if name == "sdf_solid_angle" else oc.P_SECTOR,
              args=[radius, np.cos(ca), np.sin(ca), ad, np.cos(ad), np.sin(ad)])
        elif name == "sdf_inf_sector":
            a1, a2 = params
            ad = np.abs(a2 - a1) / 2
            ca = (a2 + a1) / 2
            e(oc.P_INF_SECTOR, args=[np.cos(ca), np.sin(ca), ad, np.cos(ad), np.sin(ad)])
        elif name == "sdf_triangle_3d":
            a, b, c = (_vec3(v, "vertex") for v in params)
            s1, s2, s3 = b - a, c - b, a - c
            nrm = np.cross(s1, s3)
            e(oc.P_TRIANGLE3D, args=np.concatenate([
                a, b, c, s1, s2, s3, nrm, np.cross(s1, nrm), np.cross(s2, nrm), np.cross(s3, nrm),
                [np.dot(s1, s1), np.dot(s2, s2), np.dot(s3, s3), np.dot(nrm, nrm)]]))
        elif name == "sdf_quad_3d":
            a, b, c, d = (_vec3(v, "vertex") for v in params)
            s1, s2, s3, s4 = b - a, c - b, d - c, a - d
            nrm = np.cross(s1, s4)
            e(oc.P_QUAD3D, args=np.concatenate([
                a, b, c, d, s1, s2, s3, s4, nrm, np.cross(s1, nrm), np.cross(s2, nrm), np.cross(s3, nrm),
                np.cross(s4, nrm), [np.dot(s1, s1), np.dot(s2, s2), np.dot(s3, s3), np.dot(s4, s4)],
                [np.dot(nrm, nrm)]]))
        elif name in ("sdf_segmented_line_3d", "sdf_closed_segmented_line_3d"):
            pts = np.asarray(params[0], dtype=np.float64)
            if pts.shape[0] != 3:
                raise ValueError("3D segmented line needs points of shape (3, N)")
            if name.startswith("sdf_closed"):  # min(f1, segment(p0, p_last)), geom_3d.py:739-744
                pts = np.concatenate([pts, pts[:, :1]], axis=1)
            e(oc.P_SEGLINE, args=[float(pts.shape[1])] + list(pts.T.reshape(-1)))
        elif name in ("sdf_segmented_line_2d", "sdf_closed_segmented_line_2d"):
            pts = np.asarray(params[0], dtype=np.float64)[:2]
            if name.startswith("sdf_closed"):
                pts = np.concatenate([pts, pts[:, :1]], axis=1)
            e(oc.P_SEGLINE2D, args=[float(pts.shape[1])] + list(pts.T.reshape(-1)))
        elif name == "sdf_polygon_2d":
            pts = np.asarray(params[0], dtype=np.float64)
            if pts.ndim != 2 or 3 not in pts.shape:
                raise ValueError("The coordinates of vertices should be defined in 3D space.")
            if pts.shape[0] != 3:
                pts = pts.T
            pts = pts[:2]
            if pts.shape[1] < 3:
                raise ValueError("There must be at least 3 vertices defined by their coordinates in 3D space.")
            if _polygon_self_intersects(pts):
                raise FlattenError("self-intersecting polygons (split into loops by the reference, "
                                   "triangulation_functions.py:413-419) are not supported on the GPU path")
            e(oc.P_POLYGON2D, args=[float(pts.shape[1])] + list(pts.T.reshape(-1)))
        elif name in ("sdf_parametric_curve_2d", "sdf_parametric_curve_3d", "sdf_closed_parametric_curve_2d",
                      "sdf_closed_parametric_curve_3d"):
            # nearest SAMPLE of the curve (a KD-tree over f(t) in the reference, sdf_2D.py:215-218, sdf_3D.py:274-280):
            # the user's callable is evaluated here on the host and the samples become a point cloud blob
            f, fp, ts = params
            dim = 3 if name.endswith("3d") else 2
            fval = np.asarray(f(np.asarray(ts), *fp), dtype=np.float64)
            if fval.ndim != 2 or fval.shape[0] < dim:
                raise ValueError(f"parametric curve must return an array of shape ({dim}, len(t))")
            self.leaf(f"sdf_point_cloud_{dim}d", (fval[:dim],))
            if name.startswith("sdf_closed"):  # min(f1, segment(p0, p1)), geom_2d.py:377-383 / geom_3d.py:606-612
                p0 = np.asarray(f(ts[0], *fp), dtype=np.float64).reshape(-1)
                p1 = np.asarray(f(ts[-1], *fp), dtype=np.float64).reshape(-1)
                slot = self.cur_vd
                self.use_v(slot)
                e(oc.PUSH_V, a=slot)
                if dim == 3:
                    self.leaf("sdf_segment_3d", (p0[:3], p1[:3]))
                else:
                    self.leaf("sdf_segment_2d", (p0[:2], p1[:2]))
                e(oc.C_UNION, a=slot)
        elif name in ("sdf_segmented_curve_2d", "sdf_segmented_curve_3d", "sdf_closed_segmented_curve_2d",
                      "sdf_closed_segmented_curve_3d"):
            # nearest SAMPLE of the polyline, interpolated on the host exactly as sdf_2D.py:180-188 / sdf_3D.py:253-261
            pts, ts = np.asarray(params[0], dtype=np.float64), np.asarray(params[1], dtype=np.float64)
            dim = 3 if name.endswith("3d") else 2
            if pts.ndim != 2 or pts.shape[0] < dim:
                raise ValueError(f"points must have shape ({dim}, M)")
            v = np.floor(ts).astype(int)
            u = ts - v
            fval = pts[:dim, v + 1] * u + pts[:dim, v] * (1 - u)
            self.leaf(f"sdf_point_cloud_{dim}d", (fval,))
            if name.startswith("sdf_closed"):  # min(f1, segment(first, last)), geom_2d.py:491-496 / geom_3d.py:677-682
                slot = self.cur_vd
                self.use_v(slot)
                e(oc.PUSH_V, a=slot)
                self.leaf(f"sdf_segment_{dim}d", (pts[:dim, 0], pts[:dim, -1]))
                e(oc.C_UNION, a=slot)
        elif name in ("sdf_point_cloud_3d", "sdf_point_cloud_2d"):
            pts = np.asarray(params[0], dtype=np.float64)
            dim = 3 if name.endswith("3d") else 2
            if pts.ndim != 2 or pts.shape[0] < dim:
                raise ValueError(f"point cloud must have shape ({dim}, M)")
            if len(self.blobs) >= oc.MAX_BLOBS:
                raise FlattenError(f"more than {oc.MAX_BLOBS} point clouds in one tree")
            cloud = np.zeros((3, pts.shape[1]))
            cloud[:dim] = pts[:dim]
            self.blobs.append(cloud)
            e(oc.P_POINT_CLOUD, a=dim, b=len(self.blobs) - 1)
        elif name == "sdf_circle":
            e(oc.P_CIRCLE, args=[params[0]])
        elif name == "sdf_neu_circle":
            order = float(params[1])
            if not (order > 0):
                raise FlattenError("sdf_neu_circle: only norm orders > 0 (or inf) are supported")
            e(oc.P_NEU_CIRCLE, args=[params[0], order])
        elif name == "sdf_box_2d":
            v = np.asarray(params[0], dtype=np.float64).reshape(-1) / 2
            e(oc.P_BOX2D, args=v[:2])
        elif name == "sdf_segment_2d":
            a = np.asarray(params[0], dtype=np.float64).reshape(-1)[:2]
            ba = np.asarray(params[1], dtype=np.float64).reshape(-1)[:2] - a
            e(oc.P_SEGMENT2D, args=list(a) + list(ba) + [np.dot(ba, ba)])
        elif name == "sdf_rounded_box_2d":
            v = np.asarray(params[0], dtype=np.float64).reshape(-1) / 2
            r = np.asarray(params[1], dtype=np.float64).reshape(-1)
            e(oc.P_RBOX2D, args=list(v[:2]) + list(r[:4]))
        elif name == "sdf_triangle_2d":
            p0, p1, p2 = (np.asarray(v, dtype=np.float64).reshape(-1) for v in params)
            if p0.size != 2 or p1.size != 2 or p2.size != 2:
                raise ValueError("operands could not be broadcast together: Triangle takes 2-vectors "
                                 "(sdf_2D.py:66)")
            e0, e1, e2 = p1 - p0, p2 - p1, p0 - p2
            s = np.sign(e0[0] * e2[1] - e0[1] * e2[0])
            e(oc.P_TRIANGLE2D, args=np.concatenate([p0, p1, p2, e0, e1, e2,
                                                    [np.dot(e0, e0), np.dot(e1, e1), np.dot(e2, e2), s]]))
        elif name == "sdf_arc":
            radius, sa, ea = params
            ca = (sa + ea) / 2
            e(oc.P_ARC, args=[radius, np.cos(ca), np.sin(ca), np.abs(ea - ca)])
        elif name == "sdf_ngon":
            radius, n = params
            beta = np.pi * (0.5 - 1 / n)
            alpha = 2 * np.pi / n
            s, c = np.sin(beta), np.cos(beta)
            e(oc.P_NGON, args=[radius, alpha, -c, s, s, c, 2 * radius * np.sin(alpha / 2)])
        else:
            raise FlattenError(f"primitive '{name}' cannot enter the GPU op list")


def _polygon_self_intersects(pts):
    """True if two non-adjacent edges of the closed polygon properly intersect (O(n^2), host side)."""
    n = pts.shape[1]

    def orient(a, b, c):
        return np.sign((b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0]))

    for i in range(n):
        a, b = pts[:, i], pts[:, (i + 1) % n]
        for j in range(i + 1, n):
            if j == i or (j + 1) % n == i or (i + 1) % n == j:
                continue
            c, d = pts[:, j], pts[:, (j + 1) % n]
            if orient(a, b, c) * orient(a, b, d) < 0 and orient(c, d, a) * orient(c, d, b) < 0:
                return True
    return False


def _is_identity(M):
    return np.array_equal(M, np.eye(3))


def _peephole(ops, args, fold_frames=True):
    """Composes runs of AFFINE / TRANSLATE / SCALE_P into a single op (exact in fp64 up to rounding). With fold_frames
    the linear part of a run that directly follows an aligned curve instancing is multiplied into the instance frames
    (p' = M R_j (p - o_j) + b: the rows of every record become M R_j, only the translation stays an op): one 3 x 3
    map per point less, and one pull-back less in the gradient kernels."""
    out_ops, out_args = [], []

    def put(code, a, b, vals):
        out_ops.append((code, a, b, len(out_args)))
        out_args.extend(vals)

    pending = None  # (M, b)

    def flush():
        nonlocal pending
        if pending is None:
            return
        M, b = pending
        pending = None
        if fold_frames and out_ops and out_ops[-1][0] == oc.CURVE_INST and out_ops[-1][1] == 1 and not _is_identity(M):
            off = out_ops[-1][3]
            n = int(out_args[off])
            rec = np.asarray(out_args[off + 4:off + 4 + 12 * n], dtype=np.float64).reshape(n, 12)
            rec[:, 3:] = np.einsum("ij,njk->nik", M, rec[:, 3:].reshape(n, 3, 3)).reshape(n, 9)
            out_args[off + 4:off + 4 + 12 * n] = list(rec.reshape(-1))
            M = np.eye(3)
        if _is_identity(M):
            if np.any(b != 0):
                put(oc.TRANSLATE, 0, 0, list(b))
        elif np.all(b == 0) and np.array_equal(M, np.eye(3) * M[0, 0]):
            put(oc.SCALE_P, 0, 0, [M[0, 0]])
        else:
            put(oc.AFFINE, 0, 0, list(M.reshape(-1)) + list(b))

    for (code, a, b, off) in ops:
        if code in (oc.AFFINE, oc.TRANSLATE, oc.SCALE_P):
            if code == oc.AFFINE:
                M2 = np.asarray(args[off:off + 9]).reshape(3, 3)
                b2 = np.asarray(args[off + 9:off + 12])
            elif code == oc.TRANSLATE:
                M2, b2 = np.eye(3), np.asarray(args[off:off + 3])
            else:
                M2, b2 = np.eye(3) * args[off], np.zeros(3)
            if pending is None:
                pending = (M2, b2)
            else:
                M1, b1 = pending  # p1 = M1 p + b1 ; p2 = M2 p1 + b2
                pending = (M2 @ M1, M2 @ b1 + b2)
            continue
        flush()
        n = oc.ARG_COUNT.get(code)
        if n is None:
            cnt = int(args[off])
            if code == oc.ROTSYM:
                n = 4 + 2 * int(args[off + 2])
            elif code == oc.CURVE_INST:
                n = 4 + cnt * (12 if a == 1 else 3)
            elif code == oc.P_SEGLINE:
                n = 1 + cnt * 3
            elif code in (oc.P_SEGLINE2D, oc.P_POLYGON2D):
                n = 1 + cnt * 2
            elif code == oc.POLY_SIGN:
                n = 1 + cnt * (6 if b else 2)
        put(code, a, b, args[off:off + n])
    flush()
    return out_ops, out_args


_COMBINES = (oc.C_UNION, oc.C_INTERSECT, oc.C_SUBTRACT, oc.C_SUM, oc.C_DIFF, oc.C_SMIN2, oc.C_SMIN3, oc.C_SMAX3,
             oc.C_SSUB3, oc.C_BOLTZ_INT, oc.C_BOLTZ_SUB)


def _fuse(ops):
    """Superinstructions: every dispatch costs the interpreter ~20 issue slots per thread, so the recurring sequences of
    a combine chain are folded into one op each:
        [PUSH_V v] LOAD_P s, AFFINE|TRANSLATE   ->  NEXT_AFFINE|NEXT_TRANSLATE (a = s, b = v + 1 or 0)
        [PUSH_V v] LOAD_P s                     ->  NEXT_LOAD
        C_xxx (a = v), PUSH_V w                 ->  C_xxx (a = v, b = w + 1)
    Argument offsets are untouched (the fused op keeps the transform's arguments)."""
    out, i = [], 0
    while i < len(ops):
        code, a, b, off = ops[i]
        nxt = ops[i + 1] if i + 1 < len(ops) else None
        nn = ops[i + 2] if i + 2 < len(ops) else None
        if code == oc.PUSH_V and nxt is not None and nxt[0] == oc.LOAD_P:
            if nn is not None and nn[0] in (oc.AFFINE, oc.TRANSLATE):
                out.append((oc.NEXT_AFFINE if nn[0] == oc.AFFINE else oc.NEXT_TRANSLATE, nxt[1], a + 1, nn[3]))
                i += 3
            else:
                out.append((oc.NEXT_LOAD, nxt[1], a + 1, 0))
                i += 2
            continue
        if code == oc.LOAD_P and nxt is not None and nxt[0] in (oc.AFFINE, oc.TRANSLATE):
            out.append((oc.NEXT_AFFINE if nxt[0] == oc.AFFINE else oc.NEXT_TRANSLATE, a, 0, nxt[3]))
            i += 2
            continue
        if code in _COMBINES and b == 0 and nxt is not None and nxt[0] == oc.PUSH_V:
            out.append((code, a, nxt[1] + 1, off))
            i += 2
            continue
        out.append(ops[i])
        i += 1
    return out


def flatten(obj, optimize=True, fold_frames=True) -> Program:
    """Flattens a frontend.GenericGeometry tree (or a SPOMSO object, via introspect.to_frontend). fold_frames=False keeps
    an affine map that follows an aligned curve instancing as its own op (program_tangent needs that: tables carry no
    parameter tangents, the affine's arguments do)."""
    from .frontend import GenericGeometry
    if not isinstance(obj, GenericGeometry):
        from .introspect import to_frontend
        obj = to_frontend(obj)
    b = _Builder()
    b.node(obj, 0, 0)
    ops, args = b.ops, b.args
    if optimize:
        ops, args = _peephole(ops, args, fold_frames)
        ops = _fuse(ops)
    ops.append((oc.END, 0, 0, 0))
    if len(ops) > oc.MAX_OPS or len(args) > oc.MAX_ARGS:
        raise FlattenError(f"program too large: {len(ops)} ops / {len(args)} args "
                           f"(limits {oc.MAX_OPS} / {oc.MAX_ARGS})")
    arr = np.array(ops, dtype=OP_DTYPE)
    prog = Program(arr, np.asarray(args, dtype=np.float64), b.blobs, max(b.max_p, 1), max(b.max_v, 1), b.stages)
    prog.stages.sort(key=prog.stage_op_index)  # evaluation order (modifications are visited outermost first)
    return prog
