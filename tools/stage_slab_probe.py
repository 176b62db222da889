"""Measures the slab pipeline of trees with grid-stencil stages on the GPU, in one call:

  1. whole-grid ab_signed_field on a 513^3 fp32 field: this library against a baseline build of the library
     (--baseline-lib, e.g. the previous release), alternated in the same run, outputs compared bit for bit;
  2. whole-grid staged evaluation against the sum of its slab evaluations at 2 and 8 slabs (the halo recompute
     overhead), for the averaged tree of tests/scenarios.py (stencil_conv_averaging_tree3d) at 513^3 and the averaged
     2D point cloud (stencil_conv_averaging_cloud2d) at 4097^2;
  3. with more than one GPU: evaluate_sharded of those trees over every GPU (re-launched under torch.distributed.run).

Times are CUDA-event times of the device work on the current stream (median of --reps after a warm-up). Prints the
card's name and power limit first and one JSON line per measurement.

    python tools/stage_slab_probe.py [--baseline-lib PATH] [--reps 10] [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def tree3d(r):
    import aegolius_b200 as ab
    s = ab.Sphere(1.1)
    s.move((0.4, -0.2, 0.3))
    s.conv_averaging((2, 3, 4), 2, (r, r, r))
    s.rounding(0.05)
    b = ab.Box(1.6, 1.0, 2.0)
    b.rotate(0.5, (0, 1, 0))
    u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=0.3)
    u.conv_averaging(3, 1, (r, r, r))
    return ab.flatten(u), ab.GridSpec((4.0, 4.0, 4.0), (r, r, r))


def cloud2d(r):
    import numpy as np
    import aegolius_b200 as ab
    rng = np.random.default_rng(12)
    t = rng.uniform(0, 2 * np.pi, 60)
    pc = ab.PointCloud2D(np.stack([2.2 * np.cos(t), 1.6 * np.sin(t)]))
    pc.conv_averaging((5, 5), 4, (r, r))
    pc.onion(0.2)
    return ab.flatten(pc), ab.GridSpec((8.0, 8.0), (r, r))


def _time(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "gpus": torch.cuda.device_count()}


def signed_old_vs_new(baseline, reps, emit):
    import torch
    import aegolius_b200 as ab
    from aegolius_b200 import cabi, engine
    a = ab.Sphere(0.9)
    a.move((-0.52, 0.13, 0.07))
    t = ab.Torus(1.0, 0.35)
    t.move((0.4, -0.2, 0.1))
    u = ab.CombineGeometry("UNION2").combine(a, t)
    u.boundary()
    spec = ab.GridSpec((4.0, 4.0, 4.0), (513, 513, 513))
    field = engine.create_torch(u, spec, dtype="f32")
    res = (C.c_uint32 * 3)(*spec.res)
    thr = engine.grid_min_step(spec)
    libs = {"new": cabi.lib()}
    if baseline:
        old = C.CDLL(baseline)
        old.ab_signed_field.restype = C.c_int
        old.ab_signed_field.argtypes = cabi.lib().ab_signed_field.argtypes
        libs["baseline"] = old
    outs = {k: torch.empty_like(field) for k in libs}
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(k):
        return lambda: cabi.check(libs[k].ab_signed_field(C.c_void_p(field.data_ptr()), res, thr, cabi.AB_F32,
                                                          C.c_void_p(outs[k].data_ptr()), 0, st))
    times = {k: [] for k in libs}
    for _ in range(5):  # alternated rounds
        for k in libs:
            times[k].append(_time(run(k), reps))
    same = bool(torch.equal(outs["new"], outs["baseline"])) if baseline else None
    emit({"measure": "ab_signed_field whole grid", "res": 513, "dtype": "f32",
          "ms_median_per_round": {k: [round(v, 4) for v in vs] for k, vs in times.items()},
          "ms": {k: round(sorted(vs)[len(vs) // 2], 4) for k, vs in times.items()}, "bit_identical": same})


def halo_overhead(reps, emit):
    from aegolius_b200 import codegen, engine
    for name, (prog, spec) in (("stencil_conv_averaging_tree3d", tree3d(513)),
                               ("stencil_conv_averaging_cloud2d", cloud2d(4097))):
        whole = _time(lambda: engine.create_torch(prog, spec), reps)
        row = {"measure": "staged slabs vs whole grid", "tree": name, "res": list(spec.res), "dtype": "f32",
               "jit": codegen.mode(), "whole_ms": round(whole, 3)}
        for parts in (2, 8):
            ranges = engine.slab_ranges(spec.res[0], parts)
            tot = sum(_time(lambda s=s: engine.create_torch(prog, spec, slab=s), reps) for s in ranges)
            row[f"sum_of_{parts}_slabs_ms"] = round(tot, 3)
            row[f"overhead_{parts}"] = round(tot / whole - 1.0, 4)
        emit(row)


def sharded(reps):
    import torch
    import torch.distributed as dist
    from aegolius_b200 import distributed as D
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    for name, (prog, spec) in (("stencil_conv_averaging_tree3d", tree3d(513)),
                               ("stencil_conv_averaging_cloud2d", cloud2d(4097))):
        ms = _time(lambda: D.evaluate_sharded(prog, spec), reps)
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if dist.get_rank() == 0:
            print(json.dumps({"measure": "evaluate_sharded device time (slowest rank)", "tree": name,
                              "world": dist.get_world_size(), "ms": round(float(t), 3)}), flush=True)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--sharded", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    os.environ.setdefault("AB_JIT", "cache")  # kernels already on disk, no nvcc while timing
    if args.sharded:
        return sharded(args.reps)
    import torch
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)
    emit({"card": card()})
    signed_old_vs_new(args.baseline_lib, args.reps, emit)
    halo_overhead(args.reps, emit)
    n = torch.cuda.device_count()
    if n > 1:
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                            "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__), "--sharded",
                            "--reps", str(args.reps)], capture_output=True, text=True, timeout=1200)
        for ln in r.stdout.splitlines():
            if ln.startswith("{"):
                emit(json.loads(ln))
        if r.returncode:
            emit({"measure": "evaluate_sharded", "error": r.stderr[-2000:]})
    else:
        emit({"measure": "evaluate_sharded", "note": "not measured: one GPU"})
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "stage_slab_probe.jsonl"), "w") as fh:
            fh.writelines(json.dumps(d) + "\n" for d in lines)


if __name__ == "__main__":
    main()
