"""Sharded parameter tangents of trees with grid-stencil stages, against one GPU, bit for bit. Run under
torch.distributed.run:

    python -m torch.distributed.run --nproc-per-node 2 tools/check_stage_tangents_multi_gpu.py [--res 97]

Checks evaluate_sharded(grad="param", gather=True) of a box-stage tree and of a signed tree (field and tangent) against the
whole-grid create_torch(grad="param") of the same process. Prints one JSON line per check ({"check": ..., "ok": ...}) on
rank 0 and exits non-zero if any check fails on any rank."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def builders(r):
    import aegolius_b200 as ab

    def box(radius, w):
        s = ab.Sphere(radius)
        s.move((0.4, -0.2, 0.3))
        s.conv_averaging((4, 3, 2), 2, (r, r, r))
        b = ab.Box(1.6, 1.0, 2.0)
        b.rotate(0.5, (0, 1, 0))
        u = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=w)
        u.conv_averaging(3, 1, (r, r, r))
        return u

    def signed(radius, x):
        a = ab.Sphere(radius)
        a.move((x, 0.13, 0.07))
        t = ab.Torus(1.0, 0.35)
        t.move((0.4, -0.2, 0.1))
        sg = ab.CombineGeometry("UNION2").combine(a, t)
        sg.boundary()
        sg.signed((r, r, r))
        sg.conv_averaging(3, 1, (r, r, r))
        return sg

    return {"box": (box, (1.1, 0.3)), "signed": (signed, (0.9, -0.52))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=97)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    import aegolius_b200 as ab
    from aegolius_b200 import distributed as D, engine
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    spec = ab.GridSpec((4, 4, 4), (args.res,) * 3)
    results = []
    for name, (builder, params) in builders(args.res).items():
        for k in range(len(params)):
            prog = engine.program_tangent(builder, params, k)
            for dtype in ("f32", "f64"):
                field, tangent = engine.create_torch(prog, spec, dtype=dtype, grad="param", device=local)
                got_f, got_t = D.evaluate_sharded(prog, spec, dtype=dtype, grad="param", gather=True)
                ok = torch.equal(got_f, field) and torch.equal(got_t, tangent)
                results.append((f"evaluate_sharded/param/{name}/theta{k}/{dtype}", bool(ok)))
    flags = torch.tensor([0 if ok else 1 for _, ok in results], dtype=torch.int32, device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MAX)
    if rank == 0:
        for (name, _), bad in zip(results, flags.tolist()):
            print(json.dumps({"check": name, "world": world, "res": args.res, "ok": not bad}), flush=True)
    dist.destroy_process_group()
    sys.exit(1 if flags.any() else 0)


if __name__ == "__main__":
    main()
