"""Sharded evaluation of trees with grid-stencil stages, against one GPU, bit for bit. Run under torch.distributed.run:

    python -m torch.distributed.run --nproc-per-node 2 tools/check_stage_slabs_multi_gpu.py [--res 97]

Checks evaluate_sharded(gather=True) of a box-stage tree and of a signed tree, and from_sdf_sharded of a staged tree,
each against the whole-grid create_torch / from_sdf_torch of the same process. Prints one JSON line per check
({"check": ..., "ok": ...}) on rank 0 and exits non-zero if any check fails on any rank."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def trees(r):
    import aegolius_b200 as ab
    s = ab.Sphere(1.1)
    s.move((0.4, -0.2, 0.3))
    s.conv_averaging((4, 3, 2), 2, (r, r, r))
    b = ab.Box(1.6, 1.0, 2.0)
    b.rotate(0.5, (0, 1, 0))
    box = ab.CombineGeometry("SMOOTH_UNION2").combine_parametric(s, b, parameters=0.3)
    box.conv_averaging(3, 1, (r, r, r))
    a = ab.Sphere(0.9)
    a.move((-0.52, 0.13, 0.07))
    t = ab.Torus(1.0, 0.35)
    t.move((0.4, -0.2, 0.1))
    sg = ab.CombineGeometry("UNION2").combine(a, t)
    sg.boundary()
    sg.signed((r, r, r))
    sg.conv_averaging(3, 1, (r, r, r))
    return {"box": ab.flatten(box), "signed": ab.flatten(sg)}


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
    for name, prog in trees(args.res).items():
        for dtype in ("f32", "f64"):
            whole = engine.create_torch(prog, spec, dtype=dtype, device=local)
            got = D.evaluate_sharded(prog, spec, dtype=dtype, gather=True)
            results.append((f"evaluate_sharded/{name}/{dtype}", bool(torch.equal(got, whole))))
    prog = trees(args.res)["signed"]
    whole = engine.create_torch(prog, spec, dtype="f32", device=local)
    vec = engine.from_sdf_torch(whole, spec.res, device=local)
    field, mine = D.from_sdf_sharded(prog, spec, dtype="f32")
    x0, x1 = D.rank_slab(spec.res[0], rank, world)
    pp = spec.res[1] * spec.res[2]
    ok = torch.equal(field, whole[x0 * pp:x1 * pp]) and torch.equal(mine, vec[:, x0 * pp:x1 * pp])
    results.append(("from_sdf_sharded/signed/f32", bool(ok)))
    flags = torch.tensor([0 if ok else 1 for _, ok in results], dtype=torch.int32, device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MAX)
    if rank == 0:
        for (name, _), bad in zip(results, flags.tolist()):
            print(json.dumps({"check": name, "world": world, "res": args.res, "ok": not bad}), flush=True)
    dist.destroy_process_group()
    sys.exit(1 if flags.any() else 0)


if __name__ == "__main__":
    main()
