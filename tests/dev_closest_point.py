"""Query rate of b2rt_closest_point_device on the bench's flagship scene: the 1 M-face displaced icosphere (geodesic
frequency 224: 1 003 520 OBJ faces, 2 007 040 CLTriangles), 2^22 device-resident queries per launch by default.

Three query sets: `near` (points within 1 % of the radius of the surface, max_d2 = (2 % of R)^2), `box` (uniform in the
scene's bounding box, max_d2 = inf) and `far` (on a sphere of radius 3R, max_d2 = inf). Per set, the wide walk and the
reference-layout walk (B2RT_OPT_TRAVERSAL = 1) are timed with CUDA events around `--steps` launches on one stream, after
`--warmup` launches of each, alternating leg by leg over `--rounds` rounds; closest hit on the bench's shell stream (same
count) is timed alongside for context. The counting build (a separate launch) gives wide-node visits, leaf blocks and
distance evaluations per query. The wide and reference-layout outputs are compared bit for bit. The card's name, power
limit and max SM clock are read in the same process. One JSON line at the end.

    python tests/dev_closest_point.py [--frequency 224] [--queries 4194304] [--steps 5] [--warmup 2] [--rounds 3] [--out f.json]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def query_sets(tris, n, R, seed=2024):
    import numpy as np
    import point_query_lib as pq
    rng = np.random.default_rng(seed)
    f = tris.view(np.float32).reshape(-1, 64)
    k = rng.integers(0, tris.shape[0], n)
    w = rng.dirichlet((1.0, 1.0, 1.0), n).astype(np.float32)
    surf = f[k, 0:3] * w[:, :1] + f[k, 20:23] * w[:, 1:2] + f[k, 40:43] * w[:, 2:3]
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    near = pq.queries(surf + d * rng.uniform(-0.01 * R, 0.01 * R, (n, 1)).astype(np.float32), np.float32((0.02 * R) ** 2))
    lo, hi = f[:, 0:3].min(0), f[:, 0:3].max(0)
    box = pq.queries(rng.uniform(lo, hi, (n, 3)).astype(np.float32), np.inf)
    far = pq.queries(d * np.float32(3.0 * R), np.inf)
    return {"near": near, "box": box, "far": far}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frequency", type=int, default=224)
    ap.add_argument("--queries", type=int, default=1 << 22)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from conftest import load_product
    from dev_device_scene import card
    prod = load_product()
    if prod.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    cap = prod.capi
    res = {"card": card(), "queries_per_launch": args.queries, "steps": args.steps, "rounds": args.rounds}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    path = bench.ensure_scene(args.frequency, 0, 1, lambda: None)
    tris, nodes, mats = prod.host.load_scene(path, 4, cache=True)[:3]
    res.update(faces=20 * args.frequency ** 2, cltriangles=int(tris.shape[0]))
    n = args.queries
    sets = query_sets(tris, n, bench.RADIUS)
    rays = prod.workloads.shell_rays(n, bench.RADIUS, seed=1000)
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32)).cuda()
    d_q = {name: torch.from_numpy(q.view(np.uint8).reshape(-1, 16).copy()).cuda() for name, q in sets.items()}
    d_out = torch.empty((n, 4), dtype=torch.int32, device="cuda")
    stream = torch.cuda.Stream()
    with prod.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)

        def point_leg(name, traversal):
            def run():
                ctx.set_option(cap.OPT_TRAVERSAL, traversal)
                ctx.closest_point_device(d_q[name].data_ptr(), n, d_out.data_ptr(), stream.cuda_stream)
            return run
        legs = {"closest_hit_rays": lambda: (ctx.set_option(cap.OPT_TRAVERSAL, 0),
                                             ctx.trace_closest_device(d_rays.data_ptr(), n, d_out.data_ptr(), stream.cuda_stream))}
        for name in sets:
            legs[name + "_wide"] = point_leg(name, 0)
            legs[name + "_reference_layout"] = point_leg(name, 1)
        with torch.cuda.stream(stream):
            for fn in legs.values():
                for _ in range(args.warmup):
                    fn()
        torch.cuda.synchronize()
        rates = {name: [] for name in legs}
        for _ in range(args.rounds):
            for name, fn in legs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    fn()                                   # sets the option outside the timed window
                    e0.record()
                    for _ in range(args.steps):
                        fn()
                    e1.record()
                torch.cuda.synchronize()
                rates[name].append(n * args.steps / (e0.elapsed_time(e1) * 1e3))        # M queries (rays) / s
        res["mqueries_per_s"] = {name: {"median": statistics.median(v), "min": min(v), "max": max(v)} for name, v in rates.items()}
        ctx.set_option(cap.OPT_TRAVERSAL, 0)
        # outputs and counters, outside the timed region
        res["per_set"] = {}
        for name in sets:
            outs = []
            for traversal in (0, 1):
                ctx.set_option(cap.OPT_TRAVERSAL, traversal)
                with torch.cuda.stream(stream):
                    ctx.closest_point_device(d_q[name].data_ptr(), n, d_out.data_ptr(), stream.cuda_stream)
                torch.cuda.synchronize()
                outs.append(d_out.cpu().numpy().copy())
            ctx.set_option(cap.OPT_TRAVERSAL, 0)
            ctx.set_option(cap.OPT_COUNTERS, 1)
            ctx.reset_counters()
            with torch.cuda.stream(stream):
                ctx.closest_point_device(d_q[name].data_ptr(), n, d_out.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize()
            c = ctx.counters()
            ctx.set_option(cap.OPT_COUNTERS, 0)
            found = outs[0][:, 3].view(np.uint32) != 0xFFFFFFFF
            res["per_set"][name] = {
                "wide_equals_reference_layout": bool(np.array_equal(outs[0], outs[1])),
                "found_fraction": float(found.mean()),
                "wide_nodes_per_query": c["wide_nodes"] / max(c["rays"], 1),
                "leaf_blocks_per_query": c["leaf_blocks"] / max(c["rays"], 1),
                "distance_evaluations_per_query": c["tri_tests"] / max(c["rays"], 1),
                "stack_overflows": c["stack_overflows"], "counted_queries": c["rays"],
            }
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
