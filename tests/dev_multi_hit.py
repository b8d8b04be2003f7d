"""Ray rate of the k-nearest-hits query next to closest hit, on the bench's flagship workload: the 1 M-face displaced
icosphere (geodesic frequency 224: 1 003 520 OBJ faces, 2 007 040 CLTriangles) and its incoherent shell stream (origins on
the sphere of radius 3R, targets in the ball R), device-resident, 2^24 rays per launch by default.

trace_closest_device and trace_multi_device at k = 1, 4 and 16 are timed in the same process, alternating round by round,
with CUDA events around `--steps` launches on one stream (after `--warmup` launches of each). Also reported: the mean number
of hits per ray in the k = 16 rows (how full the lists are), whether the k = 1 rows equal the closest-hit output bit for
bit, and the card's name and power limit. One JSON line at the end.

    python tests/dev_multi_hit.py [--frequency 224] [--rays 16777216] [--steps 5] [--warmup 2] [--rounds 3]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

KS = (1, 4, 16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frequency", type=int, default=224)
    ap.add_argument("--rays", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from conftest import load_product
    from dev_device_scene import card
    prod = load_product()
    if prod.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    res = {"card": card(), "rays_per_launch": args.rays, "steps": args.steps, "rounds": args.rounds}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    path = bench.ensure_scene(args.frequency, 0, 1, lambda: None)
    tris, nodes, mats = prod.host.load_scene(path, 4, cache=True)[:3]
    res.update(faces=20 * args.frequency ** 2, cltriangles=int(tris.shape[0]))
    n = args.rays
    rays = prod.workloads.shell_rays(n, bench.RADIUS, seed=1000)
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32)).cuda()
    d_hits = torch.empty((n * max(KS), 4), dtype=torch.int32, device="cuda")
    stream = torch.cuda.Stream()
    with prod.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        legs = {"closest": lambda: ctx.trace_closest_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream.cuda_stream)}
        for k in KS:
            legs["multi_k%d" % k] = (lambda k=k: ctx.trace_multi_device(d_rays.data_ptr(), n, k, d_hits.data_ptr(), stream.cuda_stream))
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
                    e0.record()
                    for _ in range(args.steps):
                        fn()
                    e1.record()
                torch.cuda.synchronize()
                rates[name].append(n * args.steps / (e0.elapsed_time(e1) * 1e3))        # Mrays/s
        res["mrays_per_s"] = {name: {"median": statistics.median(v), "min": min(v), "max": max(v)} for name, v in rates.items()}
        # outputs (outside the timed region)
        with torch.cuda.stream(stream):
            legs["closest"]()
        torch.cuda.synchronize()
        closest = d_hits[:n].cpu().numpy().copy()
        with torch.cuda.stream(stream):
            legs["multi_k1"]()
        torch.cuda.synchronize()
        res["k1_equals_closest"] = bool(np.array_equal(d_hits[:n].cpu().numpy(), closest))
        with torch.cuda.stream(stream):
            legs["multi_k16"]()
        torch.cuda.synchronize()
        tri16 = d_hits[:n * 16, 3].cpu().numpy().view(np.uint32).reshape(n, 16)
        used = tri16 != 0xFFFFFFFF
        res["mean_hits_per_ray_k16"] = float(used.sum(1).mean())
        res["rows_full_k16"] = float(used[:, -1].mean())
        res["closest_hit_fraction"] = float((closest[:, 3].view(np.uint32) != 0xFFFFFFFF).mean())
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
