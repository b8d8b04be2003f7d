"""Path rate of b2rt_trace_radiance_device against the wavefront frame path on the bench's flagship scene: the 1 M-face
displaced icosphere (geodesic frequency 224), 2^22 paths per launch at 4 bounces by default.

Both legs trace the same paths. The frame leg draws a 2048 x 2048 frame (B2RT_OPT_RENDER_MODE = 0, the wavefront). The
radiance leg takes that frame's camera rays (b2rt_camera_rays_device) and, as seeds, the RNG state each pixel has after
CreateRay's two draws, so every path is the frame's path; only the source (stored rays instead of CreateRay) and the sink
(a 16-byte record instead of the running average) differ. Each leg runs `--steps` launches on the context's stream between
host clock reads that end in b2rt_finish, after `--warmup` launches, alternating leg by leg over `--rounds` rounds. The
counting build (a separate launch) gives the path segments traced per launch, hence segments/s. The card's name, power
limit and max SM clock are read in the same process. One JSON line at the end.

    python tests/dev_radiance.py [--frequency 224] [--side 2048] [--bounces 4] [--steps 5] [--warmup 2] [--rounds 3] [--out f.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def seeds_after_camera(n, frame_count):
    """seed = gid + hash_u32(frame_count) (kernel_bvh.cl:445) advanced by CreateRay's two rnd() draws."""
    import numpy as np
    m = np.uint64(0xFFFFFFFF)
    s = (np.arange(n, dtype=np.uint64) + np.uint64((1103515245 * frame_count + 12345) & 0xFFFFFFFF)) & m
    for _ in range(2):
        s ^= s >> np.uint64(16); s = (s * np.uint64(0x7feb352d)) & m
        s ^= s >> np.uint64(15); s = (s * np.uint64(0x846ca68b)) & m
        s ^= s >> np.uint64(16)
    return s.astype(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frequency", type=int, default=224)
    ap.add_argument("--side", type=int, default=2048)
    ap.add_argument("--bounces", type=int, default=4)
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
    W = H = args.side
    n = W * H
    res = {"card": card(), "paths_per_launch": n, "bounces": args.bounces, "steps": args.steps, "rounds": args.rounds}
    path = bench.ensure_scene(args.frequency, 0, 1, lambda: None)
    tris, nodes, mats = prod.host.load_scene(path, 4, cache=True)[:3]
    res["scene"] = {"path": os.path.basename(path), "triangles": int(tris.shape[0])}
    with prod.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        ctx.resize(W, H)
        ctx.set_option(cap.OPT_RENDER_MODE, 0)
        ctx.set_frame(1, args.bounces, light_type=1)
        d_rays = torch.empty((n, 8), dtype=torch.float32, device="cuda")
        ctx.camera_rays_device(0, n, d_rays.data_ptr())
        ctx.finish()
        d_seeds = torch.from_numpy(seeds_after_camera(n, 1).view(np.int32)).cuda()
        d_out = torch.empty((n, 4), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()

        legs = {"radiance": lambda: ctx.trace_radiance_device(d_rays.data_ptr(), d_seeds.data_ptr(), n, d_out.data_ptr(), 0),
                "frame": lambda: ctx.execute(n)}

        def timed(fn, steps):
            ctx.finish()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            ctx.finish()
            return (time.perf_counter() - t0) * 1e3 / steps

        for name, fn in legs.items():
            timed(fn, args.warmup)
        ms = {k: [] for k in legs}
        for _ in range(args.rounds):
            for name, fn in legs.items():
                ms[name].append(timed(fn, args.steps))
        segs = {}
        for name, fn in legs.items():
            ctx.set_option(cap.OPT_COUNTERS, 1)
            ctx.reset_counters()
            fn()
            segs[name] = ctx.counters()["rays"]
            ctx.set_option(cap.OPT_COUNTERS, 0)
        for name in legs:
            med = statistics.median(ms[name])
            res[name] = {"ms_per_launch": [round(x, 3) for x in ms[name]], "median_ms": round(med, 3),
                         "paths_per_s_M": round(n / med / 1e3, 1), "segments_per_launch": int(segs[name]),
                         "segments_per_s_M": round(segs[name] / med / 1e3, 1)}
        res["radiance_over_frame_time"] = round(res["radiance"]["median_ms"] / res["frame"]["median_ms"], 4)
        res["same_segments"] = segs["radiance"] == segs["frame"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
