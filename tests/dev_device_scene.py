"""Scene set-up on the bench's 1 M-face scene (geodesic frequency 224: 1 003 520 OBJ faces, 2 007 040 CLTriangles), two ways,
each ending in a device synchronise:

  host path    b2rt_build_bvh (host grouping, device tree, read-back) + host re-order + b2rt_upload_scene, whose first
               ensure_scene derives the wide BVH on the host and uploads it
  device path  b2rt_build_scene_device from loader triangles already on the device (the H2D copy that puts them there is
               reported on its own)

plus the per-phase device times of the device path (CUDA events, B2RT_TRACE_BUILD) and Mrays/s of the same closest-hit
stream through both scenes (the arrays are identical, so the rates should agree within noise). Prints one JSON line.

    python tests/dev_device_scene.py [--frequency 224] [--repeats 3] [--rays 16777216]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def capture_stderr(fn):
    """Runs fn() with file descriptor 2 redirected to a temporary file; returns (result, captured text)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            r = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        return r, f.read()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frequency", type=int, default=224)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--rays", type=int, default=1 << 24)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from conftest import load_product
    prod = load_product()
    if prod.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    path = bench.ensure_scene(args.frequency, 0, 1, lambda: None)
    lt, mats = prod.host.load_triangles(path)
    n = lt.shape[0]
    res = {"card": card(), "faces": 20 * args.frequency ** 2, "cltriangles": n}

    def sync_time(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    host_s, dev_s, h2d_s, phases = [], [], [], []
    with prod.Context(0) as hctx, prod.Context(0) as dctx:
        hctx.build_bvh(lt[:4096])                                            # warm-up: modules, allocator
        dctx.set_materials(mats)
        lt_pinned = torch.from_numpy(lt.reshape(-1)).pin_memory()
        d_lt = torch.empty(lt.nbytes, dtype=torch.uint8, device="cuda")
        d_lt[: 4096 * 256].copy_(lt_pinned[: 4096 * 256])
        previous = list(dctx.build_scene_device(d_lt.data_ptr(), 4096)[:2])

        def release_previous(built):
            # a rebuilt scene leaves the caller the buffers of the one before (unbound, not released): release them like a
            # real caller would
            for b in previous:
                dctx._ck(dctx._L.b2rt_buffer_release(dctx._h, b))
            previous[:] = built[:2]
        for _ in range(args.repeats):
            def host_path():
                t, nd, _ = hctx.build_bvh(lt)
                hctx.upload_scene(t, nd, mats)                             # first ensure_scene: host derivation + upload
                return t, nd
            dt, (h_tris, h_nodes) = sync_time(host_path)
            host_s.append(dt)
            dt, _ = sync_time(lambda: d_lt.copy_(lt_pinned, non_blocking=True))
            h2d_s.append(dt)
            os.environ["B2RT_TRACE_BUILD"] = "1"
            (dt, built), text = capture_stderr(lambda: sync_time(lambda: dctx.build_scene_device(d_lt.data_ptr(), n)))
            del os.environ["B2RT_TRACE_BUILD"]
            release_previous(built)
            dev_s.append(dt)
            line = [s for s in text.splitlines() if s.startswith("[b2rt_build_scene_device]")]
            phases.append(line[-1] if line else text.strip())
        d_tris, d_nodes = dctx.read_scene()
        res["arrays_identical"] = bool(np.array_equal(d_tris, h_tris.reshape(d_tris.shape)) and np.array_equal(d_nodes, h_nodes))
        res["host_path_s"] = host_s
        res["device_path_s"] = dev_s
        res["h2d_loader_triangles_s"] = h2d_s
        res["device_phases"] = phases
        # the same closest-hit stream through both scenes, alternating
        wl = bench.workloads_only()
        rays = wl.shell_rays(args.rays, bench.RADIUS, seed=1000)
        d_rays = torch.from_numpy(rays.view(np.uint8)).cuda()
        d_hits = [torch.empty((args.rays, 4), dtype=torch.float32, device="cuda") for _ in range(2)]
        stream = torch.cuda.Stream()                                         # a real stream: handle 0 would mean the context's own
        rates = {"host_built": [], "device_built": []}
        with torch.cuda.stream(stream):
            for ctx, key, hits in ((hctx, "host_built", d_hits[0]), (dctx, "device_built", d_hits[1])):
                ctx.trace_closest_device(d_rays.data_ptr(), args.rays, hits.data_ptr(), stream.cuda_stream)
            for _ in range(3):
                for ctx, key, hits in ((hctx, "host_built", d_hits[0]), (dctx, "device_built", d_hits[1])):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(3):
                        ctx.trace_closest_device(d_rays.data_ptr(), args.rays, hits.data_ptr(), stream.cuda_stream)
                    e1.record(stream)
                    e1.synchronize()
                    rates[key].append(3 * args.rays / (e0.elapsed_time(e1) * 1e-3) / 1e6)
        stream.synchronize()
        res["closest_mrays_s"] = rates
        res["hits_bit_identical"] = bool(torch.equal(d_hits[0].view(torch.int32), d_hits[1].view(torch.int32)))
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
