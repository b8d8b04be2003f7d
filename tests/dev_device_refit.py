"""Per-frame cost of following moving geometry on the bench's 1 M-face scene (geodesic frequency 224: 1 003 520 OBJ faces,
2 007 040 CLTriangles) whose deformed LOADER-order triangles are already on the device, four ways, alternated, each timed
with a host clock that ends in a device synchronise:

  rebuild          b2rt_build_scene_device on the deformed triangles (new buffers, new tree, new hit IDs)
  host_round_trip  D2H of the loader-order triangles, host re-order through the build's order, b2rt_refit_scene (H2D)
  device_loader    b2rt_refit_scene_device from the loader-order triangles through the build's device order
  device_in_place  b2rt_refit_scene_device on scene-order triangles already written into the bound triangle buffer

The two device refits are also timed with CUDA events (device time), against the bytes they must move, counted from the
array sizes (32-byte sectors): the gather's 256 B read + 256 B write + 4 B order per triangle, the three 16-byte vertex
positions read by the leaf and leaf-block kernels, the normals + material read by the shading kernel, node boxes read and
written, wide nodes read and written, child_bin / leaf_dir read, leaf blocks and shading records written. bytes / 7.7 TB/s
is a computed lower bound, not a measurement. Then closest-hit Mrays/s on 2^24 incoherent rays after refits under a small
and a large deformation against a rebuild of the same deformed geometry, and whether the device refit's hits equal the host
round trip's bit for bit. Prints the card's name and power limit and one JSON line.

    python tests/dev_device_refit.py [--frequency 224] [--repeats 5] [--rays 16777216]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_TBS = 7.7          # B200 HBM3e peak, TB/s (datasheet): the lower bound's denominator


def deform(torch, base, scale, wobble):
    """New positions as a function of each old position alone (the loader's duplicate pairs stay rotations)."""
    f = base.view(torch.float32).view(-1, 64)
    out = f.clone()
    for v in (0, 20, 40):
        p = f[:, v:v + 3]
        q = p * scale
        q[:, 2] += wobble * torch.sin(p[:, 0] * 0.7)
        out[:, v:v + 3] = q
    return out.view(torch.uint8).view(-1)


def refit_bytes(info, n):
    sector = 32
    gather = n * (256 + 256 + 4)
    positions = 2 * n * 3 * sector                     # leaf kernel and leaf-block kernel: three vertex positions each
    shading_in = n * 4 * sector                        # three normals + the material index
    nodes = info["n_nodes"] * 48 * 3                   # leaf boxes written, interior boxes read and written
    scratch = info["n_nodes"] * 8 * 2
    wide = info["wide_node_bytes"] * 2 + info["n_wide_nodes"] * 32 + info["n_wide_nodes"] * 8 * 48
    blocks = info["leaf_bytes"] + info["n_leaf_blocks"] * (8 + 48)
    shade_out = info["shading_bytes"]
    parts = dict(gather=gather, vertex_positions=positions, shading_inputs=shading_in, nodes=nodes + scratch, wide_nodes=wide,
                 leaf_blocks=blocks, shading_records=shade_out)
    return parts, sum(parts.values())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frequency", type=int, default=224)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--rays", type=int, default=1 << 24)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from conftest import load_product
    from dev_device_scene import card
    prod = load_product()
    if prod.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    res = {"card": card()}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    path = bench.ensure_scene(args.frequency, 0, 1, lambda: None)
    lt, mats = prod.host.load_triangles(path)
    n = lt.shape[0]
    res.update(faces=20 * args.frequency ** 2, cltriangles=n)

    def sync_time(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    d_lt = torch.from_numpy(lt.reshape(-1)).cuda()
    small = deform(torch, d_lt, 1.02, 0.05)
    large = deform(torch, d_lt, 1.0, 2.5)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    with prod.Context(0) as ctx, prod.Context(0) as rctx:
        ctx.set_materials(mats)
        rctx.set_materials(mats)
        d_order = torch.empty(n, dtype=torch.int32, device="cuda")
        ctx.build_scene_device(d_lt.data_ptr(), n, d_order=d_order.data_ptr())
        order = d_order.cpu().numpy()
        order_long = d_order.long()
        previous = list(rctx.build_scene_device(d_lt.data_ptr(), n)[:2])
        info = ctx.scene_info()
        buf, ptr = C.c_uint64(0), C.c_void_p()
        ctx._ck(ctx._L.b2rt_bound_buffer(ctx._h, 1, C.byref(buf)))
        ctx._ck(ctx._L.b2rt_device_pointer(ctx._h, buf, C.byref(ptr), None))
        bound_ptr = ptr.value

        def rebuild():
            built = rctx.build_scene_device(small.data_ptr(), n)
            for b in previous:                     # a rebuilt scene leaves the caller the buffers of the one before
                rctx._ck(rctx._L.b2rt_buffer_release(rctx._h, b))
            previous[:] = built[:2]

        def host_round_trip():
            h = small.cpu().numpy().reshape(n, 256)
            ctx.refit_scene(h[order])

        def device_loader(stream=0):
            ctx.refit_scene_device(small.data_ptr(), n, status.data_ptr(), d_order=d_order.data_ptr(), stream=stream)

        scene_order = small.view(n, 256)[order_long]                          # scene-order copy for the in-place path

        class _View:
            __cuda_array_interface__ = {"shape": (n * 256,), "typestr": "|u1", "data": (bound_ptr, False), "version": 2}
        bound = torch.as_tensor(_View(), device="cuda")

        def device_in_place(stream=0):
            ctx.refit_scene_device(bound_ptr, n, status.data_ptr(), stream=stream)

        paths = dict(rebuild=rebuild, host_round_trip=host_round_trip, device_loader=device_loader, device_in_place=device_in_place)
        status_bits = []                                                     # the status word after every device refit

        def check_status():
            torch.cuda.synchronize()
            status_bits.append(int(status.item()))

        for k, fn in paths.items():                                          # warm-up: modules, pools, pinned staging
            if fn is device_in_place:
                bound.copy_(scene_order.view(-1))
            sync_time(fn)
            if k.startswith("device"):
                check_status()
        side = torch.cuda.Stream()
        wall = {k: [] for k in paths}
        device_ms = {"device_loader": [], "device_in_place": []}
        for _ in range(args.repeats):
            for k, fn in paths.items():
                if fn is device_in_place:
                    bound.copy_(scene_order.view(-1))                        # the caller's simulation wrote the bound buffer
                dt, _ = sync_time(fn)
                wall[k].append(dt * 1e3)
                if k in device_ms:
                    check_status()
                if k in device_ms:
                    # device time: events on a side stream around the call given that stream (the call orders the context's
                    # stream behind it and it behind the refit); a sleep keeps the device busy while the host enqueues
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    if fn is device_in_place:
                        bound.copy_(scene_order.view(-1))
                    torch.cuda.synchronize()
                    with torch.cuda.stream(side):
                        torch.cuda._sleep(20_000_000)
                        e0.record(side)
                        fn(side.cuda_stream)
                        e1.record(side)
                    e1.synchronize()
                    device_ms[k].append(e0.elapsed_time(e1))
                    check_status()
        assert not any(status_bits), status_bits
        res["device_refits_checked"] = len(status_bits)
        res["wall_ms"] = wall
        res["wall_ms_median"] = {k: statistics.median(v) for k, v in wall.items()}
        res["device_refit_event_ms"] = device_ms
        parts, total = refit_bytes(info, n)
        res["device_refit_bytes"] = parts
        res["device_refit_bytes_total"] = total
        bound_ms = total / (HBM_TBS * 1e12) * 1e3
        res["lower_bound_ms_at_7.7TBs"] = bound_ms
        res["achieved_share_of_bound"] = {k: bound_ms / min(v) for k, v in device_ms.items()}

        # the device refit's hits against the host round trip's, bit for bit
        wl = bench.workloads_only()
        rays = wl.shell_rays(args.rays, bench.RADIUS, seed=1000)
        d_rays = torch.from_numpy(rays.view(np.uint8)).cuda()
        hits = [torch.empty((args.rays, 4), dtype=torch.float32, device="cuda") for _ in range(3)]
        stream = torch.cuda.Stream()
        device_loader()
        check_status()
        assert status_bits[-1] == 0
        ctx.trace_closest_device(d_rays.data_ptr(), args.rays, hits[0].data_ptr(), 0)
        ctx.finish()
        host_round_trip()
        ctx.trace_closest_device(d_rays.data_ptr(), args.rays, hits[1].data_ptr(), 0)
        ctx.finish()
        res["device_refit_hits_equal_host_round_trip"] = bool(torch.equal(hits[0].view(torch.int32), hits[1].view(torch.int32)))

        # traversal speed of a refitted tree against a rebuild of the same deformed geometry
        def rate(c):
            c.trace_closest_device(d_rays.data_ptr(), args.rays, hits[2].data_ptr(), stream.cuda_stream)
            out = []
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(3):
                    c.trace_closest_device(d_rays.data_ptr(), args.rays, hits[2].data_ptr(), stream.cuda_stream)
                e1.record(stream)
                e1.synchronize()
                out.append(3 * args.rays / (e0.elapsed_time(e1) * 1e-3) / 1e6)
            return out
        quality = {}
        for name, data in (("undeformed", d_lt), ("small", small), ("large", large)):
            ctx.refit_scene_device(data.data_ptr(), n, status.data_ptr(), d_order=d_order.data_ptr())
            ctx.finish()
            assert int(status.item()) == 0, name
            built = rctx.build_scene_device(data.data_ptr(), n)
            for b in previous:
                rctx._ck(rctx._L.b2rt_buffer_release(rctx._h, b))
            previous[:] = built[:2]
            torch.cuda.synchronize()
            quality[name] = {"refit_mrays_s": rate(ctx), "rebuild_mrays_s": rate(rctx)}
        res["closest_mrays_s_refit_vs_rebuild"] = quality
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
