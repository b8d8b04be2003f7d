#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BVH traversal + ray/triangle intersection).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2]/[4]): synthetic displaced geodesic icosphere, 1 003 520 OBJ faces ->
2 007 040 CLTriangle after the loader's duplication, built by the product's own CLOBJloader + CLBVHScene
mirror; one step = one closest-hit pass over a seeded stream of 100 M incoherent rays per GPU (origins on
a sphere of radius 3R, targets in the ball of radius R). Multi-GPU: BVH replicated, the ray stream is
sharded by rank (weak scaling), no data-path collective.

One JSON line on stdout (rank 0): value = whole-job Mrays/s with rays resident in HBM; e2e = the same
metric through b2rt_trace_closest with pinned HOST buffers (H2D + D2H inside the timed region);
roofline = algorithmic bytes (48 B/ray stream + counted node/leaf bytes) / kernel time vs the measured
HBM peak; cpu_baseline = the reference's own Intersect() (oracle/_ref) on the host cores, bounded sample.

--dump-outputs DIR (rank 0) writes what the timed closest-hit and any-hit steps returned for a fixed, seeded sample of
the stream's rays as DIR/<name>.npy, so that two builds can be compared output for output: the inputs depend only on
the arguments. The bench writes nothing into the tree (it may be read-only); generated scenes, their binary caches and
a rebuilt scene generator go to B2RT_SCENE_DIR, by default a per-user directory under the system's temp directory.
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True            # no __pycache__ in the tree for the modules imported from it

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mini-opencl-raytracer_b200")
SCENE_DIR = os.environ.get("B2RT_SCENE_DIR") or os.path.join(tempfile.gettempdir(), "b2rt_scenes-%d" % os.getuid())
RADIUS = 10.0
DUMP_RAYS = 1 << 20                       # --dump-outputs: rays drawn for the sample (about 40 MB of .npy files)


def product():
    if "mor_b200" in sys.modules:
        return sys.modules["mor_b200"]
    spec = importlib.util.spec_from_file_location("mor_b200", os.path.join(PKG, "__init__.py"), submodule_search_locations=[PKG])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["mor_b200"] = mod
    spec.loader.exec_module(mod)
    if not (os.path.exists(mod.lib_path()) and os.path.exists(mod.host.lib_path())):
        mod.build_all(verbose=False)          # built artefacts missing: compile in-tree (nvcc needs no GPU)
    return mod


def checkers():
    """The CPU checkers (oracle/): used ONLY for the cpu_baseline leg and --impl reference."""
    tests = os.path.join(ROOT, "tests")
    if tests not in sys.path:
        sys.path.insert(0, tests)
    import oracle_lib
    return oracle_lib


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def measured_traffic(frequency, rays):
    """dram__bytes_{read,write}.sum of one launch of the dominant kernel from the committed ncu --set full
    capture, when that capture was taken on this exact workload; else None. Second value: the capture's other
    headline metrics (L2 / DRAM throughput, pipes, stalls) for the same launch."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r1_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        t = json.load(f)
    w = t.get("workload", {})
    if w.get("frequency") == frequency and w.get("rays_per_launch") == rays:
        return t["dram_bytes_per_launch"] / 1e9, t.get("ncu")
    return None, None


def scenegen(*argv):
    """Synthetic scenes are written by a stand-alone executable (host/scene_gen.cpp with its own main, built by
    build.py), so that the reference arm can synthesise the identical workload without loading a product library."""
    src = os.path.join(PKG, "host", "scene_gen.cpp")

    def fresh(exe):
        return os.path.exists(exe) and os.path.getmtime(exe) >= os.path.getmtime(src)
    exe = os.path.join(PKG, "scenegen")
    if not fresh(exe):
        exe = os.path.join(SCENE_DIR, "scenegen")
        if not fresh(exe):
            os.makedirs(SCENE_DIR, exist_ok=True)
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-DB2RT_SCENEGEN_MAIN", src, "-o", exe])
    return int(subprocess.check_output([exe] + [str(a) for a in argv]).split()[-1])


def ensure_scene(frequency, rank, world, barrier):
    os.makedirs(SCENE_DIR, exist_ok=True)
    path = os.path.join(SCENE_DIR, "ico_f%d.obj" % frequency)
    done = path + ".done"
    if rank == 0 and not os.path.exists(done):
        t0 = time.time()
        faces = scenegen("icosphere", path, frequency, RADIUS, 0.08, 7)
        with open(done, "w") as f:
            f.write(str(faces))
        log("[bench] wrote %s: %d faces (%.1f s)" % (path, faces, time.time() - t0))
    barrier()
    return path


def workloads_only():
    """workloads.py + layouts.py (numpy only) without the package __init__, i.e. without any product library."""
    import types
    name = "mor_b200_numpy_only"
    if name not in sys.modules:
        pkg = types.ModuleType(name)
        pkg.__path__ = [PKG]
        sys.modules[name] = pkg
    return importlib.import_module(name + ".workloads")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100", "-i", str(gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_baseline(ol, kind_pref, tris, nodes, rays, seconds, threads):
    """Reference Intersect() on the host cores over a bounded sample of the same ray stream."""
    kind = "reference" if (kind_pref == "reference" and ol.ref() is not None) else "port"
    fn = (lambda r: ol.ref_closest(tris, nodes, r, threads)) if kind == "reference" else (lambda r: ol.oracle_closest(tris, nodes, r, threads))
    probe = rays[:20000 * max(threads, 1)]
    t0 = time.perf_counter()
    fn(probe)
    dt = time.perf_counter() - t0
    rate = probe.shape[0] / dt
    n = int(min(rays.shape[0], max(probe.shape[0], rate * seconds)))
    t0 = time.perf_counter()
    fn(rays[:n])
    dt = time.perf_counter() - t0
    return {"value": n / dt / 1e6, "unit": "Mrays/s", "cores": threads, "kind": kind,
            "sample": "%d rays of the same stream, closest-hit, %.1f s on %d host threads (%s)" % (
                n, dt, threads, "reference kernel_bvh.cl Intersect() compiled as C++; PoCL unavailable" if kind == "reference" else "oracle/rt_oracle.c port")}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores. Nothing of the product is
    loaded: the scene file comes from the stand-alone generator, CLOBJloader::Load + CLBVHScene::CreateBVHTrees are the
    reference's own (oracle/_ref, CLBVHnode.cpp:185-207), the rays come from workloads.py (numpy)."""
    if rank != 0:
        return
    ol = checkers()
    wl = workloads_only()
    path = ensure_scene(args.frequency, 0, 1, lambda: None)
    threads = os.cpu_count() or 1
    kind = "reference" if ol.ref() is not None else "port"
    if kind != "reference":
        raise RuntimeError("oracle/_ref/libref_oracle.so is missing: build it where /root/reference exists (python oracle/build_ref.py)")
    t0 = time.time()
    tris, nodes, mats = ol.ref_load_scene(path, 4)
    log("[bench reference] reference loader + builder: %d CLTriangle, %d nodes in %.1f s" % (tris.shape[0], nodes.shape[0], time.time() - t0))
    n = args.ref_rays
    rays = wl.shell_rays(n * (args.steps + args.warmup), RADIUS, seed=1000)
    fn = lambda r: ol.ref_closest(tris, nodes, r, threads)
    for w in range(args.warmup):
        fn(rays[w * n:(w + 1) * n])
    t0 = time.perf_counter()
    for s in range(args.steps):
        fn(rays[(args.warmup + s) * n:(args.warmup + s + 1) * n])
    dt = time.perf_counter() - t0
    value = n * args.steps / dt / 1e6
    emit({
        "impl": "reference", "metric": "closest_hit_ray_throughput", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, tris.shape[0]), "rays_per_step": n, "note": "bounded sample of the workload per step"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": kind,
                         "sample": "%d rays per step, %d steps, %d host threads" % (n, args.steps, threads)},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def workload_name(args, n_tris):
    return "displaced icosphere f=%d: %d OBJ faces -> %d CLTriangle; incoherent ray stream (origins on sphere 3R, targets in ball R), closest-hit" % (
        args.frequency, 20 * args.frequency ** 2, n_tris)


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    prod = product()
    if prod.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    path = ensure_scene(args.frequency, rank, world, barrier)
    t0 = time.time()
    eng = prod.host.Engine(1920, 1080, device=local_rank)        # CLEngineBase + CLRaytracer::Init on this GPU
    # CLOBJloader::Load + CreateBVHTrees (+ upload). Rank 0 parses + builds and leaves the binary scene cache behind;
    # the other ranks wait for it and restore the identical arrays from the cache instead of repeating the build.
    if rank == 0:
        cache_hit = eng.load_scene(path, 4, cache=True)
    barrier()
    if rank != 0:
        cache_hit = eng.load_scene(path, 4, cache=True)
    ctx = prod.Context.borrow(eng.context_handle(), local_rank)
    info = ctx.scene_info()
    log("[bench r%d] scene ready in %.1f s (scene cache %s): %s" % (rank, time.time() - t0, "hit" if cache_hit else "miss", info))

    n = args.rays
    stream = torch.cuda.Stream()
    host_rays = torch.empty((n, 8), dtype=torch.float32, pin_memory=True)
    rays_np = host_rays.numpy().view(prod.RAY_DTYPE).reshape(-1)
    prod.workloads.shell_rays(n, RADIUS, seed=1000 + (rank if not os.environ.get("B2RT_SAME_SEED") else 0), out=rays_np)
    d_rays = host_rays.to("cuda", non_blocking=False)
    d_hits = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    d_occ = torch.empty((n,), dtype=torch.int32, device="cuda")
    host_hits = torch.empty((n, 4), dtype=torch.float32, pin_memory=True)
    hits_np = host_hits.numpy().view(prod.HIT_DTYPE).reshape(-1)

    def timed(fn, steps, warmup, collective=True):
        """W untimed steps, then K steps between barrier+synchronize, per-step CUDA events on the launch stream.
        collective=False: a measurement only this rank takes (no barrier, no max over ranks)."""
        sync = barrier if collective else (lambda: None)
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                fn()
        torch.cuda.synchronize()
        sync()
        torch.cuda.synchronize()
        l0 = ctx.launch_count()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        with torch.cuda.stream(stream):
            evs[0].record()
            for i in range(steps):
                fn()
                evs[i + 1].record()
        torch.cuda.synchronize()
        sync()
        total_ms = evs[0].elapsed_time(evs[-1])
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        if world > 1 and collective:
            t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, per, ctx.launch_count() - l0

    # ---- counted pass (outside the timed region): algorithmic bytes per ray -------------------------
    ctx.set_option(prod.capi.OPT_COUNTERS, 1)
    ctx.reset_counters()
    ctx.finish()
    ctx.trace_closest_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    cnt = ctx.counters()
    ctx.set_option(prod.capi.OPT_COUNTERS, 0)
    trav_bytes = cnt["bytes_fetched"] / max(cnt["rays"], 1)
    bytes_per_ray = 48.0 + trav_bytes

    # ---- device-resident headline ------------------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    total_ms, per, launches = timed(lambda: ctx.trace_closest_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream.cuda_stream),
                          args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    value = world * n * args.steps / (total_ms * 1e-3) / 1e6
    kernel_ms = statistics.mean(per)
    log("[bench r%d] closest-hit per-step ms: %s" % (rank, " ".join("%.3f" % x for x in per)))
    dump = {}
    if rank == 0 and args.dump_outputs:
        sel = np.arange(n) if n <= DUMP_RAYS else np.unique(np.random.default_rng(0).integers(0, n, DUMP_RAYS))
        d_sel = torch.from_numpy(sel).cuda()
        h = d_hits[d_sel].cpu().numpy().view(prod.HIT_DTYPE).reshape(-1)
        dump.update(ray_index=sel.astype(np.float64), closest_t=h["t"].copy(), closest_u=h["u"].copy(), closest_v=h["v"].copy(),
                    closest_tri=h["tri"].astype(np.float64))                    # 4294967295 = miss

    # ---- any-hit on the same stream ---------------------------------------------------------------------------
    any_ms, _, _ = timed(lambda: ctx.trace_any_device(d_rays.data_ptr(), n, d_occ.data_ptr(), stream.cuda_stream), args.steps, args.warmup)
    any_value = world * n * args.steps / (any_ms * 1e-3) / 1e6
    if dump:
        dump["any_occluded"] = d_occ[d_sel].cpu().numpy().view(np.uint32).astype(np.float64)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        log("[bench] outputs of the last timed steps (%d sampled rays) written to %s" % (sel.size, args.dump_outputs))

    # ---- configs[2]: 1 M-face displaced-icosphere geometry, 4K camera rays from outside -> primary hits -> one cosine-weighted
    # bounce ray per hit, closest-hit on that incoherent batch. Bounces off ONE convex sphere all escape (r1: hit fraction
    # 0.0003, a miss-only traversal), so the batch is built on 196 displaced icospheres of 5 120 faces each (the same
    # 1 003 520 faces) scattered in a cube: 37 % of the bounce rays meet another surface. Rank 0 only.
    extra = {}
    if rank == 0 and not args.skip_frames:
        W4, H4 = 3840, 2160
        sp_path = os.path.join(SCENE_DIR, "spheres196_f16.obj")
        if not os.path.exists(sp_path + ".done"):
            scenegen("spheres", sp_path, 196, 16, 30.0, 4.0, 0.05, 5)
            open(sp_path + ".done", "w").close()
        sp_tris, sp_nodes, sp_mats = prod.host.load_scene(sp_path, 4)
        with prod.Context(local_rank) as sc:
            sc.upload_scene(sp_tris, sp_nodes, sp_mats)
            sc.set_arg(prod.capi.ARG_WIDTH, np.uint32(W4))        # CreateRay only needs the scalar arguments, no 4K output buffer
            sc.set_arg(prod.capi.ARG_HEIGHT, np.uint32(H4))
            sc.set_frame(1, 1, pos=(0.0, -95.0, 0.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))
            d_cam = torch.empty((W4 * H4, 8), dtype=torch.float32, device="cuda")
            d_camhits = torch.empty((W4 * H4, 4), dtype=torch.float32, device="cuda")
            sc.camera_rays_device(0, W4 * H4, d_cam.data_ptr(), stream.cuda_stream)

            reps_sc = max(args.steps, 20)            # launches of 2-3 ms: enough of them for a steady figure

            def timed_sc(fn):
                with torch.cuda.stream(stream):
                    for _ in range(max(args.warmup, 3)):
                        fn()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(reps_sc):
                        fn()
                    e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) * args.steps / reps_sc      # scaled to args.steps launches, which the rates below divide by
            prim_ms = timed_sc(lambda: sc.trace_closest_device(d_cam.data_ptr(), W4 * H4, d_camhits.data_ptr(), stream.cuda_stream))
            cam_np = d_cam.cpu().numpy().view(prod.RAY_DTYPE).reshape(-1)
            camhits_np = d_camhits.cpu().numpy().view(prod.HIT_DTYPE).reshape(-1)
            bounce = prod.workloads.diffuse_bounce_rays(cam_np, camhits_np, sp_tris, seed=2)
            d_b = torch.from_numpy(bounce.view(np.float32).reshape(-1, 8)).cuda()
            d_bh = torch.empty((bounce.shape[0], 4), dtype=torch.float32, device="cuda")
            b_ms = timed_sc(lambda: sc.trace_closest_device(d_b.data_ptr(), bounce.shape[0], d_bh.data_ptr(), stream.cuda_stream))
            any_b_ms = timed_sc(lambda: sc.trace_any_device(d_b.data_ptr(), bounce.shape[0], d_occ.data_ptr(), stream.cuda_stream))
            extra["diffuse_4k"] = {"scene": "196 displaced icospheres x 5 120 faces = 1 003 520 OBJ faces (%d CLTriangle), centres uniform in [-30,30]^3, radius 4" % sp_tris.shape[0],
                                   "workload": "3840x2160 camera rays from outside -> %d primary hits -> one cosine-weighted bounce ray each" % bounce.shape[0],
                                   "primary_mrays_s": W4 * H4 * args.steps / (prim_ms * 1e-3) / 1e6,
                                   "bounce_closest_mrays_s": bounce.shape[0] * args.steps / (b_ms * 1e-3) / 1e6,
                                   "bounce_any_hit_mrays_s": bounce.shape[0] * args.steps / (any_b_ms * 1e-3) / 1e6,
                                   "bounce_hit_fraction": float((d_bh[:, 3].view(torch.int32) != -1).float().mean().item())}
            del d_cam, d_camhits, d_b, d_bh
        del sp_tris, sp_nodes, sp_mats

    # ---- device BVH build (SURVEY.md 8f-2): b2rt_build_bvh on the loader-order triangles of the same OBJ, and the same
    # ray stream through the tree it returns. Rank 0 only, outside every timed region of the headline.
    if rank == 0 and not args.skip_frames:
        loader_tris, loader_mats = prod.host.load_triangles(path)
        with prod.Context(local_rank) as bctx:
            bctx.build_bvh(loader_tris[:4096])                       # warm-up (allocator, first launches)
            t0 = time.perf_counter()
            b_tris, b_nodes, _ = bctx.build_bvh(loader_tris)
            build_s = time.perf_counter() - t0
            del loader_tris
            bctx.upload_scene(b_tris, b_nodes, loader_mats)
            nb = min(n, 1 << 24)
            d_bh = torch.empty((nb, 4), dtype=torch.float32, device="cuda")
            for _ in range(2):
                bctx.trace_closest_device(d_rays.data_ptr(), nb, d_bh.data_ptr(), stream.cuda_stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record()
                for _ in range(3):
                    bctx.trace_closest_device(d_rays.data_ptr(), nb, d_bh.data_ptr(), stream.cuda_stream)
                e1.record()
            torch.cuda.synchronize()
            same_miss = bool(torch.equal(d_bh.view(torch.int32)[:, 3] == -1, d_hits.view(torch.int32)[:nb, 3] == -1))
            # the SAH-built scene at the same launch size, measured the same way
            for _ in range(2):
                ctx.trace_closest_device(d_rays.data_ptr(), nb, d_bh.data_ptr(), stream.cuda_stream)
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                s0.record()
                for _ in range(3):
                    ctx.trace_closest_device(d_rays.data_ptr(), nb, d_bh.data_ptr(), stream.cuda_stream)
                s1.record()
            torch.cuda.synchronize()
            extra["device_bvh_build"] = {"api": "b2rt_build_bvh (Morton order + Karras hierarchy on the GPU, reference-format tree out)",
                                         "triangles": int(b_tris.shape[0]), "nodes": int(b_nodes.shape[0]),
                                         "b2rt_build_bvh_s": bctx.last_build_seconds, "with_numpy_triangle_reorder_s": build_s,
                                         "closest_mrays_s_on_device_built_tree": nb * 3 / (e0.elapsed_time(e1) * 1e-3) / 1e6,
                                         "closest_mrays_s_on_sah_tree_same_launch_size": nb * 3 / (s0.elapsed_time(s1) * 1e-3) / 1e6,
                                         "rays_per_launch": nb, "same_hit_or_miss_as_sah_tree": same_miss}
            del d_bh, b_tris, b_nodes

    # ---- end to end through the C ABI with host buffers -----------------------------------------------------------
    def e2e_step():
        ctx.trace_closest(rays_np, hits_np)      # H2D 32 B/ray, traversal, D2H 16 B/ray; synchronous
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * n * args.steps / e2e_s / 1e6
    # the same copies alone (32 B/ray in, 16 B/ray out, both directions at once, all ranks together): the bound the
    # host-buffer path is up against on this box
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def copies():
        with torch.cuda.stream(s_in):
            d_rays.copy_(host_rays, non_blocking=True)
        with torch.cuda.stream(s_out):
            host_hits.copy_(d_hits, non_blocking=True)
        s_in.synchronize(); s_out.synchronize()
    keep_hits = hits_np.copy()
    copies()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        copies()
    copy_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([copy_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        copy_s = float(t.item())
    copy_bound = world * n * args.steps / copy_s / 1e6
    hits_np[:] = keep_hits
    del keep_hits
    dev_hits = d_hits.cpu().numpy().view(prod.HIT_DTYPE).reshape(-1)
    assert np.array_equal(dev_hits["tri"], hits_np["tri"]), "host-buffer and device-resident paths disagree"
    # full-size cross-check (not timed): the on-device walk over the REFERENCE's own 48 B / 256 B arrays in the reference's
    # order must give the same hit for every ray of the step
    d_ref = torch.empty_like(d_hits)
    ctx.set_option(prod.capi.OPT_TRAVERSAL, 1)
    ctx.trace_closest_device(d_rays.data_ptr(), n, d_ref.data_ptr(), stream.cuda_stream)
    ctx.set_option(prod.capi.OPT_TRAVERSAL, 0)
    torch.cuda.synchronize()
    same_bits = bool(torch.equal(d_ref.view(torch.int32)[:, 3], d_hits.view(torch.int32)[:, 3]) and
                     torch.equal(d_ref.view(torch.int32)[:, 0], d_hits.view(torch.int32)[:, 0]))
    del d_ref

    # ---- cornell 1920x1080, 4 bounces, 16 frames accumulated = 16 spp (configs[1]) -------------------------------------
    cornell_img = None
    if rank == 0 and not args.skip_frames:
        cornell = os.path.join(ROOT, "tests", "golden", "cornell.obj")
        with prod.host.Engine(1920, 1080, device=local_rank) as ce:
            ce.load_scene(cornell, 4)
            ce.set_render(frame_count=1, bounces=4)
            for _ in range(5):
                ce.render_frame()                                # frames 1-5 of the accumulation double as warm-up (render-mode choice settles)
            t0 = time.perf_counter()
            for _ in range(11):
                ce.render_frame()                                # RenderFrame: 8 args, kernel, full 33 MB read-back, finish
            frame_ms = (time.perf_counter() - t0) / 11 * 1e3
            cornell_img = ce.pixels().copy()
            cctx = prod.Context.borrow(ce.context_handle(), local_rank)
            t0 = time.perf_counter()
            for f in range(17, 33):
                cctx.set_frame(f, 4)
                cctx.execute(1920 * 1080)
            cctx.finish()
            cornell_kernel_ms = (time.perf_counter() - t0) / 16 * 1e3
            mode_ms = {}
            for mode, name in ((0, "wavefront"), (1, "megakernel")):
                cctx.set_option(prod.capi.OPT_RENDER_MODE, mode)
                cctx.set_frame(33, 4)
                cctx.execute(1920 * 1080)
                cctx.finish()
                t0 = time.perf_counter()
                for f in range(34, 50):
                    cctx.set_frame(f, 4)
                    cctx.execute(1920 * 1080)
                cctx.finish()
                mode_ms[name] = (time.perf_counter() - t0) / 16 * 1e3
            cctx.set_option(prod.capi.OPT_RENDER_MODE, 2)
            ce.set_display_readback(True)                        # 8-bit RGBA quantised on the device: 8 MB instead of 33 MB per frame
            for _ in range(5):
                ce.render_frame()
            t0 = time.perf_counter()
            for _ in range(15):
                ce.render_frame()
            display_ms = (time.perf_counter() - t0) / 15 * 1e3
        extra["cornell_1080p_4bounce"] = {"frame_ms": frame_ms, "kernel_only_frame_ms": cornell_kernel_ms, "spp": 16,
                                          "api": "CLRaytracer::RenderFrame (args + KernelEntry + 33 MB read-back + finish)",
                                          "render_mode": "default: the faster of wavefront / megakernel as measured per launch shape (bit-identical frames)",
                                          "kernel_only_frame_ms_by_mode": mode_ms,
                                          "frame_ms_display_readback_rgba8": display_ms}

    # ---- BASELINE.json configs[3]: a 3840x2160 4-bounce frame split into screen bands over the ranks, the framebuffer
    # gathered on rank 0 -- all of it behind the C ABI (b2rt_comm_init / b2rt_comm_share_output / b2rt_execute_shard):
    # the ranks' kernels store finished pixels straight into rank 0's image over NVLink, NCCL carries the barrier.
    # Run at every N (N=1 is the baseline of the scaling curve) on the 10 M-triangle scattered scene and on cornell.
    tiled_checks = {}
    if not args.skip_frames:
        W, H, frames = 3840, 2160, 8
        scenes_t = []
        if args.tiled_faces > 0:
            tiled_path = os.path.join(SCENE_DIR, "scatter_%d.obj" % args.tiled_faces)
            t_scene = time.time()
            if rank == 0 and not os.path.exists(tiled_path + ".done"):
                scenegen("scattered", tiled_path, args.tiled_faces, 50.0, 0.05, 0.5, 11)
                prod.host.load_scene(tiled_path, 4, cache=True)          # CLOBJloader + CreateBVHTrees once; leaves the binary cache for the other ranks
                open(tiled_path + ".done", "w").close()
            barrier()
            arrays = prod.host.load_scene(tiled_path, 4, cache=True)[:3]
            log("[bench r%d] tiled scene ready in %.1f s" % (rank, time.time() - t_scene))
            scenes_t.append(("scattered", "%d scattered triangles (%d CLTriangle), edge 0.05-0.5, centres uniform in [-50,50]^3" % (args.tiled_faces, arrays[0].shape[0]),
                             arrays, dict(pos=(0.0, -140.0, 0.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))))
            del arrays
        scenes_t.append(("cornell", "cornell.obj", prod.host.load_scene(os.path.join(ROOT, "tests", "golden", "cornell.obj"), 4), {}))
        tiled = {}
        for key, name, (tris_c, nodes_c, mats_c), cam_t in scenes_t:
            with prod.Context(local_rank) as fc:
                fc.upload_scene(tris_c, nodes_c, mats_c)
                fc.resize(W, H)
                if world > 1:
                    # one NCCL communicator per context; the 128-byte id travels over torch.distributed (plumbing)
                    uid = [prod.capi.comm_unique_id() if rank == 0 else None]
                    dist.broadcast_object_list(uid, src=0)
                    fc.comm_init(uid[0], rank, world)
                    fc.comm_share_output()                              # rank 0's image becomes everybody's store-through target

                def frame(k):
                    fc.set_frame(k, 4, **cam_t)
                    if world > 1:
                        fc.execute_shard()                              # entry fence + this rank's bands + store-through + completion barrier
                    else:
                        fc.execute(W * H)
                    fc.finish()                                         # the frame is complete in rank 0's HBM

                for k in range(1, 6):                                   # warm-up; the render-mode choice of this launch shape settles
                    frame(k)
                barrier()
                t0 = time.perf_counter()
                for k in range(6, 6 + frames):
                    frame(k)
                ms = (time.perf_counter() - t0) / frames * 1e3
                barrier()
                t = torch.tensor([ms], device="cuda", dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                entry = {"scene": name + ", 3840x2160, 4 bounces", "ms_per_frame": float(t[0].item()), "frames_timed": frames,
                         "api": "b2rt_execute_shard + b2rt_finish per frame" if world > 1 else "b2rt_execute + b2rt_finish per frame",
                         "partition": "8-row bands of gid = y*W + x round robin over %d ranks" % world}
                if world > 1:
                    entry["gather"] = dict(fc.group_info(), how="kernels store finished pixels into rank 0's image (CUDA IPC mapping over NVLink); one 4-byte ncclAllReduce as entry fence (orders the stores behind rank 0's reads of the previous frame) and one as completion barrier")
                if rank == 0:
                    img = fc.read_pixels().copy()
                    tiled_checks[key] = (img, tris_c, nodes_c, mats_c, cam_t, 5 + frames)
                    if world > 1:
                        # the gathered frame must equal what one GPU renders alone, bit for bit
                        with prod.Context(local_rank) as one:
                            one.upload_scene(tris_c, nodes_c, mats_c)
                            one.resize(W, H)
                            for k in range(1, 6 + frames):
                                one.set_frame(k, 4, **cam_t)
                                one.execute(W * H)
                            alone = one.read_pixels()
                        entry["bit_identical_to_single_gpu"] = bool(np.array_equal(img.view(np.uint32), alone.view(np.uint32)))
                        del alone
                tiled[key] = entry
                barrier()
            del tris_c, nodes_c, mats_c
        if rank == 0:
            extra["tiled_frame_4k"] = tiled.get("scattered", tiled["cornell"])
            extra["tiled_frame_4k_cornell"] = tiled["cornell"]

    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        ol = checkers()
        tris, nodes, _ = eng.scene_arrays()
        cpu = cpu_baseline(ol, "reference", tris, nodes, rays_np, args.cpu_seconds, os.cpu_count() or 1)
        # parity spot check of the timed output against the checker (not timed)
        want = ol.oracle_closest(tris, nodes, rays_np[:100000])
        same = float((want["tri"] == hits_np["tri"][:100000]).mean())
        extra["parity_ids_identical_frac_100k"] = same
        extra["parity_t_bit_identical_frac_100k"] = float((want["t"] == hits_np["t"][:100000]).mean())
        # configs[0]: cornell.obj 512x512, primary rays + one shadow ray per hit towards the kernel's light (kernel_bvh.cl:307):
        # the reference's Intersect() on the host cores (stand-in for the PoCL CPU device), and the same rays on the B200
        ct0, cn0, cm0 = prod.host.load_scene(os.path.join(ROOT, "tests", "golden", "cornell.obj"), 4)
        cam = ol.oracle_camera_rays(512, 512, 1)
        threads = os.cpu_count() or 1
        closest_fn = (lambda r: ol.ref_closest(ct0, cn0, r, threads)) if ol.ref() is not None else (lambda r: ol.oracle_closest(ct0, cn0, r, threads))
        closest_fn(cam)
        t0 = time.perf_counter()
        for _ in range(5):
            closest_fn(cam)
        cpu_primary_ms = (time.perf_counter() - t0) / 5 * 1e3
        ph = ol.oracle_closest(ct0, cn0, cam, threads)
        hitm = ph["tri"] != 0xFFFFFFFF
        o = np.stack([cam["ox"], cam["oy"], cam["oz"]], 1)[hitm] + np.stack([cam["dx"], cam["dy"], cam["dz"]], 1)[hitm] * ph["t"][hitm, None]
        dl = np.array([0.0, -10.0, 16.0], dtype=np.float32) - o
        shadow = prod.workloads.pack((o + 0.01 * dl / np.linalg.norm(dl, axis=1, keepdims=True)).astype(np.float32), dl.astype(np.float32))
        ol.oracle_any(ct0, cn0, shadow, threads)
        t0 = time.perf_counter()
        for _ in range(5):
            occ_cpu = ol.oracle_any(ct0, cn0, shadow, threads)
        cpu_shadow_ms = (time.perf_counter() - t0) / 5 * 1e3
        with prod.Context(local_rank) as c0:
            c0.upload_scene(ct0, cn0, cm0)
            c0.trace_closest(cam); c0.trace_any(shadow)
            t0 = time.perf_counter()
            for _ in range(20):
                gh = c0.trace_closest(cam)
            gpu_primary_ms = (time.perf_counter() - t0) / 20 * 1e3
            t0 = time.perf_counter()
            for _ in range(20):
                occ_gpu = c0.trace_any(shadow)
            gpu_shadow_ms = (time.perf_counter() - t0) / 20 * 1e3
        extra["cornell_512_primary_plus_shadow"] = {
            "rays": {"primary": int(cam.shape[0]), "shadow": int(shadow.shape[0])},
            "cpu_reference_ms": {"primary": cpu_primary_ms, "shadow": cpu_shadow_ms, "threads": threads,
                                 "what": "reference Intersect() compiled as C++ on the host cores (PoCL unavailable); shadow rays: the oracle's early-exit variant"},
            "b200_host_buffers_ms": {"primary": gpu_primary_ms, "shadow": gpu_shadow_ms, "api": "b2rt_trace_closest / b2rt_trace_any, synchronous, copies included"},
            "identical": bool(np.array_equal(gh["tri"], ph["tri"]) and np.array_equal(occ_gpu != 0, occ_cpu != 0))}
        if cornell_img is not None:
            # the same 16 accumulated frames by the reference's KernelEntry on the host cores
            ct, cn, cm = prod.host.load_scene(os.path.join(ROOT, "tests", "golden", "cornell.obj"), 4)
            ref_img = np.zeros((1920 * 1080, 4), dtype=np.float32)
            render = ol.ref_render if ol.ref() is not None else ol.oracle_render
            t0 = time.perf_counter()
            for fc in range(1, 17):
                render(ct, cn, cm, ref_img, 1920, 1080, fc, 4, threads=os.cpu_count() or 1)
            cpu_ms = (time.perf_counter() - t0) / 16 * 1e3
            a = np.clip(np.nan_to_num(cornell_img[:, :3].astype(np.float64)), 0, 1)
            b = np.clip(np.nan_to_num(ref_img[:, :3].astype(np.float64)), 0, 1)
            mse = float(np.mean((a - b) ** 2))
            extra["cornell_1080p_4bounce"].update({"cpu_reference_frame_ms": cpu_ms, "cpu_threads": os.cpu_count() or 1,
                                                   "psnr_vs_reference_db": (10 * np.log10(1.0 / mse)) if mse > 0 else 999.0,
                                                   "pixels_bit_identical_frac": float((cornell_img[:, :3] == ref_img[:, :3]).all(axis=1).mean())})

        # configs[3] parity at FULL size: image rows of the 4K frames timed above (all accumulated frames) re-rendered by the
        # checker (oracle_render over gid ranges) and compared with the product's image
        for key, (img, t_c, n_c, m_c, cam_t, last_frame) in tiled_checks.items():
            rows = (3, 777, 1080, 2100)
            want = np.zeros((3840 * 2160, 4), dtype=np.float32)
            for fcnt in range(1, last_frame + 1):
                for y in rows:
                    ol.oracle_render(t_c, n_c, m_c, want, 3840, 2160, fcnt, 4, gid0=y * 3840, gid1=(y + 1) * 3840, threads=os.cpu_count() or 1, **cam_t)
            sel = np.concatenate([np.arange(y * 3840, (y + 1) * 3840) for y in rows])
            a = np.clip(np.nan_to_num(img[sel, :3].astype(np.float64)), 0, 1)
            b = np.clip(np.nan_to_num(want[sel, :3].astype(np.float64)), 0, 1)
            mse = float(np.mean((a - b) ** 2))
            extra["tiled_frame_4k" if key == "scattered" or "scattered" not in tiled_checks else "tiled_frame_4k_cornell"].update({
                "parity_vs_oracle_pixels": {"pixels": int(sel.size), "frames_accumulated": last_frame, "psnr_db": (10 * np.log10(1.0 / mse)) if mse > 0 else 999.0,
                                            "bit_identical_frac": float((img[sel, :3] == want[sel, :3]).all(axis=1).mean())}})
    tiled_checks.clear()

    if rank == 0:
        peaks, which = measured_peaks()
        achieved = n * bytes_per_ray / (kernel_ms * 1e-3) / 1e9
        traffic_gb, ncu_metrics = measured_traffic(args.frequency, n)
        compulsory = (info["wide_node_bytes"] + info["leaf_bytes"] + 48.0 * n) / (kernel_ms * 1e-3) / 1e9
        # instruction-issue roofline: warp instructions per ray (ncu smsp__inst_executed.sum of the same launch, profiles/) x rays
        # against SMs x 4 schedulers x the SM clock sampled during the timed region
        issue_frac, issue_what = None, "no ncu capture of this workload committed"
        wipr = (ncu_metrics or {}).get("warp_instructions_per_ray")
        sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz")
        if wipr and sm_mhz:
            issue_peak = info["sm_count"] * 4 * sm_mhz * 1e6
            issue_frac = wipr * n / (kernel_ms * 1e-3) / issue_peak
            issue_what = "%.1f warp instructions per ray (ncu, profiles/) x %d rays / %.2f ms, against %d SMs x 4 issue slots x %.0f MHz" % (
                wipr, n, kernel_ms, info["sm_count"], sm_mhz)
        out = {
            "metric": "closest_hit_ray_throughput", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args, info["n_triangles"]), "rays_per_gpu_per_step": n,
                       "bvh": "replicated per GPU; %d wide nodes (%.1f MB) + %d leaf blocks (%.1f MB)" % (
                           info["n_wide_nodes"], info["wide_node_bytes"] / 1e6, info["n_leaf_blocks"], info["leaf_bytes"] / 1e6),
                       "parallelism": "ray stream sharded by rank, no data-path collective" if world > 1 else "single GPU",
                       "l2": "ray + hit streams (%.0f MB per step) exceed the 126 MB L2; the BVH is re-used from L2 across steps by design" % (n * 48 / 1e6)},
            "any_hit": {"value": any_value, "unit": "Mrays/s"},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": n * 16,
                    "api": "b2rt_trace_closest (pinned host buffers, chunked H2D/kernel/D2H pipeline)",
                    "copy_only_bound": copy_bound, "frac_of_copy_only_bound": e2e_value / copy_bound,
                    "copy_only_bound_what": "the step's pinned H2D + D2H copies alone, both directions at once, all ranks together (max over ranks)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "issue", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         "what": "achieved = ALGORITHMIC (requested) bytes per launch / kernel time, against the measured HBM copy peak as the contract asks; "
                                 "the bytes are served by L1/L2 (see traffic), and the kernel's limiter is instruction issue: issue_frac is the roofline that bounds it",
                         "issue_frac": issue_frac, "issue_what": issue_what,
                         "traffic": traffic_gb, "traffic_unit": "GB per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/)",
                         "dram_frac_of_hbm_peak": (traffic_gb / (kernel_ms * 1e-3) / peaks["hbm_gbs"]) if traffic_gb else None,
                         "compulsory_floor_gbs": compulsory, "ncu_same_launch": ncu_metrics,
                         "algorithmic_gb_per_launch": n * bytes_per_ray / 1e9, "peak_source": "measured copy bandwidth (MEASURED_PEAKS.json)" if which == "measured" else "of fallback (6.65 TB/s, B200_PROFILING.md; MEASURED_PEAKS.json absent)",
                         "kernel": "trace_persistent<closest> (+ trace_tail_kernel)", "kernel_ms": kernel_ms,
                         "bytes_per_ray": bytes_per_ray, "traversal_bytes_per_ray": trav_bytes,
                         "per_ray": {k: v / max(cnt["rays"], 1) for k, v in cnt.items() if k not in ("rays", "max_steps_per_ray", "stack_overflows")},
                         "max_steps_of_one_ray": cnt["max_steps_per_ray"], "stack_overflows": cnt["stack_overflows"]},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        out["parity_full_step_vs_reference_layout_walk"] = {"rays": n, "ids_and_t_bit_identical": same_bits,
                                                            "kind": "self-comparison: the wide-BVH kernel against the product's own one-thread-per-ray walk over the reference's "
                                                                    "48 B / 256 B arrays in the reference's order (itself oracle-checked at test sizes); the oracle comparison of "
                                                                    "this run is parity_ids_identical_frac_100k"}
        out.update(extra)
        emit(out)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def emit(obj):
    """The ONE JSON line goes to the process's original stdout; everything else (NCCL banners, library
    chatter) was re-pointed at stderr in main()."""
    line = json.dumps(obj) + "\n"
    if _JSON_FD is None:
        sys.stdout.write(line)
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line.encode())


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rays", type=int, default=100_000_000, help="rays per GPU per step (BASELINE.json configs[4]: 100M random rays)")
    ap.add_argument("--frequency", type=int, default=224, help="geodesic frequency: 20*f^2 OBJ faces")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--ref-rays", type=int, default=1 << 22, help="--impl reference: rays per step (bounded sample)")
    ap.add_argument("--tiled-faces", type=int, default=10_000_000, help="tiled 4K frame (BASELINE.json configs[3]): OBJ faces of the scattered scene; 0 = cornell.obj only")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-frames", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's hits (and any-hit flags) for a seeded sample of the rays as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.warmup < 3 and args.impl == "b200":
        log("[bench] note: --warmup %d < 3; the timing rules ask for >= 3" % args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
