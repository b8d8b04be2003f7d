"""-m gpu: path-traced radiance of a caller's ray stream (b2rt_trace_radiance[_device]) through the C ABI, bit for bit
against the radiance oracle (tests/radiance/oracle_radiance.c: the oracle's path loop over the kernels' powf / sinf / cosf),
radiance and RNG state of every record: cornell under every light type, sky and bounce count, the GGX material sweep and
seeds whose rnd() is exactly 0 or 1, degenerate directions, rays from inside closed meshes, a tie grid, deep chains at every
stack capacity, device-built and refitted scenes, and the 1 M-face bench scene (wavefront against the reference-layout walk,
and a sample against the oracle). Also: wavefront lanes, the multi-pass split, host against device entries, the counting
build, rejected arguments, a device group, the C++ mirror, and frames interleaved with radiance launches on another stream."""
import ctypes as C
import os

import numpy as np
import pytest

import deep_trees as dt
import frame_oracle_lib as fl
import radiance_lib as rl
import scenes
from test_gpu_frame_exact import _assert_frame, _material_sweep, seeds_drawing_one
from test_gpu_round2 import _counted, _deform
from test_radiance_oracle import cornell_rays, seeds_for

pytestmark = pytest.mark.gpu


def _check(product, ctx, scene, rays, seeds, bounces, light_type=0, sky=1.0, binary=True):
    """Host entry (and, with binary, the reference-layout walk) against the oracle; returns the records."""
    tris, nodes, mats = scene
    ctx.set_shading(bounces, light_type, sky)
    want = rl.oracle_radiance(tris, nodes, mats, rays, seeds, bounces, light_type, sky)
    rl.same(ctx.trace_radiance(rays, seeds), want)
    if binary:
        ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
        try:
            rl.same(ctx.trace_radiance(rays, seeds), want)
        finally:
            ctx.set_option(product.capi.OPT_TRAVERSAL, 0)
    return want


def _odd_rays(lo, hi, seed):
    """Zero, NaN and inf direction components, a zero direction, and axis-parallel rays."""
    rng = np.random.default_rng(seed)
    o = rng.uniform(lo, hi, (64, 3))
    d = rng.normal(size=(64, 3))
    d[0:8, 0] = 0.0; d[8:16, 1] = 0.0; d[16:20, :2] = 0.0; d[20:24] = 0.0
    d[24:28, 0] = np.nan; d[28:32, 2] = np.nan; d[32:36, 1] = np.inf; d[36:40, 2] = -np.inf; d[40:42] = np.inf
    o[42:44, 0] = np.nan
    return np.concatenate([scenes.pack_rays(o, d), scenes.axis_rays(lo, hi, 16, seed=seed + 1)])


def test_cornell_every_light_type_sky_and_bounce_count(product, cornell_ref):
    tris, nodes, mats = cornell_ref
    sets = cornell_rays(tris, nodes)
    rays = np.concatenate([sets["camera"], sets["bounce"], sets["inside"], _odd_rays((-4, -4, 1), (4, 4, 9), 601)])
    seeds = seeds_for(rays.shape[0], 602)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        for lt in (0, 1, 2):
            for bounces in (0, 1, 4, 8):
                for sky in ((1.0, 0.3) if bounces == 4 else (1.0,)):
                    want = _check(product, ctx, cornell_ref, rays, seeds, bounces, lt, sky, binary=bounces in (0, 4))
                    if bounces == 0:
                        assert (want["r"] == 0).all() and (want["seed"] == seeds).all()
        for bounces in (-1, -7):                                         # bounces <= 0: {0, 0, 0, seed}
            ctx.set_shading(bounces, 1, 1.0)
            got = ctx.trace_radiance(rays, seeds)
            assert (got["r"] == 0).all() and (got["g"] == 0).all() and (got["b"] == 0).all() and (got["seed"] == seeds).all()
        # a short tmax: segment 0 misses and takes the sky, no random number is drawn
        short = sets["camera"].copy()
        short["tmax"] = 0.5
        want = _check(product, ctx, cornell_ref, short, seeds[: short.shape[0]], 4, 1, 0.6)
        assert (want["seed"] == seeds[: short.shape[0]]).all()


def test_material_sweep_and_extreme_seeds(product, cornell_ref):
    """GGX lobes of every roughness, and seeds whose n-th rnd() is exactly 1.0 (or 0.0: seed 0 stays 0)."""
    tris, nodes, _ = cornell_ref
    t2, m2 = _material_sweep(cornell_ref[2], tris, np.random.default_rng(603))
    scene = (t2, nodes, m2)
    cam = cornell_rays(tris, nodes)["camera"]
    extreme = [0] + [s for draw in (1, 2, 3, 4) for above in (True, False) for s in seeds_drawing_one(draw, above, 6)]
    extreme = np.array(extreme, dtype=np.uint32)
    rays = np.concatenate([cam, np.tile(cam[200:232], (extreme.size + 31) // 32)[: extreme.size]])
    seeds = np.concatenate([seeds_for(cam.shape[0], 604), extreme])
    with product.Context(0) as ctx:
        ctx.upload_scene(*scene)
        for lt in (0, 1, 2):
            _check(product, ctx, scene, rays, seeds, 6, lt, 1.0, binary=lt == 1)
        _check(product, ctx, scene, rays, seeds, 9, 1, 2.5, binary=False)


def test_inside_closed_meshes_and_tie_grid(product, bumpy_ref, tmp_scene_dir):
    tris, nodes, mats = bumpy_ref
    rays = np.concatenate([scenes.box_rays(3000, (-9, -9, -9), (9, 9, 9), seed=605), scenes.shell_rays(3000, 10.0, seed=606),
                           _odd_rays((-9, -9, -9), (9, 9, 9), 607)])
    seeds = seeds_for(rays.shape[0], 608)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        _check(product, ctx, bumpy_ref, rays, seeds, 5, 1, 1.0)
        _check(product, ctx, bumpy_ref, rays, seeds, 3, 2, 0.5, binary=False)
    p, n, f = scenes.tie_grid(24, layers=3)
    scene = product.host.load_scene(scenes.write_obj(os.path.join(tmp_scene_dir, "rad_ties.obj"), p, n, f), 4)
    rays = scenes.tie_rays(24, seed=609)
    with product.Context(0) as ctx:
        ctx.upload_scene(*scene)
        _check(product, ctx, scene, rays, seeds_for(rays.shape[0], 610), 4, 1, 1.0)


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255])
def test_chain_at_every_stack_capacity(product, tmp_scene_dir, depth):
    scene = dt.chain(product.host, tmp_scene_dir, depth)
    tris, nodes, _ = scene
    rays = dt.chain_rays(depth + 1, 1200, 611 + depth)
    with product.Context(0) as ctx:
        ctx.upload_scene(*scene)
        want = _check(product, ctx, scene, rays, seeds_for(rays.shape[0], 613 + depth), 4, 1, 1.0)
        got, c = _counted(product, ctx, lambda: ctx.trace_radiance(rays, seeds_for(rays.shape[0], 613 + depth)))
        rl.same(got, want)
        assert c["stack_overflows"] == 0, c


def test_device_built_then_refitted_scene(product, tmp_scene_dir):
    """A device-built scene, then the same scene refitted on the device (b2rt_refit_scene_device)."""
    import torch
    from test_gpu_device_refit import _dev, _device_build, _load, _refit_device, _to_loader
    lt, mats = _load(product, tmp_scene_dir, "rad_dev.obj", *scenes.displaced_sphere(4))
    with product.Context(0) as ctx:
        order, d_order = _device_build(ctx, lt, mats)
        tris, nodes = ctx.read_scene()
        rays = np.concatenate([scenes.shell_rays(4000, 10.0, seed=614), scenes.box_rays(1000, (-8, -8, -8), (8, 8, 8), seed=615)])
        seeds = seeds_for(rays.shape[0], 616)
        _check(product, ctx, (tris, nodes, mats), rays, seeds, 4, 1, 1.0)
        new = _deform(tris, 1.2, 0.7)
        assert _refit_device(ctx, _dev(_to_loader(new, order)), tris.shape[0], d_order) == 0
        _check(product, ctx, (new, ctx.read_nodes(), mats), rays, seeds, 4, 2, 1.0)
        torch.cuda.synchronize()


def test_bench_scene_full_size(product):
    """The 1 M-face bench scene: 2^20 rays (half of them diffuse bounce rays, which mostly leave the sphere, half the shell
    rays they came from) on the wavefront equal the reference-layout walk, and a 2 000-ray sample equals the oracle."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    path = bench.ensure_scene(224, 0, 1, lambda: None)
    tris, nodes, mats = product.host.load_scene(path, 4, cache=True)[:3]
    shell = product.workloads.shell_rays(1300000, bench.RADIUS, seed=617)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        bounce = product.workloads.diffuse_bounce_rays(shell, ctx.trace_closest(shell), tris, seed=618)[: 1 << 19]
        bounce = np.concatenate([bounce, shell[: 1 << 19]])
        assert bounce.shape[0] == 1 << 20
        seeds = seeds_for(bounce.shape[0], 619)
        ctx.set_shading(4, 1, 1.0)
        wide = ctx.trace_radiance(bounce, seeds)
        ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
        rl.same(ctx.trace_radiance(bounce, seeds), wide)
        ctx.set_option(product.capi.OPT_TRAVERSAL, 0)
        sample = np.linspace(0, bounce.shape[0] - 1, 2000).astype(np.int64)
        rl.same(wide[sample], rl.oracle_radiance(tris, nodes, mats, bounce[sample], seeds[sample], 4, 1, 1.0))
        assert (wide["seed"] != seeds).mean() > 0.4                   # the shell half shades at least one hit


def test_lanes_chunks_and_counters(product, bumpy_ref):
    import torch
    tris, nodes, mats = bumpy_ref
    rays = np.concatenate([scenes.shell_rays(20000, 10.0, seed=620), scenes.box_rays(5003, (-9, -9, -9), (9, 9, 9), seed=621)])
    assert rays.shape[0] % 32 != 0
    seeds = seeds_for(rays.shape[0], 622)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        want = _check(product, ctx, bumpy_ref, rays, seeds, 4, 1, 1.0, binary=False)
        for lanes in (1, 2, 3, 4):
            ctx.set_option(product.capi.OPT_WAVEFRONT_LANES, lanes)
            rl.same(ctx.trace_radiance(rays, seeds), want)
        ctx.set_option(product.capi.OPT_WAVEFRONT_LANES, 0)
        for coop in (0, 16):
            ctx.set_option(product.capi.OPT_COOP_MAX, coop)
            rl.same(ctx.trace_radiance(rays, seeds), want)
        ctx.set_option(product.capi.OPT_COOP_MAX, -1)
        ctx.set_option(product.capi.OPT_RESUME_MAX, 12)
        rl.same(ctx.trace_radiance(rays, seeds), want)
        ctx.set_option(product.capi.OPT_RESUME_MAX, 0)
        ctx.set_option(product.capi.OPT_RENDER_MODE, 1)                  # ignored
        rl.same(ctx.trace_radiance(rays, seeds), want)
        ctx.set_option(product.capi.OPT_RENDER_MODE, 2)
        # the counting build: the same records; rays = segments traced, at least one per path with bounces > 0
        got, c = _counted(product, ctx, lambda: ctx.trace_radiance(rays, seeds))
        rl.same(got, want)
        assert rays.shape[0] <= c["rays"] <= 4 * rays.shape[0] and c["wide_nodes"] > 0 and c["stack_overflows"] == 0, c
        # the device entry on a side stream, and the host entry over small chunks, equal one whole device launch
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda()
        d_seeds = torch.from_numpy(seeds.view(np.int32).copy()).cuda()
        d_out = torch.full((rays.shape[0], 4), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            ctx.trace_radiance_device(d_rays.data_ptr(), d_seeds.data_ptr(), rays.shape[0], d_out.data_ptr(), side.cuda_stream)
        side.synchronize()
        whole = d_out.cpu().numpy().view(rl.RADIANCE).reshape(-1)
        rl.same(whole, want)
        os.environ["B2RT_STREAM_CHUNK"] = "1024"
        try:
            rl.same(ctx.trace_radiance(rays, seeds), whole)
        finally:
            del os.environ["B2RT_STREAM_CHUNK"]


def test_one_device_launch_over_several_wavefront_passes(product, cornell_ref):
    """WF_MAX_PATHS + 37 paths in ONE b2rt_trace_radiance_device call: two wavefront passes (the second of 37 paths, its
    work items starting at gid 2^24), the first of them cut into two lanes. Every record equals the host entry's (whose
    2^22-ray chunks cut the same paths elsewhere), and the records around both cuts and a spread sample equal the oracle."""
    import torch
    WF_MAX_PATHS = 1 << 24
    ct, cn, cm = cornell_ref
    cam = cornell_rays(ct, cn)["camera"]
    n = WF_MAX_PATHS + 37
    big = np.resize(cam, n)
    big_seeds = (np.arange(n, dtype=np.uint64) * 2654435761 % (1 << 32)).astype(np.uint32)
    with product.Context(0) as ctx:
        ctx.upload_scene(ct, cn, cm)
        ctx.set_shading(2, 1, 1.0)
        d_rays = torch.from_numpy(big.view(np.uint8).reshape(-1, 32)).cuda()
        d_seeds = torch.from_numpy(big_seeds.view(np.int32)).cuda()
        d_out = torch.full((n, 4), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            ctx.trace_radiance_device(d_rays.data_ptr(), d_seeds.data_ptr(), n, d_out.data_ptr(), side.cuda_stream)
        side.synchronize()
        got = d_out.cpu().numpy().view(rl.RADIANCE).reshape(-1)
        del d_rays, d_seeds, d_out
        pick = np.concatenate([np.arange(2000), (1 << 23) - 500 + np.arange(1000), WF_MAX_PATHS - 1000 + np.arange(1037),
                               np.linspace(0, n - 1, 3000).astype(np.int64)])
        rl.same(got[pick], rl.oracle_radiance(ct, cn, cm, big[pick], big_seeds[pick], 2, 1, 1.0))
        rl.same(got, ctx.trace_radiance(big, big_seeds))


def test_rejected_arguments(product, cornell_ref):
    import torch
    tris, nodes, mats = cornell_ref
    rays = cornell_rays(tris, nodes)["camera"][:100].copy()
    seeds = seeds_for(100, 623)
    out = np.full(400, 0xA5A5A5A5, dtype=np.uint32)
    before = out.copy()
    rp, sp, op = C.c_void_p(rays.ctypes.data), C.c_void_p(seeds.ctypes.data), C.c_void_p(out.ctypes.data)
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda()
    d_seeds = torch.from_numpy(seeds.view(np.int32).copy()).cuda()
    d_out = torch.full((100, 4), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    drp, dsp, dp = C.c_void_p(d_rays.data_ptr()), C.c_void_p(d_seeds.data_ptr()), C.c_void_p(d_out.data_ptr())

    def both(h, want):
        """The host and the device entry give the same status; neither writes a record."""
        assert ctx._L.b2rt_trace_radiance(h, rp, sp, 100, op) == want
        assert ctx._L.b2rt_trace_radiance_device(h, drp, dsp, 100, dp, None) == want
        ctx.finish()
        assert np.array_equal(out, before) and (d_out == -7).all()

    with product.Context(0) as ctx:
        L, h = ctx._L, ctx._h
        both(h, -52)                                                     # no scene
        ctx.upload_scene(tris, nodes, mats)
        both(h, -52)                                                     # slots 8-10 never set
        ctx.set_arg(product.capi.ARG_LIGHT_BOUNCES, np.int32(4))
        ctx.set_arg(product.capi.ARG_LIGHT_TYPE, np.int32(1))
        both(h, -52)                                                     # slot 10 never set
        ctx.set_arg(product.capi.ARG_SKYBOX_INTENSITY, np.float32(1.0))
        for args in ((None, sp, op), (rp, None, op), (rp, sp, None)):
            assert L.b2rt_trace_radiance(h, *args[:2], 100, args[2]) == -30
        for args in ((None, dsp, dp), (drp, None, dp), (drp, dsp, None)):
            assert L.b2rt_trace_radiance_device(h, *args[:2], 100, args[2], None) == -30
        assert L.b2rt_trace_radiance(h, None, None, 0, None) == 0
        assert L.b2rt_trace_radiance_device(h, None, None, 0, None, None) == 0
        assert L.b2rt_trace_radiance(None, rp, sp, 100, op) == -34
        assert L.b2rt_trace_radiance_device(None, drp, dsp, 100, dp, None) == -34
        ctx.finish()
        assert np.array_equal(out, before) and (d_out == -7).all()
        # the frame-only slots are not needed, and an unbound material slot is refused
        rl.same(ctx.trace_radiance(rays, seeds), rl.oracle_radiance(tris, nodes, mats, rays, seeds, 4, 1, 1.0))
    with product.Context(0) as ctx:
        for slot, data in ((1, tris), (2, nodes)):                     # a scene without a material buffer
            a, buf = np.ascontiguousarray(data), C.c_uint64(0)
            flags = product.capi.MEM_READ_ONLY | product.capi.MEM_COPY_HOST_PTR
            assert ctx._L.b2rt_buffer_create(ctx._h, flags, a.nbytes, C.c_void_p(a.ctypes.data), C.byref(buf)) == 0
            ctx.set_arg(slot, buf.value)
        ctx.set_shading(4, 1, 1.0)
        both(ctx._h, -52)


def test_device_group_and_cpp_mirror(product, cornell_ref):
    tris, nodes, mats = cornell_ref
    rays = np.concatenate([cornell_rays(tris, nodes)["camera"], scenes.box_rays(997, (-4, -4, 1), (4, 4, 9), seed=624)])
    seeds = seeds_for(rays.shape[0], 625)
    with product.Context(0) as one:
        one.upload_scene(tris, nodes, mats)
        want = _check(product, one, cornell_ref, rays, seeds, 4, 1, 1.0, binary=False)
    with product.host.Engine(160, 120, device=0) as eng:
        eng.load_scene(scenes.CORNELL, 4)
        eng.set_render(1, 4, 1, 1.0)
        eng.render_frame()
        rl.same(eng.trace_radiance(rays, seeds), want)
    if product.device_count() < 2:
        pytest.skip("needs two GPUs")
    with product.Context([0, 1]) as grp:
        grp.upload_scene(tris, nodes, mats)
        grp.set_shading(4, 1, 1.0)
        rl.same(grp.trace_radiance(rays, seeds), want)


def test_frames_interleaved_with_radiance_on_another_stream(product, cornell_ref):
    """Frames on the context's stream and radiance launches on a torch side stream, no host sync in between; both stay
    exact. The ordering is the caller's both ways: the side stream writes each launch's seeds just before the call (behind
    a delay, so a launch that did not wait for them would read the stale zeros) and copies the records right after it, and
    the copies are read after a wait for the side stream alone, before anything waits for the context's stream."""
    import torch
    tris, nodes, mats = cornell_ref
    sets = cornell_rays(tris, nodes)
    rays = np.concatenate([sets["bounce"], sets["inside"]] * 8)
    seeds = [seeds_for(rays.shape[0], 626 + k) for k in range(3)]
    W, H = 96, 80
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        ctx.resize(W, H)
        ctx.set_option(product.capi.OPT_RENDER_MODE, 0)
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda()
        d_seed_src = [torch.from_numpy(s.view(np.int32).copy()).cuda() for s in seeds]
        d_seeds = [torch.zeros_like(x) for x in d_seed_src]
        d_out = [torch.full((rays.shape[0], 4), -7, dtype=torch.int32, device="cuda") for _ in seeds]
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        copies = []
        for k in range(3):
            ctx.set_frame(k + 1, 4, light_type=1)                      # also sets the shading slots the radiance launch reads
            ctx.execute(W * H)
            with torch.cuda.stream(side):
                torch.cuda._sleep(20000000)                            # ~10 ms of the side stream before the seeds exist
                d_seeds[k].copy_(d_seed_src[k])
                ctx.trace_radiance_device(d_rays.data_ptr(), d_seeds[k].data_ptr(), rays.shape[0], d_out[k].data_ptr(), side.cuda_stream)
                copies.append(d_out[k].clone())
        side.synchronize()                                             # the side stream only: the context's stream is not waited for
        got = [c.cpu().numpy().view(rl.RADIANCE).reshape(-1) for c in copies]
        img = ctx.read_pixels()
        want_img = np.zeros((W * H, 4), dtype=np.float32)
        for k in range(3):
            fl.oracle_render(tris, nodes, mats, want_img, W, H, k + 1, 4, light_type=1)
            rl.same(got[k], rl.oracle_radiance(tris, nodes, mats, rays, seeds[k], 4, 1, 1.0))
        _assert_frame(img, want_img, "interleaved frames")
