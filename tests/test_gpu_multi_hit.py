"""-m gpu: the k nearest hits per ray (b2rt_trace_multi[_device]) through the C ABI. k = 1 must equal b2rt_trace_closest bit
for bit; larger k must equal the oracle's k-list walk (tests/multi_hit/oracle_multi.c) bit for bit, on the wide BVH and on
the reference-layout walk, in the counting build, from host and device buffers, on device-built and refitted scenes and on
a device group."""
import ctypes as C
import os

import numpy as np
import pytest

import deep_trees as dt
import multi_hit_lib as ml
import oracle_lib as ol
import scenes
from test_gpu_round2 import _counted, _deform, _device_list
from test_multi_hit_oracle import _same_rows

pytestmark = pytest.mark.gpu
MISS = 0xFFFFFFFF
KS = (2, 3, 8, 64)


@pytest.fixture(scope="module")
def bumpy(product, bumpy_ref):
    ctx = product.Context(0)
    ctx.upload_scene(*bumpy_ref)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def cornell(product, cornell_ref):
    ctx = product.Context(0)
    ctx.upload_scene(*cornell_ref)
    yield ctx
    ctx.close()


def _bounce(tris, hits, rays, seed):
    return scenes.bounce_rays(rays, hits, scenes.tri_normals(tris, hits), seed=seed)


def _vs_oracle(ctx, tris, nodes, rays, ks=KS):
    for k in ks:
        _same_rows(ctx.trace_multi(rays, k), ml.oracle_trace_multi(tris, nodes, rays, k))


def _negative_rows(h):
    return ((h["tri"] != MISS) & (h["t"] < 0)).any(-1).sum()


def test_k1_equals_closest(bumpy, bumpy_ref, cornell, cornell_ref):
    """k = 1: bit-identical to trace_closest (t, u, v, tri; misses included) on the 1 M-ray shell stream over the displaced
    sphere and its bounce rays, and on cornell camera and bounce rays."""
    rays = scenes.shell_rays(1 << 20, 10.0, seed=201)
    for ctx, (tris, _, _), r in ((bumpy, bumpy_ref, rays), (cornell, cornell_ref, ol.oracle_camera_rays(512, 512, 1))):
        c = ctx.trace_closest(r)
        _same_rows(ctx.trace_multi(r, 1), c[:, None])
        b = _bounce(tris, c, r, seed=202)
        _same_rows(ctx.trace_multi(b, 1), ctx.trace_closest(b)[:, None])


def test_cornell_loader_copies(cornell, cornell_ref):
    tris, nodes, _ = cornell_ref
    rays = np.concatenate([ol.oracle_camera_rays(256, 256, 1), scenes.box_rays(40000, (-9, -2, -1), (9, 16, 17), seed=203)])
    _vs_oracle(cornell, tris, nodes, rays)
    h = cornell.trace_multi(rays, 2)
    pair = (h["tri"][:, 1] != MISS) & (h["t"][:, 0].view(np.uint32) == h["t"][:, 1].view(np.uint32))
    assert pair.mean() > 0.3                                   # the two copies of a face: two hits at one t


def test_ties_scattered_and_negative_t(product, tmp_scene_dir, bumpy, bumpy_ref):
    p, n, f = scenes.tie_grid(24, layers=3)
    path = scenes.write_obj(os.path.join(tmp_scene_dir, "gm_ties.obj"), p, n, f)
    tris, nodes, mats = product.host.load_scene(path)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        rays = scenes.tie_rays(24)
        _vs_oracle(ctx, tris, nodes, rays)
        h = ctx.trace_multi(rays, 8)
        assert ((h["tri"][:, 1:] != MISS) & (h["t"][:, 1:].view(np.uint32) == h["t"][:, :-1].view(np.uint32))).any(-1).mean() > 0.5
    p, n, f = scenes.scattered_triangles(20000)
    path = scenes.write_obj(os.path.join(tmp_scene_dir, "gm_scatter.obj"), p, n, f)
    tris, nodes, mats = product.host.load_scene(path)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        _vs_oracle(ctx, tris, nodes, scenes.box_rays(30000, (-55, -55, -55), (55, 55, 55), seed=204))
    tris, nodes, _ = bumpy_ref
    rays = scenes.shell_rays(30000, 10.0, seed=205)
    b = _bounce(tris, bumpy.trace_closest(rays), rays, seed=206)
    inside = scenes.box_rays(20000, (-9, -9, -9), (9, 9, 9), seed=207)
    r = np.concatenate([b, inside])
    _vs_oracle(bumpy, tris, nodes, r)
    assert _negative_rows(bumpy.trace_multi(r, 8)) > 100


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255])
def test_chain_at_every_stack_capacity(product, tmp_scene_dir, depth):
    tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, depth)
    rays = dt.chain_rays(depth + 1, 6000, seed=depth)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        for k in (1, 3, 64):
            want = ml.oracle_trace_multi(tris, nodes, rays, k)
            got, c = _counted(product, ctx, lambda: ctx.trace_multi(rays, k))
            _same_rows(got, want)
            assert c["rays"] == rays.shape[0] and c["stack_overflows"] == 0, c
            ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
            _same_rows(ctx.trace_multi(rays, k), want)
            ctx.set_option(product.capi.OPT_TRAVERSAL, 0)


def test_reference_layout_walk_and_counting_build(product, bumpy, bumpy_ref):
    tris, nodes, _ = bumpy_ref
    rays = scenes.shell_rays(200000, 10.0, seed=208)
    r = np.concatenate([rays, _bounce(tris, bumpy.trace_closest(rays), rays, seed=209)])
    for k in (1,) + KS:
        wide = bumpy.trace_multi(r, k)
        bumpy.set_option(product.capi.OPT_TRAVERSAL, 1)
        try:
            _same_rows(bumpy.trace_multi(r, k), wide)
        finally:
            bumpy.set_option(product.capi.OPT_TRAVERSAL, 0)
        got, c = _counted(product, bumpy, lambda: bumpy.trace_multi(r, k))
        _same_rows(got, wide)
        assert c["rays"] == r.shape[0] and c["stack_overflows"] == 0, c


def test_device_entry_matches_host_entry(product, bumpy, bumpy_ref):
    """Device buffers on a non-default torch stream, n = 1 (mod 64), launches of 16 rays (the pool is dry at once), small
    tmax; the cooperative tail options are accepted and have no effect."""
    import torch
    tris, _, _ = bumpy_ref
    rays = scenes.shell_rays(64 * 1500 + 1, 10.0, seed=210)
    rays = np.concatenate([rays[:60000], _bounce(tris, bumpy.trace_closest(rays[60000:]), rays[60000:], seed=211)])
    rays = rays[:(rays.shape[0] - 1) // 64 * 64 + 1].copy()     # bounce rays exist only for hits: trim to n = 1 (mod 64)
    rays["tmax"][::3] = np.float32(2.5)
    assert rays.shape[0] % 64 == 1
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda()
    side = torch.cuda.Stream()
    cap = product.capi
    for coop, resume in ((-1, 0), (16, 0), (8, 16)):
        bumpy.set_option(cap.OPT_COOP_MAX, coop)
        bumpy.set_option(cap.OPT_RESUME_MAX, resume)
        for k in (1, 3, 64):
            want = bumpy.trace_multi(rays, k)
            d_hits = torch.full((rays.shape[0] * k, 4), -7, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()                           # the fill ran on torch's stream
            with torch.cuda.stream(side):
                bumpy.trace_multi_device(d_rays.data_ptr(), rays.shape[0], k, d_hits.data_ptr(), side.cuda_stream)
            side.synchronize()
            got = d_hits.cpu().numpy().view(ol.HIT).reshape(rays.shape[0], k)
            _same_rows(got, want)
            m = 1024 if k < 64 else 256
            d_small = torch.full((m * k, 4), -7, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            for i in range(0, m, 16):
                bumpy.trace_multi_device(d_rays[i:].data_ptr(), 16, k, d_small[i * k:].data_ptr(), 0)
            bumpy.finish()
            _same_rows(d_small.cpu().numpy().view(ol.HIT).reshape(m, k), want[:m])
    bumpy.set_option(cap.OPT_COOP_MAX, -1)
    bumpy.set_option(cap.OPT_RESUME_MAX, 0)


def test_invalid_arguments_write_nothing(product, cornell):
    import torch
    L, h, cap = cornell._L, cornell._h, product.capi
    rays = scenes.box_rays(100, (-9, -2, -1), (9, 16, 17), seed=212)
    hits = np.full(100 * 65 * 4, 0xA5A5A5A5, dtype=np.uint32)
    before = hits.copy()
    rp, hp = C.c_void_p(rays.ctypes.data), C.c_void_p(hits.ctypes.data)
    for k in (0, 65, 1 << 31):
        assert L.b2rt_trace_multi(h, rp, 100, k, hp) == -30
    assert L.b2rt_trace_multi(h, None, 100, 4, hp) == -30
    assert L.b2rt_trace_multi(h, rp, 100, 4, None) == -30
    assert L.b2rt_trace_multi(h, None, 0, 4, None) == 0
    assert L.b2rt_trace_multi(None, rp, 100, 4, hp) == -34
    assert np.array_equal(hits, before)
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda()
    d_hits = torch.full((100 * 65, 4), -7, dtype=torch.int32, device="cuda")
    for k in (0, 65):
        assert L.b2rt_trace_multi_device(h, C.c_void_p(d_rays.data_ptr()), 100, k, C.c_void_p(d_hits.data_ptr()), None) == -30
    assert L.b2rt_trace_multi_device(h, None, 100, 2, C.c_void_p(d_hits.data_ptr()), None) == -30
    assert L.b2rt_trace_multi_device(h, C.c_void_p(d_rays.data_ptr()), 100, 2, None, None) == -30
    assert L.b2rt_trace_multi_device(h, None, 0, 2, None, None) == 0
    cornell.finish()
    assert (d_hits == -7).all()
    with pytest.raises(cap.B2RTError):
        cornell.trace_multi(rays, 0)
    assert cornell.trace_multi(rays, cap.MULTI_MAX_HITS).shape == (100, cap.MULTI_MAX_HITS)   # still usable


def test_device_built_and_refitted_scene(product, tmp_scene_dir):
    import torch
    from test_gpu_device_scene import _device_build
    p, n, f = scenes.displaced_sphere(4)
    lt, mats = product.host.load_triangles(scenes.write_obj(os.path.join(tmp_scene_dir, "gm_dev.obj"), p, n, f))
    with product.Context(0) as ctx:
        _device_build(product, ctx, lt, mats)
        tris, nodes = ctx.read_scene()
        rays = scenes.shell_rays(30000, 10.0, seed=213)
        r = np.concatenate([rays, _bounce(tris, ctx.trace_closest(rays), rays, seed=214)])
        _vs_oracle(ctx, tris, nodes, r)
        new = _deform(tris, 1.03, 0.3)
        d_new = torch.from_numpy(new.copy()).cuda()
        status = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.refit_scene_device(d_new.data_ptr(), new.shape[0], status.data_ptr())
        ctx.finish()
        assert int(status.item()) == 0
        tris2, nodes2 = ctx.read_scene()
        assert np.array_equal(tris2, new)
        _vs_oracle(ctx, tris2, nodes2, r)


def test_device_group_equals_one_device(product, bumpy_ref):
    tris, nodes, mats = bumpy_ref
    rays = scenes.shell_rays(300001, 10.0, seed=215)
    with product.Context(0) as one, product.Context(_device_list(product, 2)) as grp:
        one.upload_scene(tris, nodes, mats)
        grp.upload_scene(tris, nodes, mats)
        for k in (1, 8, 64):
            want = one.trace_multi(rays, k)
            _same_rows(grp.trace_multi(rays, k), want)
        import torch
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1, 32).copy()).cuda(0)
        d_hits = torch.empty((rays.shape[0] * 8, 4), dtype=torch.int32, device="cuda:0")
        grp.trace_multi_device(d_rays.data_ptr(), rays.shape[0], 8, d_hits.data_ptr())
        grp.finish()
        _same_rows(d_hits.cpu().numpy().view(ol.HIT).reshape(-1, 8), one.trace_multi(rays, 8))


def test_cpp_mirror(product, cornell):
    """CLRaytracer::TraceMulti through the C shim and host.Engine: the same rows as the C ABI."""
    rays = ol.oracle_camera_rays(128, 128, 1)
    with product.host.Engine(160, 120, device=0) as eng:
        eng.load_scene(scenes.CORNELL, 4)
        for k in (1, 4):
            _same_rows(eng.trace_multi(rays, k), cornell.trace_multi(rays, k))
