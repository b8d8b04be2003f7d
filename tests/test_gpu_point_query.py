"""-m gpu: the closest-point query (b2rt_closest_point[_device]) through the C ABI, bit for bit against the brute-force
oracle (tests/point_query/oracle_point.c) on every record: cornell, a tie grid, scattered and degenerate triangles, deep
chains at every stack capacity, the 1 M-face bench scene (wide walk against the reference-layout walk, and a sample against
the oracle), device-built and refitted scenes, host against device entries, the counting build, a device group and the C++
mirror."""
import ctypes as C
import os

import numpy as np
import pytest

import deep_trees as dt
import point_query_lib as pq
import scenes
from test_gpu_round2 import _counted, _deform, _device_list
from test_point_query_oracle import positions, query_sets, same

pytestmark = pytest.mark.gpu
MISS = 0xFFFFFFFF


def _vs_oracle(product, ctx, tris, q):
    want = pq.oracle_closest_point(tris, q)
    same(ctx.closest_point(q), want)
    ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
    try:
        same(ctx.closest_point(q), want)
    finally:
        ctx.set_option(product.capi.OPT_TRAVERSAL, 0)
    return want


def _upload(product, tmp_scene_dir, name, p, n, f, max_prims=4):
    tris, nodes, mats = product.host.load_scene(scenes.write_obj(os.path.join(tmp_scene_dir, name), p, n, f), max_prims)
    ctx = product.Context(0)
    ctx.upload_scene(tris, nodes, mats)
    return ctx, tris


def test_cornell_and_max_d2_cases(product, cornell_ref):
    tris, nodes, mats = cornell_ref
    q = query_sets(positions(tris), 301)
    odd = pq.queries(np.array([[np.nan, 0, 0], [0, 0, np.nan], [np.inf, 0, 0], [0, -np.inf, 1], [3e38, 0, 0]], dtype=np.float32), np.inf)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        want = _vs_oracle(product, ctx, tris, np.concatenate([q, odd]))
        assert (want["tri"] != MISS).mean() > 0.5


def test_tie_grid_scattered_and_degenerate(product, tmp_scene_dir):
    p, n, f = scenes.tie_grid(24, layers=3)
    ctx, tris = _upload(product, tmp_scene_dir, "gp_ties.obj", p, n, f)
    with ctx:
        lattice = np.stack(np.meshgrid(np.arange(0, 24.5, 0.5), np.arange(0, 24.5, 0.5), [0.0, 0.25, -0.5, 2.0], indexing="ij"), -1)
        _vs_oracle(product, ctx, tris, np.concatenate([pq.queries(lattice.reshape(-1, 3)), query_sets(positions(tris), 302)]))
    p, n, f = scenes.scattered_triangles(20000)
    ctx, tris = _upload(product, tmp_scene_dir, "gp_scatter.obj", p, n, f)
    with ctx:
        _vs_oracle(product, ctx, tris, query_sets(positions(tris), 303))
    # degenerate triangles: repeated vertices, collinear vertices, points, next to slivers
    rng = np.random.default_rng(304)
    k = 3000
    a = rng.uniform(-5, 5, (k, 3)); b = a + rng.normal(0, 1, (k, 3)); c = rng.uniform(-5, 5, (k, 3))
    kind = np.arange(k) % 4
    b[kind == 0] = a[kind == 0]
    c[kind == 1] = a[kind == 1] + 2.0 * (b[kind == 1] - a[kind == 1])
    b[kind == 2] = a[kind == 2]; c[kind == 2] = a[kind == 2]
    c[kind == 3] = a[kind == 3] + 0.5 * (b[kind == 3] - a[kind == 3]) + rng.normal(0, 1e-3, (int((kind == 3).sum()), 3))
    pos = np.stack([a, b, c], 1).reshape(-1, 3).astype(np.float32)
    nrm = np.tile(np.array([[0.0, 0.0, 1.0]], dtype=np.float32), (pos.shape[0], 1))
    ctx, tris = _upload(product, tmp_scene_dir, "gp_degen.obj", pos, nrm, np.arange(3 * k).reshape(k, 3))
    with ctx:
        _vs_oracle(product, ctx, tris, query_sets(positions(tris), 305))


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255])
def test_chain_at_every_stack_capacity(product, tmp_scene_dir, depth):
    tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, depth)
    q = query_sets(positions(tris), 400 + depth)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        want = _vs_oracle(product, ctx, tris, q)
        got, c = _counted(product, ctx, lambda: ctx.closest_point(q))
        same(got, want)
        assert c["rays"] == q.shape[0] and c["stack_overflows"] == 0, c


def test_bench_scene_full_size(product):
    """The 1 M-face bench scene: the wide walk equals the reference-layout walk on 2^20 queries of the three measured
    kinds, and a 2 000-query sample equals the oracle."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from dev_closest_point import query_sets as bench_sets
    path = bench.ensure_scene(224, 0, 1, lambda: None)
    tris, nodes, mats = product.host.load_scene(path, 4, cache=True)[:3]
    sets = bench_sets(tris, 1 << 20, bench.RADIUS, seed=306)
    q = np.concatenate([sets["near"][: 1 << 19], sets["box"][: 1 << 18], sets["far"][: 1 << 18]])
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        wide = ctx.closest_point(q)
        ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
        same(ctx.closest_point(q), wide)
        ctx.set_option(product.capi.OPT_TRAVERSAL, 0)
        sample = np.linspace(0, q.shape[0] - 1, 2000).astype(np.int64)
        same(wide[sample], pq.oracle_closest_point(tris, q[sample]))
        assert (wide["tri"] != MISS).mean() > 0.9


def test_entries_options_and_invalid_arguments(product, bumpy_ref):
    import torch
    tris, nodes, mats = bumpy_ref
    q = query_sets(positions(tris), 307)
    q = q[:(q.shape[0] - 1) // 32 * 32 + 1].copy()
    assert q.shape[0] % 32 == 1
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        want = ctx.closest_point(q)
        same(want, pq.oracle_closest_point(tris, q))
        # device entry on a non-default torch stream
        d_q = torch.from_numpy(q.view(np.uint8).reshape(-1, 16).copy()).cuda()
        d_out = torch.full((q.shape[0], 4), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            ctx.closest_point_device(d_q.data_ptr(), q.shape[0], d_out.data_ptr(), side.cuda_stream)
        side.synchronize()
        same(d_out.cpu().numpy().view(pq.PHIT).reshape(-1), want)
        # small launches (the pool is dry at once), the counting build, the cooperative tail options (ignored)
        small = torch.full((1024, 4), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        for i in range(0, 1024, 16):
            ctx.closest_point_device(d_q[i:].data_ptr(), 16, small[i:].data_ptr(), 0)
        ctx.finish()
        same(small.cpu().numpy().view(pq.PHIT).reshape(-1), want[:1024])
        got, c = _counted(product, ctx, lambda: ctx.closest_point(q))
        same(got, want)
        assert c["rays"] == q.shape[0] and c["wide_nodes"] > 0 and c["stack_overflows"] == 0, c
        ctx.set_option(product.capi.OPT_COOP_MAX, 16)
        same(ctx.closest_point(q), want)
        ctx.set_option(product.capi.OPT_COOP_MAX, -1)
        # n = 0 and NULL pointers: status, and nothing written
        L, h = ctx._L, ctx._h
        out = np.full(q.shape[0] * 4, 0xA5A5A5A5, dtype=np.uint32)
        before = out.copy()
        qp, op = C.c_void_p(q.ctypes.data), C.c_void_p(out.ctypes.data)
        assert L.b2rt_closest_point(h, None, 100, op) == -30
        assert L.b2rt_closest_point(h, qp, 100, None) == -30
        assert L.b2rt_closest_point(h, None, 0, None) == 0
        assert L.b2rt_closest_point(h, qp, 0, op) == 0
        assert L.b2rt_closest_point(None, qp, 100, op) == -34
        assert np.array_equal(out, before)
        d_out.fill_(-7)
        torch.cuda.synchronize()
        assert L.b2rt_closest_point_device(h, None, 100, C.c_void_p(d_out.data_ptr()), None) == -30
        assert L.b2rt_closest_point_device(h, C.c_void_p(d_q.data_ptr()), 100, None, None) == -30
        assert L.b2rt_closest_point_device(h, None, 0, None, None) == 0
        ctx.finish()
        assert (d_out == -7).all()
        assert ctx.closest_point(q[:0]).shape == (0,)


def test_device_built_and_refitted_scene(product, tmp_scene_dir):
    """A device-built scene, then b2rt_refit_scene_device with deformed geometry and the query on the caller's stream with
    no synchronisation in between: the records equal the oracle over the new triangles."""
    import torch
    from test_gpu_device_scene import _device_build
    p, n, f = scenes.displaced_sphere(4)
    lt, mats = product.host.load_triangles(scenes.write_obj(os.path.join(tmp_scene_dir, "gp_dev.obj"), p, n, f))
    with product.Context(0) as ctx:
        _device_build(product, ctx, lt, mats)
        tris, nodes = ctx.read_scene()
        q = query_sets(positions(tris), 308)
        same(ctx.closest_point(q), pq.oracle_closest_point(tris, q))
        new = _deform(tris, 1.03, 0.3)
        d_new = torch.from_numpy(new.copy()).cuda()
        d_q = torch.from_numpy(q.view(np.uint8).reshape(-1, 16).copy()).cuda()
        d_out = torch.empty((q.shape[0], 4), dtype=torch.int32, device="cuda")
        status = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            ctx.refit_scene_device(d_new.data_ptr(), new.shape[0], status.data_ptr(), stream=side.cuda_stream)
            ctx.closest_point_device(d_q.data_ptr(), q.shape[0], d_out.data_ptr(), side.cuda_stream)
        side.synchronize()
        assert int(status.item()) == 0
        tris2, _ = ctx.read_scene()
        assert np.array_equal(tris2, new)
        same(d_out.cpu().numpy().view(pq.PHIT).reshape(-1), pq.oracle_closest_point(new, q))


def test_device_group_and_cpp_mirror(product, bumpy_ref, cornell_ref):
    tris, nodes, mats = bumpy_ref
    q = query_sets(positions(tris), 309)
    with product.Context(0) as one:
        one.upload_scene(tris, nodes, mats)
        want = one.closest_point(q)
    with product.Context(_device_list(product, 2)) as grp:
        grp.upload_scene(tris, nodes, mats)
        same(grp.closest_point(q), want)
    ct, cn, cm = cornell_ref
    qc = query_sets(positions(ct), 310)
    with product.host.Engine(160, 120, device=0) as eng, product.Context(0) as ctx:
        eng.load_scene(scenes.CORNELL, 4)
        ctx.upload_scene(ct, cn, cm)
        same(eng.closest_point(qc), ctx.closest_point(qc))
