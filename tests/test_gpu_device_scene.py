"""b2rt_build_scene_device: a whole scene built on the GPU from loader-order triangles already in device memory. The binary
tree, triangle order and re-ordered triangles must equal b2rt_build_bvh's (host-fed) byte for byte, and the compressed wide
BVH derived on the device must equal the host derivation of b2rt_upload_scene on the same arrays byte for byte."""
import ctypes as C
import os

import numpy as np
import pytest

import device_scene_lib as dsl
import oracle_lib as ol
import scenes
from test_gpu_parity import _check_hits, _render

pytestmark = pytest.mark.gpu
MISS = 0xFFFFFFFF
INVALID_VALUE, INVALID_ARG_VALUE = -30, -50


def _device_build(product, ctx, lt, mats):
    """Materials bound, loader triangles to the device, b2rt_build_scene_device; returns (order, n_nodes)."""
    ctx.set_materials(mats)
    src = dsl.DeviceTriangles(ctx, lt, product.capi)
    n = src.n
    obuf, optr = C.c_uint64(0), C.c_void_p()
    ctx._ck(ctx._L.b2rt_buffer_create(ctx._h, product.capi.MEM_WRITE_ONLY, 4 * n, None, C.byref(obuf)))
    ctx._ck(ctx._L.b2rt_device_pointer(ctx._h, obuf, C.byref(optr), None))
    try:
        _, _, n_nodes = ctx.build_scene_device(src.ptr, n, d_order=optr.value)
        order = np.empty(n, dtype=np.uint32)
        ctx._ck(ctx._L.b2rt_read_buffer(ctx._h, obuf, C.c_void_p(order.ctypes.data), order.nbytes))
        ctx.finish()
    finally:
        src.release()
        ctx._ck(ctx._L.b2rt_buffer_release(ctx._h, obuf.value))
    return order, n_nodes


def _load(product, path):
    return product.host.load_triangles(path)


def _scenes(product, tmp):
    """(name, loader triangles, materials) for every scene of the comparison."""
    out = []
    p, n, f = scenes.displaced_sphere(5)
    lt, mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_bumpy.obj"), p, n, f))
    out.append(("bumpy", lt, mats))
    p, n, f = scenes.tie_grid(24, layers=3)
    tie, tie_mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_ties.obj"), p, n, f))
    out.append(("tie_grid", tie, tie_mats))
    p = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]], dtype=np.float32)
    n = np.tile(np.array([[0, 0, 1]], dtype=np.float32), (4, 1))
    one, one_mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_one.obj"), p, n, np.array([[0, 1, 2]])))
    out.append(("one_face", one, one_mats))
    quad, quad_mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_quad.obj"), p, n, np.array([[0, 1, 2]]), [[0, 1, 3, 2]]))
    out.append(("quad", quad, quad_mats))
    k = 5000
    x = np.arange(k, dtype=np.float32)
    p = np.stack([np.stack([x, np.zeros(k), np.zeros(k)], 1), np.stack([x + 0.9, np.zeros(k), np.zeros(k)], 1),
                  np.stack([x + 0.45, np.ones(k), np.zeros(k)], 1)], 1).reshape(-1, 3).astype(np.float32)
    n = np.tile(np.array([[0, 0, 1]], dtype=np.float32), (3 * k, 1))
    line, line_mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_line.obj"), p, n, np.arange(3 * k).reshape(k, 3)))
    out.append(("collinear", line, line_mats))
    rng = np.random.default_rng(2024)
    for case in range(12):
        pos, faces = scenes.fuzz_scene(case, rng)
        nrm = np.tile(np.array([[0.0, 0.0, 1.0]], dtype=np.float32), (pos.shape[0], 1))
        lt, mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_fuzz%d.obj" % case), pos, nrm, faces))
        out.append(("fuzz%d" % case, lt, mats))
    # > 65536 triangles, shifted by one so that loader pairs straddle the 65536-triangle chunk cuts
    p, n, f = scenes.displaced_sphere(6)
    big, big_mats = _load(product, scenes.write_obj(os.path.join(tmp, "ds_big.obj"), p, n, f))
    out.append(("chunk_cuts", np.concatenate([big[:1], big]), big_mats))
    # a run of 700 identical triangles (groups of at most 255) in front of the lattice
    out.append(("long_run", np.concatenate([np.repeat(one[:1], 700, axis=0), tie]), tie_mats))
    # coordinates mixing tiny non-zero values (subnormals included) with large ones: the quantisation edge
    bumpy = out[0][1].copy()
    v = bumpy.view(np.float32).reshape(-1, 64)
    for base in (0, 20, 40):
        q = v[:, base:base + 3]
        q[:] = np.where(np.abs(q) < 3.0, q * np.float32(1e-38), q * np.float32(3e4)).astype(np.float32)
    out.append(("tiny_and_large", bumpy, out[0][2]))
    return out


def _same_derived(a, b, what):
    for key in ("wide", "leaf", "shade", "child_bin", "leaf_dir"):
        assert a[key].shape == b[key].shape, "%s: %s sizes differ" % (what, key)
        assert np.array_equal(a[key], b[key]), "%s: %s differs" % (what, key)
    assert a["stack_bound"] == b["stack_bound"], what
    assert a["scene_info"] == b["scene_info"], what


def test_same_tree_and_same_wide_bvh_as_the_host_paths(product, tmp_scene_dir):
    """(1) nodes, re-ordered triangles and order equal b2rt_build_bvh byte for byte; (2) the wide BVH, leaf blocks, shading
    records, child_bin, leaf_dir, stack bound and scene info equal the host derivation of the read-back arrays."""
    with product.Context(0) as dev, product.Context(0) as host:
        for name, lt, mats in _scenes(product, tmp_scene_dir):
            want_t, want_n, want_o = dev.build_bvh(lt)
            order, n_nodes = _device_build(product, dev, lt, mats)
            got_t, got_n = dev.read_scene()
            assert n_nodes == want_n.shape[0], name
            assert np.array_equal(order, want_o), name
            assert np.array_equal(got_n, want_n), name
            assert np.array_equal(got_t, want_t.reshape(got_t.shape)), name
            host.upload_scene(got_t, got_n, mats)
            _same_derived(dsl.derived_arrays(dev), dsl.derived_arrays(host), name)


@pytest.fixture(scope="module")
def bumpy_pair(product, tmp_scene_dir):
    """The bumpy sphere built on the device (dev) and the same arrays uploaded the old way (host)."""
    p, n, f = scenes.displaced_sphere(5)
    lt, mats = _load(product, scenes.write_obj(os.path.join(tmp_scene_dir, "ds_pair.obj"), p, n, f))
    dev, host = product.Context(0), product.Context(0)
    _device_build(product, dev, lt, mats)
    tris, nodes = dev.read_scene()
    host.upload_scene(tris, nodes, mats)
    yield dev, host, lt, tris, nodes, mats
    dev.close()
    host.close()


def test_traversal_and_frames_on_the_device_built_scene(product, bumpy_pair):
    dev, host, _, tris, nodes, _ = bumpy_pair
    rays = np.concatenate([scenes.shell_rays(200000, 10.0, seed=31), ol.oracle_camera_rays(256, 256, 1)])
    got = dev.trace_closest(rays)
    _check_hits(got, ol.oracle_closest(tris, nodes, rays))
    assert np.array_equal(dev.trace_any(rays) != 0, ol.oracle_any(tris, nodes, rays) != 0)
    b = scenes.bounce_rays(rays[:200000], got[:200000], scenes.tri_normals(tris, got[:200000]), seed=32)
    _check_hits(dev.trace_closest(b), ol.oracle_closest(tris, nodes, b))            # negative-t bounce rays included
    cam = dict(pos=(0.0, -30.0, 4.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))
    for mode in (0, 1):                                                                 # wavefront, megakernel
        for ctx in (dev, host):
            ctx.set_option(product.capi.OPT_RENDER_MODE, mode)
        a = _render(dev, 160, 120, (1, 2), 3, **cam)
        h = _render(host, 160, 120, (1, 2), 3, **cam)
        assert np.array_equal(a.view(np.uint32), h.view(np.uint32)), "render mode %d" % mode
    for ctx in (dev, host):
        ctx.set_option(product.capi.OPT_RENDER_MODE, 2)


def test_refit_after_a_device_build_and_rebinding(product, tmp_scene_dir):
    p, n, f = scenes.displaced_sphere(4)
    lt, mats = _load(product, scenes.write_obj(os.path.join(tmp_scene_dir, "ds_refit.obj"), p, n, f))
    with product.Context(0) as dev, product.Context(0) as host:
        _device_build(product, dev, lt, mats)
        tris, nodes = dev.read_scene()
        host.upload_scene(tris, nodes, mats)
        new = tris.copy()
        v = new.view(np.float32).reshape(-1, 64)
        for base in (0, 20, 40):                      # a deterministic function of each position keeps the loader's pairs
            q = v[:, base:base + 3]
            q[:] = (q * np.float32(1.1) + np.sin(q[:, [1, 2, 0]]).astype(np.float32) * np.float32(0.05)).astype(np.float32)
        dev.refit_scene(new)
        host.refit_scene(new)
        _same_derived(dsl.derived_arrays(dev), dsl.derived_arrays(host), "refit")
        assert np.array_equal(dev.read_nodes(), host.read_nodes())
        rays = scenes.shell_rays(50000, 10.0, seed=33)
        _check_hits(dev.trace_closest(rays), host.trace_closest(rays))
        # rebinding slot 1 falls back to the host derivation of whatever is bound now
        buf = C.c_uint64(0)
        dev._ck(dev._L.b2rt_buffer_create(dev._h, product.capi.MEM_READ_ONLY | product.capi.MEM_COPY_HOST_PTR, tris.nbytes,
                                          C.c_void_p(tris.ctypes.data), C.byref(buf)))
        dev.set_arg(1, buf.value)
        host.upload_scene(tris, host.read_nodes(), mats)
        _check_hits(dev.trace_closest(rays), host.trace_closest(rays))


def test_rejected_inputs_leave_the_old_scene_usable(product, bumpy_pair):
    dev, host, lt, tris, nodes, mats = bumpy_pair
    rays = scenes.shell_rays(20000, 10.0, seed=34)
    want = host.trace_closest(rays)
    L, h = dev._L, dev._h
    out = [C.c_uint64(0) for _ in range(3)]
    args = lambda: [C.byref(o) for o in out] + [None]                                     # noqa: E731
    host_tris = np.ascontiguousarray(lt)
    assert L.b2rt_build_scene_device(h, C.c_void_p(host_tris.ctypes.data), lt.shape[0], None, *args()) == INVALID_VALUE
    assert "device memory" in L.b2rt_last_error(h).decode()
    assert L.b2rt_build_scene_device(h, None, lt.shape[0], None, *args()) == INVALID_VALUE
    src = dsl.DeviceTriangles(dev, lt, product.capi)
    try:
        assert L.b2rt_build_scene_device(h, C.c_void_p(src.ptr), 0, None, *args()) == INVALID_VALUE
        assert L.b2rt_build_scene_device(h, C.c_void_p(src.ptr + 8), src.n - 1, None, *args()) == INVALID_VALUE
        assert "aligned" in L.b2rt_last_error(h).decode()
    finally:
        src.release()
    for bad in (np.nan, np.inf):
        broken = np.ascontiguousarray(lt).copy()
        broken.view(np.float32).reshape(-1, 64)[77, 21] = bad
        src = dsl.DeviceTriangles(dev, broken, product.capi)
        try:
            assert L.b2rt_build_scene_device(h, C.c_void_p(src.ptr), src.n, None, *args()) == INVALID_ARG_VALUE
        finally:
            src.release()
    _check_hits(dev.trace_closest(rays), want)
    t2, n2 = dev.read_scene()
    assert np.array_equal(t2, tris) and np.array_equal(n2, nodes)


def test_device_group_frames_equal_a_single_device(product, tmp_scene_dir):
    if product.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    p, n, f = scenes.displaced_sphere(5)
    lt, mats = _load(product, scenes.write_obj(os.path.join(tmp_scene_dir, "ds_group.obj"), p, n, f))
    cam = dict(pos=(0.0, -30.0, 4.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))
    with product.Context(0) as one, product.Context([0, 1]) as grp:
        _device_build(product, one, lt, mats)
        _device_build(product, grp, lt, mats)
        a = _render(one, 160, 120, (1,), 3, **cam)
        b = _render(grp, 160, 120, (1,), 3, **cam)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        rays = scenes.shell_rays(50000, 10.0, seed=35)
        _check_hits(grp.trace_closest(rays), one.trace_closest(rays))


def test_cpp_mirror_renders_the_python_frame(product, tmp_scene_dir):
    """CLBVHScene::CreateBVHTreesFromDevice renders the frame the Python path renders, bit for bit, and reads back the same
    arrays. The Python build is given the caller's stream while the copy that fills its input is still running there."""
    torch = pytest.importorskip("torch")
    p, n, f = scenes.displaced_sphere(5)
    lt, mats = _load(product, scenes.write_obj(os.path.join(tmp_scene_dir, "ds_mirror.obj"), p, n, f))
    lt = np.ascontiguousarray(lt)
    cam = dict(pos=(0.0, -30.0, 4.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))
    host_t = torch.from_numpy(lt.reshape(-1)).pin_memory()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d = torch.empty(host_t.numel(), dtype=torch.uint8, device="cuda")
        d.copy_(host_t, non_blocking=True)
    with product.Context(0) as ctx:
        ctx.set_materials(mats)
        ctx.build_scene_device(d.data_ptr(), lt.shape[0], stream=side.cuda_stream)     # ordered behind the copy
        tris, nodes = ctx.read_scene()
        want_t, want_n, _ = ctx.build_bvh(lt)
        assert np.array_equal(nodes, want_n) and np.array_equal(tris, want_t.reshape(tris.shape))
        py = _render(ctx, 160, 120, (1,), 3, **cam)
    side.synchronize()
    with product.host.Engine(160, 120, device=0) as eng:
        eng.build_scene_device(d.data_ptr(), lt.shape[0], mats)
        eng.set_camera(cam["pos"], cam["front"], cam["up"])
        eng.set_render(frame_count=1, bounces=3)
        eng.render_frame()
        assert np.array_equal(eng.pixels()[:, :3].view(np.uint32), py[:, :3].view(np.uint32))
        eng.read_back_scene()
        t2, n2, _ = eng.scene_arrays()
        assert np.array_equal(n2, nodes) and np.array_equal(t2.reshape(tris.shape), tris)
