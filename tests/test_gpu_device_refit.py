"""b2rt_refit_scene_device: refit the bound scene from triangles already in device memory -- scene order in a separate
buffer, in place in the bound triangle buffer, or loader order gathered through the build's order. The refitted arrays
must equal b2rt_refit_scene's (host-fed) on the same scene-order data byte for byte, hits must equal the oracle's walk over
(new triangles, refitted nodes), the call must follow the caller's stream without a host wait, report bad data in the
status word and refuse bad arguments without touching the scene."""
import ctypes as C
import os

import numpy as np
import pytest

import deep_trees as dt
import device_scene_lib as dsl
import oracle_lib as ol
import scenes
from test_gpu_device_scene import _same_derived
from test_gpu_parity import _check_hits, _render
from test_gpu_round2 import _deform

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
MISS = 0xFFFFFFFF
INVALID_VALUE, INVALID_ARG_VALUE, INVALID_KERNEL_ARGS = -30, -50, -52
CAM = dict(pos=(0.0, -30.0, 4.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))


def _dev(a, device=0):
    """A numpy record array as a CUDA uint8 tensor (16-byte aligned: torch allocations are)."""
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).to("cuda:%d" % device)


class _View:
    """Device memory at `ptr` as a torch tensor (CUDA array interface), e.g. a bound b2rt buffer."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _bound_view(ctx, slot=1):
    buf, ptr, size = C.c_uint64(0), C.c_void_p(), C.c_size_t(0)
    ctx._ck(ctx._L.b2rt_bound_buffer(ctx._h, slot, C.byref(buf)))
    ctx._ck(ctx._L.b2rt_device_pointer(ctx._h, buf, C.byref(ptr), C.byref(size)))
    return torch.as_tensor(_View(ptr.value, size.value), device="cuda:%d" % ctx.device)


def _device_build(ctx, lt, mats):
    """b2rt_build_scene_device from loader triangles in a torch tensor; returns (order as numpy, order tensor)."""
    ctx.set_materials(mats)
    d_lt = _dev(lt, ctx.device)
    d_order = torch.empty(lt.shape[0], dtype=torch.int32, device=d_lt.device)
    ctx.build_scene_device(d_lt.data_ptr(), lt.shape[0], d_order=d_order.data_ptr())
    torch.cuda.synchronize(d_lt.device)
    return d_order.cpu().numpy().view(np.uint32), d_order


def _refit_device(ctx, d_tris, n, d_order=None, stream=0, status=None):
    """b2rt_refit_scene_device; waits for the device and returns the status word."""
    st = torch.full((1,), 12345, dtype=torch.int32, device=d_tris.device) if status is None else status
    torch.cuda.synchronize(d_tris.device)
    ctx.refit_scene_device(d_tris.data_ptr(), n, st.data_ptr(), d_order=0 if d_order is None else d_order.data_ptr(), stream=stream)
    ctx.finish()
    return int(st.item())


def _to_loader(scene_tris, order):
    """Loader-order data of the scene-order triangles: loader[order[k]] = scene[k]."""
    out = np.empty_like(scene_tris)
    out[order] = scene_tris
    return out


def _load(product, tmp, name, p, n, f, max_prims=None):
    path = scenes.write_obj(os.path.join(tmp, name), p, n, f)
    return product.host.load_triangles(path) if max_prims is None else product.host.load_scene(path, max_prims)


def _cases(product, tmp):
    """(name, loader triangles, materials) to build on the device, or (name, scene tris, nodes, materials) to upload."""
    built, uploaded = [], []
    lt, mats = _load(product, tmp, "dr_bumpy.obj", *scenes.displaced_sphere(5))
    built.append(("bumpy", lt, mats))
    tie, tie_mats = _load(product, tmp, "dr_ties.obj", *scenes.tie_grid(24, layers=3))
    built.append(("tie_grid", tie, tie_mats))
    big, big_mats = _load(product, tmp, "dr_big.obj", *scenes.displaced_sphere(6))
    built.append(("chunk_cuts", np.concatenate([big[:1], big]), big_mats))      # > 65536 triangles, pairs across the cuts
    p = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    one, _ = _load(product, tmp, "dr_one.obj", p, np.tile(np.array([[0, 0, 1]], dtype=np.float32), (3, 1)), np.array([[0, 1, 2]]))
    built.append(("long_run", np.concatenate([np.repeat(one[:1], 700, axis=0), tie]), tie_mats))
    uploaded.append(("chain200",) + dt.chain(product.host, tmp, 200, axes=(0, 1, 2)))
    uploaded.append(("max_prims16",) + _load(product, tmp, "dr_mp16.obj", *scenes.displaced_sphere(4), max_prims=16))
    return built, uploaded


def test_same_bytes_as_the_host_refit(product, tmp_scene_dir):
    """Every input mode on every scene: derived arrays, refitted nodes and the bound triangles equal b2rt_refit_scene's on a
    second context given the same scene-order data, and the status is 0."""
    built, uploaded = _cases(product, tmp_scene_dir)
    rng = np.random.default_rng(77)
    for case in built + uploaded:
        name = case[0]
        with product.Context(0) as dev, product.Context(0) as host:
            if len(case) == 3:
                order, d_order = _device_build(dev, case[1], case[2])
                tris, nodes = dev.read_scene()
                mats = case[2]
            else:
                _, tris, nodes, mats = case
                dev.upload_scene(tris, nodes, mats)
                order = rng.permutation(tris.shape[0]).astype(np.uint32)          # any order serves the gather
                d_order = torch.from_numpy(order.view(np.int32)).cuda()
            host.upload_scene(tris, nodes, mats)
            n = tris.shape[0]
            for mode, (scale, wobble) in (("separate", (1.2, 0.8)), ("in_place", (0.9, 0.05)), ("loader", (1.1, 0.3))):
                new = _deform(tris, scale, wobble)
                if mode == "separate":
                    status = _refit_device(dev, _dev(new), n)
                elif mode == "in_place":
                    target = _bound_view(dev)
                    target.copy_(_dev(new))
                    status = _refit_device(dev, target, n)
                else:
                    status = _refit_device(dev, _dev(_to_loader(new, order)), n, d_order)
                host.refit_scene(new)
                what = "%s / %s" % (name, mode)
                assert status == 0, what
                _same_derived(dsl.derived_arrays(dev), dsl.derived_arrays(host), what)
                assert np.array_equal(dev.read_nodes(), host.read_nodes()), what
                got_t, got_n = dev.read_scene()
                want_t, want_n = host.read_scene()
                assert np.array_equal(got_t, want_t) and np.array_equal(got_n, want_n), what
                assert np.array_equal(got_t, new.reshape(got_t.shape)), what


@pytest.fixture(scope="module")
def bumpy_built(product, tmp_scene_dir):
    """The bumpy sphere built on the device (dev) and the same arrays uploaded the old way (host)."""
    lt, mats = _load(product, tmp_scene_dir, "dr_pair.obj", *scenes.displaced_sphere(5))
    dev, host = product.Context(0), product.Context(0)
    order, d_order = _device_build(dev, lt, mats)
    tris, nodes = dev.read_scene()
    host.upload_scene(tris, nodes, mats)
    yield dev, host, lt, order, d_order, tris, nodes, mats
    dev.close()
    host.close()


def test_oracle_parity_after_a_device_refit(product, bumpy_built):
    dev, host, _, order, d_order, tris, nodes, _ = bumpy_built
    cap = product.capi
    rays = np.concatenate([scenes.shell_rays(150000, 12.0, seed=301), ol.oracle_camera_rays(256, 256, 1, **CAM)])
    for scale, wobble in ((1.25, 0.6), (0.8, 1.5)):
        new = _deform(tris, scale, wobble)
        assert _refit_device(dev, _dev(_to_loader(new, order)), tris.shape[0], d_order) == 0
        host.refit_scene(new)
        rn = dev.read_nodes()
        assert np.array_equal(rn[:, 32:39], nodes[:, 32:39])                     # topology untouched
        want = ol.oracle_closest(new, rn, rays)
        assert (want["tri"] != MISS).mean() > 0.05
        b = scenes.bounce_rays(rays[:150000], want[:150000], scenes.tri_normals(new, want[:150000]), seed=302)
        want_b = ol.oracle_closest(new, rn, b)
        assert (want_b["t"] < 0).mean() > 0.001                                # negative-t bounce rays included
        occ = ol.oracle_any(new, rn, b) != 0
        for traversal in (0, 1):
            dev.set_option(cap.OPT_TRAVERSAL, traversal)
            _check_hits(dev.trace_closest(rays), want)
            _check_hits(dev.trace_closest(b), want_b)
            assert np.array_equal(dev.trace_any(b) != 0, occ)
        dev.set_option(cap.OPT_TRAVERSAL, 0)
        for mode in (0, 1):                                                    # wavefront, megakernel
            for ctx in (dev, host):
                ctx.set_option(cap.OPT_RENDER_MODE, mode)
            a = _render(dev, 160, 120, (1, 2), 3, **CAM)
            h = _render(host, 160, 120, (1, 2), 3, **CAM)
            assert np.array_equal(a.view(np.uint32), h.view(np.uint32)), "render mode %d" % mode
        for ctx in (dev, host):
            ctx.set_option(cap.OPT_RENDER_MODE, 2)


def _torch_deform(base, scale, wobble):
    """_deform's positions in torch on the device (normals kept): a function of each old position alone."""
    f = base.view(torch.float32).view(-1, 64)
    out = f.clone()
    for v in (0, 20, 40):
        p = f[:, v:v + 3]
        q = p * scale
        q[:, 2] += wobble * torch.sin(p[:, 0] * 0.7)
        out[:, v:v + 3] = q
    return out.view(torch.uint8).view(-1)


def test_animation_loop_on_the_callers_stream(product, tmp_scene_dir):
    """simulate (torch) -> refit -> trace on a side stream, some frames rendered on the context's stream, no host wait
    until the end; every frame equals a second context refitted frame by frame through the host path. A sleep kernel
    enqueued on the side stream just before the call is still running when the call returns."""
    cap = product.capi
    lt, mats = _load(product, tmp_scene_dir, "dr_anim.obj", *scenes.displaced_sphere(5))
    n = lt.shape[0]
    W, H = 160, 120
    rays = scenes.shell_rays(100000, 12.0, seed=311)
    with product.Context(0) as dev, product.Context(0) as host:
        order, d_order = _device_build(dev, lt, mats)
        tris, nodes = dev.read_scene()
        host.upload_scene(tris, nodes, mats)
        for ctx in (dev, host):
            ctx.resize(W, H)
        base = _dev(lt)
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
        status = torch.zeros(8, dtype=torch.int32, device="cuda")
        side = torch.cuda.Stream()
        frames, hits, images, still_running = [], [], {}, None
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for f in range(6):
                d_new = _torch_deform(base, 1.0 + 0.05 * f, 0.3 * f)
                frames.append(d_new)
                if f == 1:
                    torch.cuda._sleep(1 << 30)
                dev.refit_scene_device(d_new.data_ptr(), n, status[f:f + 1].data_ptr(), d_order=d_order.data_ptr(), stream=side.cuda_stream)
                if f == 1:
                    still_running = side.query()
                d_hits = torch.empty((rays.shape[0], 4), dtype=torch.float32, device="cuda")
                dev.trace_closest_device(d_rays.data_ptr(), rays.shape[0], d_hits.data_ptr(), side.cuda_stream)
                hits.append(d_hits)
                if f % 2 == 0:
                    dev.set_option(cap.OPT_RENDER_MODE, f // 2 % 2)           # wavefront, megakernel, wavefront
                    dev.set_frame(1, 3, **CAM)
                    dev.execute(W * H)
                    img = np.zeros((W * H, 4), dtype=np.float32)
                    dev.host_register(img)
                    dev.read_pixels_async(img)
                    images[f] = img
        assert still_running is False, "b2rt_refit_scene_device waited for the caller's stream"
        side.synchronize()
        dev.finish()
        assert status[:6].cpu().tolist() == [0] * 6
        for f in range(6):
            new = frames[f].cpu().numpy().reshape(n, 256)[order]
            host.refit_scene(new)
            got = hits[f].cpu().numpy().view(product.HIT_DTYPE).reshape(-1)
            _check_hits(got, host.trace_closest(rays))
            if f in images:
                host.set_option(cap.OPT_RENDER_MODE, f // 2 % 2)
                want = _render(host, W, H, (1,), 3, **CAM)
                assert np.array_equal(images[f].view(np.uint32), want.view(np.uint32)), "frame %d" % f
                dev.host_unregister(images[f])


@pytest.fixture
def uploaded_bumpy(product, bumpy_ref):
    tris, nodes, mats = bumpy_ref
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        yield ctx, tris


def test_status_bits_and_recovery(product, uploaded_bumpy):
    """Bad data: return code 0, the status bit set; a following refit with valid data restores the hits bit for bit."""
    ctx, tris = uploaded_bumpy
    cap = product.capi
    n = tris.shape[0]
    rays = scenes.shell_rays(100000, 12.0, seed=321)
    before = ctx.trace_closest(rays)
    identity = torch.arange(n, dtype=torch.int32, device="cuda")
    broken = tris.copy()
    broken.view(np.float32).reshape(-1, 64)[0, 0] += np.float32(0.25)        # one copy of a duplicated face moves alone
    nan = tris.copy()
    nan.view(np.float32).reshape(-1, 64)[:, 21] = np.nan                     # v2.x of every triangle: both copies of each pair agree
    one_nan = tris.copy()
    one_nan.view(np.float32).reshape(-1, 64)[77, 41] = np.nan                # a single NaN coordinate
    bad_order = identity.clone()
    bad_order[n // 2] = n
    for data, order, bit in ((broken, None, cap.REFIT_DUPLICATE), (nan, None, cap.REFIT_NONFINITE), (one_nan, None, cap.REFIT_NONFINITE),
                             (tris, bad_order, cap.REFIT_ORDER)):
        status = _refit_device(ctx, _dev(data), n, order)
        assert status & bit, (bit, status)
        ctx.trace_closest(rays)                                                # the scene stays safe to traverse
        assert _refit_device(ctx, _dev(tris), n, identity) == 0
        assert np.array_equal(ctx.trace_closest(rays).view(np.uint32), before.view(np.uint32))


def test_rejected_inputs_leave_the_scene_untouched(product, uploaded_bumpy):
    ctx, tris = uploaded_bumpy
    n = tris.shape[0]
    L, h = ctx._L, ctx._h
    rays = scenes.shell_rays(50000, 12.0, seed=331)
    before = ctx.trace_closest(rays)
    d_new = _dev(_deform(tris, 1.3, 0.5))
    status = torch.full((2,), 12345, dtype=torch.int32, device="cuda")
    order = torch.arange(n, dtype=torch.int32, device="cuda")
    host_tris = np.ascontiguousarray(tris)
    host_order = np.arange(n, dtype=np.uint32)
    bound = _bound_view(ctx)
    s = status.data_ptr()
    vp = C.c_void_p
    cases = [
        ("host triangles", vp(host_tris.ctypes.data), n, None, vp(s), "device memory"),
        ("misaligned triangles", vp(d_new.data_ptr() + 8), n, None, vp(s), "aligned"),
        ("misaligned status", vp(d_new.data_ptr()), n, None, vp(s + 2), "aligned"),
        ("wrong n", vp(d_new.data_ptr()), n - 2, None, vp(s), "triangles given"),
        ("no triangles", None, n, None, vp(s), "null"),
        ("empty", vp(d_new.data_ptr()), 0, None, vp(s), "null"),
        ("null status", vp(d_new.data_ptr()), n, None, None, "status"),
        ("host status", vp(d_new.data_ptr()), n, None, vp(host_order.ctypes.data), "device memory"),
        ("host order", vp(d_new.data_ptr()), n, vp(host_order.ctypes.data), vp(s), "device memory"),
        ("gather in place", vp(bound.data_ptr()), n, vp(order.data_ptr()), vp(s), "gather"),
        ("overlapping the bound buffer", vp(bound.data_ptr() + 256), n, None, vp(s), "overlap"),
    ]
    torch.cuda.synchronize()
    for what, tri_ptr, count, order_ptr, status_ptr, text in cases:
        assert L.b2rt_refit_scene_device(h, tri_ptr, count, order_ptr, status_ptr, None) == INVALID_VALUE, what
        assert text in L.b2rt_last_error(h).decode(), (what, L.b2rt_last_error(h).decode())
        ctx.finish()
        assert status.cpu().tolist() == [12345, 12345], what
        assert np.array_equal(ctx.trace_closest(rays).view(np.uint32), before.view(np.uint32)), what
    assert L.b2rt_refit_scene_device(None, vp(d_new.data_ptr()), n, None, vp(s), None) == -34
    with product.Context(0) as empty:
        assert empty._L.b2rt_refit_scene_device(empty._h, vp(d_new.data_ptr()), n, None, vp(s), None) == INVALID_KERNEL_ARGS
    assert status.cpu().tolist() == [12345, 12345]


def test_device_group_equals_a_single_device(product, tmp_scene_dir):
    if product.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    lt, mats = _load(product, tmp_scene_dir, "dr_group.obj", *scenes.displaced_sphere(5))
    n = lt.shape[0]
    rays = scenes.shell_rays(50000, 12.0, seed=341)
    with product.Context(0) as one, product.Context([0, 1]) as grp:
        order, d_order = _device_build(one, lt, mats)
        order_g, d_order_g = _device_build(grp, lt, mats)
        assert np.array_equal(order, order_g)
        tris, _ = one.read_scene()
        new = _deform(tris, 1.15, 0.7)
        d_new = _dev(_to_loader(new, order))
        assert _refit_device(one, d_new, n, d_order) == 0
        assert _refit_device(grp, d_new, n, d_order_g) == 0
        a = _render(one, 160, 120, (1,), 3, **CAM)
        b = _render(grp, 160, 120, (1,), 3, **CAM)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        _check_hits(grp.trace_closest(rays), one.trace_closest(rays))
        broken = new.copy()
        broken.view(np.float32).reshape(-1, 64)[0, 0] += np.float32(0.25)
        assert _refit_device(grp, _dev(broken), n) & product.capi.REFIT_DUPLICATE
        assert _refit_device(grp, d_new, n, d_order_g) == 0
        _check_hits(grp.trace_closest(rays), one.trace_closest(rays))


def test_cpp_mirror_refits_from_device(product, tmp_scene_dir):
    """CLBVHScene::RefitFromDevice on deformed loader-order data renders the frame the Python Context path renders, bit
    for bit; a broken pair raises HostError with status -50."""
    lt, mats = _load(product, tmp_scene_dir, "dr_mirror.obj", *scenes.displaced_sphere(5))
    n = lt.shape[0]
    d_lt = _dev(lt)
    base = torch.from_numpy(np.ascontiguousarray(lt).reshape(-1)).cuda()
    d_def = _torch_deform(base, 1.2, 0.9)
    torch.cuda.synchronize()
    with product.Context(0) as ctx:
        _, d_order = _device_build(ctx, lt, mats)
        assert _refit_device(ctx, d_def, n, d_order) == 0
        py = _render(ctx, 160, 120, (1,), 3, **CAM)
        py_t, py_n = ctx.read_scene()
    with product.host.Engine(160, 120, device=0) as eng:
        eng.build_scene_device(d_lt.data_ptr(), n, mats)
        eng.refit_scene_device(d_def.data_ptr(), n)
        eng.set_camera(CAM["pos"], CAM["front"], CAM["up"])
        eng.set_render(frame_count=1, bounces=3)
        eng.render_frame()
        assert np.array_equal(eng.pixels()[:, :3].view(np.uint32), py[:, :3].view(np.uint32))
        eng.read_back_scene()
        t2, n2, _ = eng.scene_arrays()
        assert np.array_equal(n2, py_n) and np.array_equal(t2.reshape(py_t.shape), py_t)
        broken = d_def.clone()
        broken.view(torch.float32)[0] += 0.25                                 # loader triangle 0 moves alone: its copy does not
        torch.cuda.synchronize()
        with pytest.raises(product.host.HostError) as e:
            eng.refit_scene_device(broken.data_ptr(), n)
        assert e.value.status == INVALID_ARG_VALUE and "duplicate" in str(e.value)
