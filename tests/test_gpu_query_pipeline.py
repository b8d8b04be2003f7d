"""-m gpu: the host-buffer entries (b2rt_trace_closest / _any / _multi, b2rt_closest_point) run their items through a
chunked copy-in / launch / copy-out pipeline on two staging slots. Over many chunks (slots reused, the ramp down, the chunk
shrinking with k) every kind must return what its device entry returns over the whole array in one launch, bit for bit;
the chunk schedule itself is pinned through the launch count; a device group must equal one device, empty ranges
included."""
import numpy as np
import pytest

import point_query_lib as pq
import scenes
from test_gpu_round2 import _device_list

pytestmark = pytest.mark.gpu
SMALL = 9 * 1024 + 37           # ten chunks of B2RT_STREAM_CHUNK = 1024, the last one short
FULL = 3 * (1 << 20) + 37       # ramp up, ramp down (halving) and a short last chunk at the default chunk
RAMP = 1 << 19                  # first chunk of the ramp
STREAM_CHUNK = 1 << 22          # default items per chunk


def _chunk_sizes(n, stream_chunk=STREAM_CHUNK, k=0):
    """The host pipeline's chunk schedule, restated: the chunk shrinks with k > 1 (floor 1024), sizes ramp up from
    min(chunk, 2^19) by doubling and, while more than one ramp is left, never take more than half of what is left (rounded
    up to 32)."""
    cap = max(stream_chunk // k, 1024) if k > 1 else stream_chunk
    chunk = min(n, cap)
    ramp = min(chunk, RAMP)
    sizes, off, c = [], 0, 0
    while off < n:
        left = n - off
        m = min(chunk, ramp << min(c, 16))
        if left <= ramp:
            m = left
        else:
            m = min(m, max(ramp, (left // 2 + 31) & ~31))
        sizes.append(m)
        off += m
        c += 1
    return sizes


def _queries(tris, n, seed):
    p = tris.view(np.float32).reshape(-1, 64)[:, 0:3]
    lo, hi = p.min(0), p.max(0)
    rng = np.random.default_rng(seed)
    return pq.queries(rng.uniform(lo - 0.2 * (hi - lo), hi + 0.2 * (hi - lo), (n, 3)))


def _on_device(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda()


def _device_results(ctx, rays, q, ks):
    """Every kind through its device entry, once over the whole array: {kind: bytes}."""
    import torch
    n = rays.shape[0]
    d_rays = _on_device(torch, rays)
    out = {}
    for name, size, call in (
            ("closest", n * 16, lambda d: ctx.trace_closest_device(d_rays.data_ptr(), n, d.data_ptr())),
            ("any", n * 4, lambda d: ctx.trace_any_device(d_rays.data_ptr(), n, d.data_ptr()))):
        d = torch.full((size,), 0xA5, dtype=torch.uint8, device="cuda")
        call(d)
        ctx.finish()
        out[name] = d.cpu().numpy()
    for k in ks:
        d = torch.full((n * k * 16,), 0xA5, dtype=torch.uint8, device="cuda")
        ctx.trace_multi_device(d_rays.data_ptr(), n, k, d.data_ptr())
        ctx.finish()
        out["multi", k] = d.cpu().numpy()
    if q is not None:
        d_q = _on_device(torch, q)
        d = torch.full((q.shape[0] * 16,), 0xA5, dtype=torch.uint8, device="cuda")
        ctx.closest_point_device(d_q.data_ptr(), q.shape[0], d.data_ptr())
        ctx.finish()
        out["point"] = d.cpu().numpy()
    return out


def _host_results(ctx, rays, q, ks):
    out = {"closest": ctx.trace_closest(rays), "any": ctx.trace_any(rays)}
    for k in ks:
        out["multi", k] = ctx.trace_multi(rays, k)
    if q is not None:
        out["point"] = ctx.closest_point(q)
    return {key: np.ascontiguousarray(v).view(np.uint8).reshape(-1) for key, v in out.items()}


def _same(got, want):
    assert got.keys() == want.keys()
    for key in want:
        assert np.array_equal(got[key], want[key]), key


def test_small_chunks_every_kind(product, bumpy_ref, monkeypatch):
    """B2RT_STREAM_CHUNK = 1024: ten chunks per call, so both staging slots are reused four times; k = 64 keeps the 1024
    floor. The reference-layout walk (OPT_TRAVERSAL = 1) goes through the same pipeline."""
    monkeypatch.setenv("B2RT_STREAM_CHUNK", "1024")
    assert len(_chunk_sizes(SMALL, 1024)) == 10
    tris, nodes, mats = bumpy_ref
    rays = scenes.shell_rays(SMALL, 10.0, seed=801)
    q = _queries(tris, SMALL, seed=802)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        want = _device_results(ctx, rays, q, (1, 3, 64))
        _same(_host_results(ctx, rays, q, (1, 3, 64)), want)
        ctx.set_option(product.capi.OPT_TRAVERSAL, 1)
        binary = _device_results(ctx, rays, q, (3,))
        _same(_host_results(ctx, rays, q, (3,)), binary)


def test_full_ramp(product, bumpy_ref):
    """The default chunk over 3 * 2^20 + 37 items: ramp up (2^19, 2^20), ramp down (half of what is left) and a short last
    chunk, for closest-point queries and for k = 4 hits per ray (the chunk shrinks to 2^20 rays)."""
    sizes = _chunk_sizes(FULL)
    assert sizes[:2] == [RAMP, 2 * RAMP] and sizes[2] < sizes[1] and sizes[-1] < RAMP
    assert _chunk_sizes(FULL, k=4) == [RAMP, 2 * RAMP, sizes[2], sizes[3], sizes[4]]
    tris, nodes, mats = bumpy_ref
    rays = scenes.shell_rays(FULL, 10.0, seed=803)
    q = _queries(tris, FULL, seed=804)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        import torch
        d_q = _on_device(torch, q)
        d = torch.empty((FULL * 16,), dtype=torch.uint8, device="cuda")
        ctx.closest_point_device(d_q.data_ptr(), FULL, d.data_ptr())
        ctx.finish()
        assert np.array_equal(ctx.closest_point(q).view(np.uint8), d.cpu().numpy())
        del d_q, d
        d_rays = _on_device(torch, rays)
        d = torch.empty((FULL * 4 * 16,), dtype=torch.uint8, device="cuda")
        ctx.trace_multi_device(d_rays.data_ptr(), FULL, 4, d.data_ptr())
        ctx.finish()
        assert np.array_equal(ctx.trace_multi(rays, 4).view(np.uint8).reshape(-1), d.cpu().numpy())


@pytest.mark.parametrize("stream_chunk", [None, "1024", "5000"])
def test_chunk_schedule(product, bumpy_ref, monkeypatch, stream_chunk):
    """Without the cooperative tail every chunk is one launch, so the launch count of a host call is its number of chunks."""
    if stream_chunk is not None:
        monkeypatch.setenv("B2RT_STREAM_CHUNK", stream_chunk)
    else:
        monkeypatch.delenv("B2RT_STREAM_CHUNK", raising=False)
    chunk = int(stream_chunk) if stream_chunk else STREAM_CHUNK
    n, ks = (FULL, (4,)) if stream_chunk is None else (SMALL, (3, 64))
    tris, nodes, mats = bumpy_ref
    rays = scenes.shell_rays(n, 10.0, seed=805)
    q = _queries(tris, n, seed=806)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        ctx.set_option(product.capi.OPT_COOP_MAX, 0)
        calls = [("closest", 0, lambda: ctx.trace_closest(rays)), ("any", 0, lambda: ctx.trace_any(rays)),
                 ("point", 0, lambda: ctx.closest_point(q))]
        calls += [("multi", k, lambda k=k: ctx.trace_multi(rays, k)) for k in ks]
        for what, k, call in calls:
            before = ctx.launch_count()
            call()
            assert ctx.launch_count() - before == len(_chunk_sizes(n, chunk, k)), (what, k)


@pytest.mark.parametrize("n", [1, 2 * 1024 + 1])
def test_device_group_equals_one_device(product, bumpy_ref, monkeypatch, n):
    """Two members split [0, n) into [0, n/2) and [n/2, n): with n = 1 the first range is empty; with 2049 items and
    1024-item chunks the second member runs two chunks."""
    monkeypatch.setenv("B2RT_STREAM_CHUNK", "1024")
    tris, nodes, mats = bumpy_ref
    rays = scenes.shell_rays(n, 10.0, seed=807)
    q = _queries(tris, n, seed=808)
    with product.Context(0) as one:
        one.upload_scene(tris, nodes, mats)
        want = _host_results(one, rays, q, (1, 3))
    with product.Context(_device_list(product, 2)) as grp:
        assert grp.group_size() == 2
        grp.upload_scene(tris, nodes, mats)
        _same(_host_results(grp, rays, q, (1, 3)), want)
