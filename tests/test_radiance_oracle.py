"""The radiance checker (tests/radiance/oracle_radiance.c) against the oracle's own path loop, the record layout against the
header, and the entry points without a GPU. No GPU needed."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_lib as ol
import radiance_lib as rl
import scenes


def cornell_rays(tris, nodes):
    """Camera rays, their diffuse bounce rays (origins just off the surface) and rays from inside the box."""
    cam = ol.oracle_camera_rays(24, 24, 3)
    h = ol.oracle_closest(tris, nodes, cam)
    bounce = scenes.bounce_rays(cam, h, scenes.tri_normals(tris, h), seed=501)
    inside = scenes.box_rays(400, (-4, -4, 1), (4, 4, 9), seed=502)
    return {"camera": cam, "bounce": bounce, "inside": inside}


def seeds_for(n, seed):
    return np.random.default_rng(seed).integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)


@pytest.mark.parametrize("light_type", [0, 1, 2])
def test_loop_equals_render_path_at_full_range(cornell_ref, light_type):
    tris, nodes, mats = cornell_ref
    for name, rays in cornell_rays(tris, nodes).items():
        seeds = seeds_for(rays.shape[0], 503 + light_type)
        for bounces in (0, 1, 4):
            for sky in (1.0, 0.25):
                got = rl.oracle_radiance(tris, nodes, mats, rays, seeds, bounces, light_type, sky)
                rl.same(got, rl.oracle_render_path(tris, nodes, mats, rays, seeds, bounces, light_type, sky))
                if bounces == 0:
                    assert (got["r"] == 0).all() and (got["seed"] == seeds).all(), name
                else:
                    assert (got["seed"] != seeds).any(), name       # the paths consumed random numbers


def test_short_tmax_takes_the_sky(cornell_ref):
    tris, nodes, mats = cornell_ref
    rays = cornell_rays(tris, nodes)["camera"]
    h = ol.oracle_closest(tris, nodes, rays)
    keep = (h["tri"] != 0xFFFFFFFF) & (h["t"] > 1.0)
    rays, h = rays[keep].copy(), h[keep]
    assert rays.shape[0] > 300
    rays["tmax"] = h["t"] * np.float32(0.5)                          # every first hit lies beyond tmax
    seeds = seeds_for(rays.shape[0], 504)
    got = rl.oracle_radiance(tris, nodes, mats, rays, seeds, 4, 1, 0.75)
    sky = np.float32(0.5) * np.float32(0.75)
    assert (got["r"] == sky).all() and (got["g"] == sky).all() and (got["b"] == sky).all()
    assert (got["seed"] == seeds).all()                             # a miss draws no random number
    # a tmax past the first hit gives the full-range path
    rays["tmax"] = h["t"] * np.float32(2.0)
    full = rays.copy()
    full["tmax"] = 100000.0
    rl.same(rl.oracle_radiance(tris, nodes, mats, rays, seeds, 4, 1, 0.75), rl.oracle_render_path(tris, nodes, mats, full, seeds, 4, 1, 0.75))


def test_record_layout_matches_the_header(product):
    text = open(os.path.join(ol.ROOT, "include", "b2rt.h")).read()
    m = re.search(r"typedef struct \{ float r, g, b; uint32_t seed; \} b2rt_radiance;", text)
    assert m, "b2rt_radiance is {float r, g, b; uint32_t seed}"
    dt = product.layouts.RADIANCE_DTYPE
    assert dt.itemsize == 16 and dt.names == ("r", "g", "b", "seed")
    assert [dt.fields[n][1] for n in dt.names] == [0, 4, 8, 12] and dt["seed"] == np.dtype("<u4")
    assert dt == rl.RADIANCE


def test_entries_fail_without_a_gpu(product):
    if product.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = product.capi.lib()
    h = C.c_void_p()
    assert L.b2rt_create(0, C.byref(h)) == -1                       # B2RT_DEVICE_NOT_FOUND: no handle, so no entry is reachable
    with pytest.raises(product.capi.B2RTError) as e:
        product.Context(0)
    assert e.value.status == -1
    rays = np.zeros(4, dtype=product.layouts.RAY_DTYPE)
    out = np.zeros(4, dtype=product.layouts.RADIANCE_DTYPE)
    assert L.b2rt_trace_radiance(None, rays.ctypes.data, rays.ctypes.data, 4, out.ctypes.data) == -34
    assert L.b2rt_trace_radiance_device(None, None, None, 0, None, None) == -34
