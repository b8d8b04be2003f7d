"""-m gpu: traversal on deep trees (tests/deep_trees.py) through the C ABI, bit for bit against the oracle on the same
arrays. The kernels size their stacks from the tree (32, 64, 128 or 256 entries), the tail kernel its frontier
(max(256, 4 (bound + 8)) words) and its records (bound + 8 stack words); the chains here put every one of them on both
sides of each size, and the reference-layout walk, whose stack follows the binary depth, beyond 64 levels."""
import numpy as np
import pytest

import deep_trees as dt
import oracle_lib as ol
import scenes
from test_gpu_parity import _check_hits, _render, _tree_is_valid
from test_gpu_round2 import _counted, _deform, _device_list

pytestmark = pytest.mark.gpu
MISS = 0xFFFFFFFF
W, H = 160, 120


def _chain_camera(depth):
    """Just above the far end of an x chain, looking down along it: every camera ray walks the whole spine."""
    return dict(pos=(depth + 1.5, 0.4, 0.7), front=(-1.0, 0.0, -0.25), up=(0.0, 0.0, 1.0))


GEOMETRIC_CAMERA = dict(pos=(2.0, 2.0, 60.0), front=(0.2, 0.2, -1.0), up=(0.0, 1.0, 0.0))


def _oracle_frame(tris, nodes, mats, cam, frames=(1, 2), bounces=4):
    img = np.zeros((W * H, 4), dtype=np.float32)
    for fc in frames:
        ol.oracle_render(tris, nodes, mats, img, W, H, fc, bounces, **cam)
    return img


def _in_launches(trace, rays, size):
    return np.concatenate([trace(rays[i:i + size]) for i in range(0, rays.shape[0], size)])


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255])
def test_chain_at_every_stack_capacity(product, tmp_scene_dir, depth):
    """Stack bounds 32 | 33, 64 | 65, 128 | 129 and 256, closest and any-hit: the solo walk alone, every ray through the
    tail kernel (16-ray launches under COOP_MAX 16: its frontier above 256 words from bound 57 on), and the two-step tail
    (records of bound + 8 stack words resumed by a second persistent launch)."""
    cap = product.capi
    tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, depth)
    rays = dt.chain_rays(depth + 1, 20000, seed=depth)
    want = ol.oracle_closest(tris, nodes, rays)
    occ = ol.oracle_any(tris, nodes, rays) != 0
    short = rays[:1600]
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        assert ctx.scene_info()["max_depth_binary"] == depth
        try:
            for coop, resume in ((0, 0), (16, 0), (8, 16)):
                ctx.set_option(cap.OPT_COOP_MAX, coop)
                ctx.set_option(cap.OPT_RESUME_MAX, resume)
                got, c = _counted(product, ctx, lambda: ctx.trace_closest(rays))
                _check_hits(got, want)
                assert c["rays"] == rays.shape[0] and c["stack_overflows"] == 0, c
                assert (c["resumed_rays"] > 0) == (resume > coop), c
                assert np.array_equal(ctx.trace_any(rays) != 0, occ)
                # launches of 16 rays: the pool is dry at once, so every ray goes to the tail (or is suspended) at once
                got, c = _counted(product, ctx, lambda: _in_launches(ctx.trace_closest, short, 16))
                _check_hits(got, want[:short.shape[0]])
                assert c["stack_overflows"] == 0 and (c["coop_rays"] > 0) == (coop > 0), c
                assert (c["resumed_rays"] > 0) == (resume > coop), c
                assert np.array_equal(_in_launches(ctx.trace_any, short, 16) != 0, occ[:short.shape[0]])
        finally:
            ctx.set_option(cap.OPT_COOP_MAX, -1)
            ctx.set_option(cap.OPT_RESUME_MAX, 0)


@pytest.mark.parametrize("name", ["chain255", "spine60x4", "geometric"])
def test_deep_frames(product, tmp_scene_dir, name):
    """Frames on the deepest chain, a bushy spine and the loader-built geometric scene: the wavefront (with and without
    the tail kernel) and the megakernel bit-identical, PSNR >= 50 dB against the oracle, and a device group drawing the
    same frame bit for bit."""
    cap = product.capi
    if name == "chain255":
        tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, 255)
        cam = _chain_camera(255)
    elif name == "spine60x4":
        tris, nodes, mats = dt.spine(product.host, tmp_scene_dir, 60, 4, axes=(0, 2))
        cam = _chain_camera(240)
    else:
        tris, nodes, mats, _ = dt.geometric(product.host, tmp_scene_dir)
        cam = GEOMETRIC_CAMERA
    assert (ol.oracle_closest(tris, nodes, ol.oracle_camera_rays(W, H, 1, **cam))["tri"] != MISS).mean() > 0.05    # the camera sees the scene
    want = _oracle_frame(tris, nodes, mats, cam)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        imgs = []
        for mode, coop in ((0, 0), (0, 8), (1, -1)):
            ctx.set_option(cap.OPT_RENDER_MODE, mode)
            ctx.set_option(cap.OPT_COOP_MAX, coop)
            imgs.append(_render(ctx, W, H, (1, 2), 4, **cam))
        for img in imgs[1:]:
            assert np.array_equal(img.view(np.uint32), imgs[0].view(np.uint32))
        assert scenes.psnr(imgs[0][:, :3], want[:, :3]) >= 50.0
    with product.Context(_device_list(product, 2)) as grp:
        grp.upload_scene(tris, nodes, mats)
        for mode in (0, 1):
            grp.set_option(cap.OPT_RENDER_MODE, mode)
            img = _render(grp, W, H, (1, 2), 4, **cam)
            assert np.array_equal(img.view(np.uint32), imgs[0].view(np.uint32)), mode


@pytest.mark.parametrize("name", ["chain64", "chain65", "chain100", "chain255", "geometric"])
def test_reference_layout_walk_on_deep_trees(product, tmp_scene_dir, name):
    """B2RT_OPT_TRAVERSAL=1 walks the reference's own arrays with a stack of one entry per binary level. The reference's
    int[64] would lose the far subtrees of rays that go more than 64 levels deep: on the chains from 65 levels on, those
    rays and frames only match the oracle if nothing is dropped."""
    cap = product.capi
    if name == "geometric":
        tris, nodes, mats, p = dt.geometric(product.host, tmp_scene_dir)
        rays, cam = dt.geometric_rays(p, 20000, seed=11), GEOMETRIC_CAMERA
    else:
        depth = int(name[5:])
        tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, depth)
        rays, cam = dt.chain_rays(depth + 1, 20000, seed=depth + 1), _chain_camera(depth)
    want = ol.oracle_closest(tris, nodes, rays)
    occ = ol.oracle_any(tris, nodes, rays) != 0
    ref_img = _oracle_frame(tris, nodes, mats, cam)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        ctx.set_option(cap.OPT_TRAVERSAL, 1)
        ctx.reset_counters()
        _check_hits(ctx.trace_closest(rays), want)
        assert np.array_equal(ctx.trace_any(rays) != 0, occ)
        assert scenes.psnr(_render(ctx, W, H, (1, 2), 4, **cam)[:, :3], ref_img[:, :3]) >= 50.0
        assert ctx.counters()["stack_overflows"] == 0


def test_too_deep_tree_is_refused_and_the_context_stays_usable(product, tmp_scene_dir):
    """Stack bound 257 is beyond the largest kernels: refused with CL_OUT_OF_RESOURCES when the scene is first used, and on
    every later use while it stays bound. The same context then takes a valid scene and traces it correctly."""
    deep = dt.chain(product.host, tmp_scene_dir, 256)
    tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, 255)
    rays = dt.chain_rays(256, 20000, seed=257)
    want = ol.oracle_closest(tris, nodes, rays)
    with product.Context(0) as ctx:
        for attempt in (lambda: ctx.upload_scene(*deep), lambda: ctx.trace_closest(rays)):
            with pytest.raises(product.B2RTError) as e:
                attempt()
            assert e.value.status == -5 and "too deep" in str(e.value)       # CL_OUT_OF_RESOURCES
        ctx.upload_scene(tris, nodes, mats)
        _check_hits(ctx.trace_closest(rays), want)
        assert np.array_equal(ctx.trace_any(rays) != 0, ol.oracle_any(tris, nodes, rays) != 0)


def test_refit_of_a_deep_chain(product, tmp_scene_dir):
    """b2rt_refit_scene on a 200-level chain: deformations that keep the loader's pairs, then hits of the wide walk and of
    the reference-layout walk against the oracle on the refitted nodes read back from the device."""
    cap = product.capi
    tris, nodes, mats = dt.chain(product.host, tmp_scene_dir, 200, axes=(0, 1, 2))
    rays = dt.chain_rays(201, 20000, seed=201)
    with product.Context(0) as ctx:
        ctx.upload_scene(tris, nodes, mats)
        for scale, wobble in ((1.2, 0.8), (0.9, 0.05)):
            new = _deform(tris, scale, wobble)
            ctx.refit_scene(new)
            rn = ctx.read_nodes()
            assert np.array_equal(rn[:, 32:39], nodes[:, 32:39])                # topology untouched
            _tree_is_valid(new, rn)                                            # boxes: exact unions again
            want = ol.oracle_closest(new, rn, rays)
            assert (want["tri"] != MISS).mean() > 0.05
            occ = ol.oracle_any(new, rn, rays) != 0
            for traversal in (0, 1):
                ctx.set_option(cap.OPT_TRAVERSAL, traversal)
                _check_hits(ctx.trace_closest(rays), want)
                assert np.array_equal(ctx.trace_any(rays) != 0, occ)
            ctx.set_option(cap.OPT_TRAVERSAL, 0)
