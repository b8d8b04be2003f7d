"""CPU checks of the product's traversal logic (tests/emu, see test_emu_traversal.py) on deep trees (tests/deep_trees.py):
chains whose stack bound lies on either side of every stack capacity the kernels are built for (32, 64, 128, 256
entries), spines with bushy side trees, and a deep tree from the loader and SAH builder. Every walk must reproduce the
oracle bit for bit, and the rays that run down a whole chain must really fill the stack to its bound."""
import numpy as np
import pytest

import deep_trees as dt
import oracle_lib as ol
from conftest import load_product
from test_emu_traversal import _same
from test_gpu_parity import _tree_is_valid

MISS = 0xFFFFFFFF
B2_COOP_NODES = 8                                               # csrc/coop.cuh


def _kernel_frontier(bound):
    """(fcap, wide_limit) of the tail kernel for a tree of this stack bound, as launch_trace_wide (csrc/kernels.cu) sets them."""
    fcap = max(256, 4 * (bound + 8))
    return fcap, fcap - (bound + 8) - (7 * B2_COOP_NODES + 4)


def _check_walks(tris, nodes, rays):
    """Every emulated walk against the oracle: the solo walk under two schedules, the kernels' split between shared and
    local stack, and the cooperative tail with the kernels' own frontier geometry for this tree, after hand-overs at any
    point of the walk (also deep in it) and the two-step tail's resume. Returns the tree's EmuStats."""
    st = ol.emu_build(tris, nodes)
    want = ol.oracle_closest(tris, nodes, rays)
    occ = ol.oracle_any(tris, nodes, rays) != 0
    assert 0.05 < (want["tri"] != MISS).mean() < 0.99
    for schedule in (0, 13):
        s = ol.EmuStats()
        _same(ol.emu_trace(rays, stats=s, schedule=schedule), want)
        assert s.overflow == 0 and s.max_stack <= st.stack_bound
        assert np.array_equal(ol.emu_trace(rays, any_hit=True, schedule=schedule) != 0, occ)
    for schedule in (0, 5):
        _same(ol.emu_trace_hybrid(rays, depth=12, schedule=schedule), want)
    assert np.array_equal(ol.emu_trace_hybrid(rays, any_hit=True, depth=12) != 0, occ)
    fcap, wide_limit = _kernel_frontier(st.stack_bound)
    for handoff, resume in ((0, 0), (9, 0), (60, 0), (400, 0), (5, 7), (30, 40), (400, 400)):
        s = ol.EmuStats()
        _same(ol.emu_trace_coop(rays, stats=s, handoff=handoff, wide_limit=wide_limit, fcap=fcap, resume=resume), want)
        assert s.overflow == 0, (handoff, resume)
    for handoff, resume in ((0, 0), (400, 400)):
        got = ol.emu_trace_coop(rays, any_hit=True, handoff=handoff, wide_limit=wide_limit, fcap=fcap, resume=resume)
        assert np.array_equal(got != 0, occ)
    assert ol.emu_culling_violations() == 0
    return st


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255, 256])
def test_chain_depth_and_stack_bound(tmp_scene_dir, depth):
    """The chains of the GPU tests: binary depth D and stack bound exactly D + 1, i.e. on both sides of each capacity."""
    tris, nodes, _ = dt.chain(load_product().host, tmp_scene_dir, depth)
    _tree_is_valid(tris, nodes)
    st = ol.emu_build(tris, nodes)
    assert (st.max_depth_binary, st.stack_bound) == (depth, depth + 1)


@pytest.mark.parametrize("depth, axes, direction", [(31, (0,), 1), (64, (2, 0), 1), (65, (0,), -1), (128, (0, 1, 2), 1),
                                                    (200, (1, 0), -1), (255, (0,), 1), (255, (2, 1, 0), -1)])
def test_chain_walks(tmp_scene_dir, depth, axes, direction):
    """Chains with split axes that do and do not follow the chain: rays that run down the whole chain from either end,
    rays from all around it, short rays. The rays from the far end push one entry per level."""
    tris, nodes, _ = dt.chain(load_product().host, tmp_scene_dir, depth, axes, direction)
    _tree_is_valid(tris, nodes)
    st = _check_walks(tris, nodes, dt.chain_rays(depth + 1, 3000, seed=depth, direction=direction))
    grazing = np.concatenate([dt.grazing_rays(depth + 1, 1000, seed=7, direction=direction),
                              dt.grazing_rays(depth + 1, 1000, seed=8, direction=direction, y_jitter=0.003)])
    s = ol.EmuStats()
    ol.emu_trace(grazing, stats=s)
    assert s.overflow == 0 and s.max_stack >= st.stack_bound - 1         # the deepest entries are used


@pytest.mark.parametrize("depth, side, bound", [(60, 4, 67), (30, 8, 42)])
def test_bushy_spine_walks(tmp_scene_dir, depth, side, bound):
    """A balanced subtree of `side` leaves at every level of the spine: long and wide frontiers at once."""
    tris, nodes, _ = dt.spine(load_product().host, tmp_scene_dir, depth, side, axes=(0, 2))
    _tree_is_valid(tris, nodes)
    st = _check_walks(tris, nodes, dt.chain_rays(depth * side + 1, 3000, seed=side))
    assert st.max_depth_binary == depth + int(np.log2(side)) and st.stack_bound == bound


def test_loader_built_geometric_scene(tmp_scene_dir):
    """An ordinary OBJ through the loader and the SAH builder that gives a deep tree: 600 faces in geometric progression
    select the 256-entry kernels. The preconditions are asserted so that a builder change cannot make it shallow unnoticed."""
    tris, nodes, _, p = dt.geometric(load_product().host, tmp_scene_dir)
    _tree_is_valid(tris, nodes)
    st = _check_walks(tris, nodes, dt.geometric_rays(p, 3000, seed=5))
    assert st.max_depth_binary >= 65 and 128 < st.stack_bound <= 256
