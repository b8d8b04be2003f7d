"""CPU checks of the k-nearest-hits query (b2rt_trace_multi, include/b2rt.h): the oracle's k-list walk
(tests/multi_hit/oracle_multi.c) against the oracle's closest-hit walk and against brute-force Moller-Trumbore, and the
product's HIT_MULTI traversal policy (csrc/traverse.cuh, host emulation in tests/multi_hit/emu_multi.cpp) against the
oracle under random node / leaf interleavings."""
import os

import numpy as np
import pytest

import deep_trees as dt
import multi_hit_lib as ml
import oracle_lib as ol
import scenes
from conftest import _reference_scene, load_product

MISS = 0xFFFFFFFF
KS = (1, 2, 3, 8, 64)


def _bits(h):
    """(rows..., 4) uint32 view of HIT records: t, u, v, tri bit for bit."""
    return np.stack([h["t"].view(np.uint32), h["u"].view(np.uint32), h["v"].view(np.uint32), h["tri"]], -1)


def _same_rows(a, b):
    assert a.shape == b.shape
    bad = np.nonzero((_bits(a) != _bits(b)).any(-1).any(-1))[0]
    assert bad.size == 0, "%d rows differ, first %d: %s vs %s" % (bad.size, bad[0], a[bad[0]], b[bad[0]])


def _check_rows(tris, rays, hits, sample=400):
    """Rows sorted by t, padded exactly, each triangle at most once; every listed hit of a sample of rays is accepted by
    brute-force RayTriangle with the same fp32 t, u, v."""
    n, k = hits.shape
    used = hits["tri"] != MISS
    assert not (~used[:, :-1] & used[:, 1:]).any()                               # padding only at the end of a row
    pad = ~used
    tmax = np.broadcast_to(rays["tmax"][:, None], hits.shape)
    assert np.array_equal(hits["t"][pad].view(np.uint32), tmax[pad].view(np.uint32))
    assert not hits["u"][pad].view(np.uint32).any() and not hits["v"][pad].view(np.uint32).any()
    t = np.where(used, hits["t"], np.inf)
    with np.errstate(invalid="ignore"):                                           # inf - inf between padded slots
        assert (np.diff(t, axis=1)[used[:, 1:]] >= 0).all()                      # sorted
    assert (t[used] < tmax[used]).all()
    srt = np.sort(np.where(used, hits["tri"].astype(np.int64), -np.arange(1, k + 1)), axis=1)
    assert not (np.diff(srt, axis=1) == 0).any()                                 # no triangle twice
    sub = np.nonzero(used[:, 0])[0]
    sub = sub[np.linspace(0, sub.size - 1, min(sample, sub.size)).astype(np.int64)] if sub.size else sub
    ok, t_all = scenes.moller_trumbore_all(tris, rays[sub])
    for r, i in enumerate(sub):
        m = used[i]
        tri = hits["tri"][i][m].astype(np.int64)
        assert ok[r, tri].all()
        assert np.array_equal(t_all[r, tri].view(np.uint32), hits["t"][i][m].view(np.uint32))


def _scene(tmp_scene_dir, name, p, n, f):
    return _reference_scene(scenes.write_obj(os.path.join(tmp_scene_dir, name), p, n, f))


def _fuzz(tmp_scene_dir, cases=8):
    """(tris, nodes, rays) of small awkward scenes (scenes.fuzz_scene), rays from around, on and inside the geometry."""
    host = load_product().host
    rng = np.random.default_rng(77)
    for case in range(cases):
        pos, faces = scenes.fuzz_scene(case, rng)
        nrm = np.tile(np.array([[0.0, 0.0, 1.0]], dtype=np.float32), (pos.shape[0], 1))
        path = scenes.write_obj(os.path.join(tmp_scene_dir, "mfuzz%d.obj" % case), pos, nrm, faces)
        tris, nodes, _ = host.load_scene(path, int(rng.choice([1, 2, 4, 8])))
        lo, hi = pos.min(0) - 1.0, pos.max(0) + 1.0
        rays = np.concatenate([scenes.box_rays(800, lo, hi, seed=case), scenes.axis_rays(lo, hi, 12, seed=case),
                               scenes.pack_rays(pos[rng.integers(0, pos.shape[0], 200)], rng.normal(size=(200, 3)))])
        rays["tmax"][::5] = rng.uniform(0.1, 20.0, size=rays["tmax"][::5].shape).astype(np.float32)
        yield tris, nodes, rays


def _bumpy_rays(tris, nodes):
    """Shell rays, their bounce rays (origins just off the surface: many hits at negative t) and rays from inside."""
    rays = scenes.shell_rays(6000, 10.0, seed=141)
    h = ol.oracle_closest(tris, nodes, rays)
    b = scenes.bounce_rays(rays, h, scenes.tri_normals(tris, h), seed=142)
    short = b[:1500].copy()
    short["tmax"] = 3.0
    return np.concatenate([rays, b, short, scenes.box_rays(3000, (-9, -9, -9), (9, 9, 9), seed=143)])


def test_k1_equals_closest(cornell_ref, tmp_scene_dir):
    """k = 1 is the closest-hit query, misses included, bit for bit."""
    tris, nodes, _ = cornell_ref
    g = np.load(os.path.join(scenes.GOLDEN, "cornell_hits.npz"))
    rays = np.ascontiguousarray(g["rays"]).view(ol.RAY).reshape(-1)
    cases = [(tris, nodes, rays)]
    t2, n2, _ = _scene(tmp_scene_dir, "mties.obj", *scenes.tie_grid(24, layers=3))
    cases.append((t2, n2, scenes.tie_rays(24)))
    cases += list(_fuzz(tmp_scene_dir, 6))
    for tr, nd, ry in cases:
        _same_rows(ml.oracle_trace_multi(tr, nd, ry, 1), ol.oracle_closest(tr, nd, ry)[:, None])


def test_cornell_rows_are_real_hits_with_loader_copies(cornell_ref):
    """Every listed hit is a real RayTriangle hit; the loader's two copies of a face appear as a pair at the same t."""
    tris, nodes, _ = cornell_ref
    g = np.load(os.path.join(scenes.GOLDEN, "cornell_hits.npz"))
    rays = np.ascontiguousarray(g["rays"]).view(ol.RAY).reshape(-1)
    for k in KS:
        h = ml.oracle_trace_multi(tris, nodes, rays, k)
        _check_rows(tris, rays, h)
        if k >= 2:
            pair = (h["tri"][:, 1] != MISS) & (h["t"][:, 0].view(np.uint32) == h["t"][:, 1].view(np.uint32))
            assert pair.mean() > 0.3
            # the list is a prefix of every longer list
            for kk in KS:
                if kk > k:
                    _same_rows(h, ml.oracle_trace_multi(tris, nodes, rays, kk)[:, :k])
                    break


def test_bumpy_rows_with_negative_t(bumpy_ref):
    tris, nodes, _ = bumpy_ref
    rays = _bumpy_rays(tris, nodes)
    for k in (2, 8):
        h = ml.oracle_trace_multi(tris, nodes, rays, k)
        _check_rows(tris, rays, h, sample=60)
        assert ((h["tri"] != MISS) & (h["t"] < 0)).any(-1).mean() > 0.005          # rows with negative t occur


def _emu_matches_oracle(tris, nodes, rays, ks=KS, schedules=(0, 7, 12345)):
    st = ml.emu_build(tris, nodes)
    for k in ks:
        want = ml.oracle_trace_multi(tris, nodes, rays, k)
        for schedule in schedules:
            s = ol.EmuStats()
            _same_rows(ml.emu_trace_multi(rays, k, schedule=schedule, stats=s), want)
            assert s.overflow == 0 and s.max_stack <= st.stack_bound
    assert ml.emu_culling_violations() == 0
    return st


def test_emu_icosphere_and_bumpy(bumpy_ref, tmp_scene_dir):
    tris, nodes, _ = _scene(tmp_scene_dir, "mico.obj", *_icosphere(3))
    _emu_matches_oracle(tris, nodes, np.concatenate([scenes.shell_rays(3000, 3.0, seed=151),
                                                     scenes.box_rays(2000, (-1.5,) * 3, (1.5,) * 3, seed=152)]))
    tris, nodes, _ = bumpy_ref
    rays = _bumpy_rays(tris, nodes)[::3]
    _emu_matches_oracle(tris, nodes, rays)
    h = ml.emu_trace_multi(rays, 8, schedule=3)
    assert ((h["tri"] != MISS) & (h["t"] < 0)).any(-1).any()


def _icosphere(subdiv):
    p, f = scenes.icosphere(subdiv)
    return p.astype(np.float32), (p / np.linalg.norm(p, axis=1, keepdims=True)).astype(np.float32), f


def test_emu_ties_across_leaves(tmp_scene_dir):
    """Coincident lattices: equal-t candidates in different leaves keep the reference's visiting order in the list."""
    tris, nodes, _ = _scene(tmp_scene_dir, "mties2.obj", *scenes.tie_grid(24, layers=3))
    rays = scenes.tie_rays(24)
    st = _emu_matches_oracle(tris, nodes, rays)
    h = ml.oracle_trace_multi(tris, nodes, rays, 8)
    ties = (h["tri"][:, 1:] != MISS) & (h["t"][:, 1:].view(np.uint32) == h["t"][:, :-1].view(np.uint32))
    assert ties.any(-1).mean() > 0.5 and st.n_leaf_blocks > 1


def test_emu_fuzz(tmp_scene_dir):
    for tris, nodes, rays in _fuzz(tmp_scene_dir):
        _emu_matches_oracle(tris, nodes, rays, schedules=(0, 99))


@pytest.mark.parametrize("depth", [31, 64, 127, 255])
def test_emu_deep_chains(tmp_scene_dir, depth):
    tris, nodes, _ = dt.chain(load_product().host, tmp_scene_dir, depth)
    rays = dt.chain_rays(depth + 1, 1500, seed=depth)
    st = _emu_matches_oracle(tris, nodes, rays, ks=(1, 3, 64), schedules=(0, 5))
    assert st.stack_bound == depth + 1
