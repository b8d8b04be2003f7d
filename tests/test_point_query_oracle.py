"""CPU checks of the closest-point query (b2rt_closest_point, include/b2rt.h): the brute-force oracle
(tests/point_query/oracle_point.c) against a float64 evaluation of the exact distance, the product's distance routine and
wide-BVH walk (csrc/point_query.cuh, host emulation in tests/point_query/emu_point.cpp) against the oracle bit for bit,
the culling lemma lb <= d2 checked directly, and the SASS of the lb and d2 sequences (no contraction)."""
import collections
import importlib.util
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import deep_trees as dt
import point_query_lib as pq
import scenes
from conftest import ROOT, _reference_scene, load_product

MISS = 0xFFFFFFFF


def bits(h):
    """(n, 4) uint32 view of point-hit records: d2, u, v, tri bit for bit."""
    return np.stack([h["d2"].view(np.uint32), h["u"].view(np.uint32), h["v"].view(np.uint32), h["tri"]], -1)


def same(a, b):
    assert a.shape == b.shape
    bad = np.nonzero((bits(a) != bits(b)).any(-1))[0]
    assert bad.size == 0, "%d records differ, first %d: %s vs %s" % (bad.size, bad[0], a[bad[0]], b[bad[0]])


def positions(tris):
    """(n, 3, 3) float32 vertex positions of CLTriangle records."""
    f = tris.view(np.float32).reshape(-1, 64)
    return np.stack([f[:, 0:3], f[:, 20:23], f[:, 40:43]], 1)


def query_sets(p, seed, far=True):
    """Points near the surface, exactly on vertices, on edges and on faces, uniform in the box, and far away, with a mix of
    max_d2 values (tight, +inf, 0, negative, NaN)."""
    rng = np.random.default_rng(seed)
    lo, hi = p.reshape(-1, 3).min(0), p.reshape(-1, 3).max(0)
    ext = float(np.max(hi - lo)) + 1e-3
    k = rng.integers(0, p.shape[0], 600)
    w = rng.dirichlet((1.0, 1.0, 1.0), 600)
    face = np.einsum("nk,nkd->nd", w, p[k].astype(np.float64))
    t = rng.random((600, 1))
    edge = p[k, 0] * (1 - t) + p[k, 1] * t
    pts = [p[k[:300], rng.integers(0, 3, 300)].astype(np.float64),                 # exactly on vertices
           edge, face, face + rng.normal(0, 0.01 * ext, face.shape),               # on edges, on faces, near the surface
           rng.uniform(lo - 0.2 * ext, hi + 0.2 * ext, (1500, 3))]                 # anywhere in and around the box
    if far:
        d = rng.normal(size=(200, 3))
        pts.append((lo + hi) / 2 + d / np.linalg.norm(d, axis=1, keepdims=True) * 8 * ext)
    pts = np.concatenate(pts).astype(np.float32)
    q = pq.queries(pts, np.inf)
    n = q.shape[0]
    q["max_d2"][::5] = (0.02 * ext) ** 2                                            # tight radius
    q["max_d2"][1::11] = rng.uniform(0, (0.3 * ext) ** 2, q["max_d2"][1::11].shape)
    q["max_d2"][2::37] = 0.0
    q["max_d2"][3::41] = -1.0
    q["max_d2"][4::43] = np.nan
    assert n > 3000
    return q


def exact_d2(pt, tri):
    """float64 squared distance from points (n, 3) to triangles (n, 3, 3): the plane's foot if it lies inside the triangle,
    else the nearest of the three segments (zero-area triangles: the segments)."""
    p, a, b, c = pt.astype(np.float64), tri[:, 0].astype(np.float64), tri[:, 1].astype(np.float64), tri[:, 2].astype(np.float64)

    def seg(o, e):
        ee = np.einsum("ij,ij->i", e, e)
        with np.errstate(all="ignore"):
            t = np.where(ee > 0, np.einsum("ij,ij->i", p - o, e) / ee, 0.0)
        t = np.clip(np.nan_to_num(t), 0.0, 1.0)
        d = p - (o + e * t[:, None])
        return np.einsum("ij,ij->i", d, d)
    best = np.minimum(np.minimum(seg(a, b - a), seg(a, c - a)), seg(b, c - b))
    n = np.cross(b - a, c - a)
    nn = np.einsum("ij,ij->i", n, n)
    with np.errstate(all="ignore"):
        s = np.einsum("ij,ij->i", p - a, n) / nn
        foot = p - n * s[:, None]
        inside = np.ones(p.shape[0], dtype=bool)
        for u, v in ((a, b), (b, c), (c, a)):
            inside &= np.einsum("ij,ij->i", np.cross(v - u, foot - u), n) >= 0
        plane = s * s * nn
    return np.where((nn > 0) & inside, np.minimum(best, plane), best)


def awkward_triangles(rng, n):
    """Random triangles, slivers, collinear and zero-area ones, repeated vertices, huge and tiny coordinates, each with a
    query point that is random, or exactly on a vertex, an edge or the face. Returns (points, triangles, kinds)."""
    a = rng.normal(size=(n, 3)); b = rng.normal(size=(n, 3)); c = rng.normal(size=(n, 3))
    kind = rng.integers(0, 6, n)
    c = np.where((kind == 1)[:, None], a + (b - a) * 0.5 + rng.normal(0, 1e-4, (n, 3)), c)   # sliver
    c = np.where((kind == 2)[:, None], a + (b - a) * 2.0, c)                                  # collinear
    b = np.where((kind == 3)[:, None], a, b)                                                  # repeated vertex
    b = np.where((kind == 4)[:, None], a, b); c = np.where((kind == 4)[:, None], a, c)        # a point
    # huge and tiny: the region values va, vb, vc are fourth powers of the coordinates; fp32 holds them as normal numbers
    # for coordinates of about 1e-9 .. 1e9
    scale = np.where(rng.random(n) < 0.2, 1e8, np.where(rng.random(n) < 0.25, 1e-4, 1.0))[:, None]
    tri = (np.stack([a, b, c], 1) * scale[:, :, None]).astype(np.float32)
    w = rng.dirichlet((1.0, 1.0, 1.0), n)
    where = rng.integers(0, 4, n)
    on_face = np.einsum("nk,nkd->nd", w, tri.astype(np.float64))
    on_edge = tri[:, 0] + (tri[:, 1].astype(np.float64) - tri[:, 0]) * w[:, :1]
    pt = np.where((where == 0)[:, None], rng.normal(size=(n, 3)) * 2 * scale, np.where((where == 1)[:, None], tri[:, 0],
                  np.where((where == 2)[:, None], on_edge, on_face))).astype(np.float32)
    return pt, tri, kind


def test_oracle_distance_agrees_with_float64():
    rng = np.random.default_rng(5)
    pt, tri, kind = awkward_triangles(rng, 4000)
    got = np.array([pq.oracle_on_triangle(pt[i], *tri[i]) for i in range(pt.shape[0])])
    want = exact_d2(pt, tri)
    scale = np.max(np.abs(np.concatenate([pt[:, None], tri], 1).astype(np.float64)), axis=(1, 2))
    err = np.abs(np.sqrt(got[:, 0].astype(np.float64)) - np.sqrt(want)) / scale
    # the distance to within 1e-5 of the coordinates' magnitude (~100 fp32 ulp: cancellation in the dot products) ...
    t64 = tri.astype(np.float64)
    cr = np.linalg.norm(np.cross(t64[:, 1] - t64[:, 0], t64[:, 2] - t64[:, 0]), axis=1)
    longest = np.max(np.linalg.norm(t64 - np.roll(t64, 1, axis=1), axis=2), axis=1)
    with np.errstate(all="ignore"):
        quality = np.where(longest > 0, cr / (longest * longest), 0.0)
    well = (quality > 1e-2) | (quality == 0)
    assert (err[well] <= 1e-5).all(), np.max(err[well])
    # ... except on slivers (area small against the longest edge squared), whose barycentrics (vb, vc over their sum) are
    # ill-conditioned in fp32: the clamp into the vertex box still bounds the point, and most are accurate
    assert (err[~well] <= 2.0 * np.sqrt(3.0)).all() and np.mean(err[~well] <= 1e-5) > 0.8, np.mean(err[~well] <= 1e-5)
    assert np.isfinite(got).all() and (got[:, 0] >= 0).all()
    u, v = got[:, 1], got[:, 2]
    assert (u >= 0).all() and (v >= 0).all() and (u + v <= 1.0 + 1e-6).all()
    # the product's distance routine gives the oracle's records bit for bit
    emu = pq.emu_on_triangles(pt, tri)
    assert np.array_equal(emu.view(np.uint32), got.astype(np.float32).view(np.uint32))


def test_vertex_edge_face_points_are_at_distance_zero():
    tri = np.array([[0.0, 0.0, 0.0], [4.0, 0.0, 0.0], [0.0, 2.0, 0.0]], dtype=np.float32)
    for p, uv in (((0, 0, 0), (0, 0)), ((4, 0, 0), (1, 0)), ((0, 2, 0), (0, 1)), ((2, 0, 0), (0.5, 0)), ((0, 1, 0), (0, 0.5)),
                  ((1, 0.5, 0), (0.25, 0.25))):
        d2, u, v = pq.oracle_on_triangle(np.array(p, dtype=np.float32), *tri)
        assert d2 == 0.0 and (u, v) == uv
    d2, u, v = pq.oracle_on_triangle(np.array((1, 0.5, 3), dtype=np.float32), *tri)
    assert d2 == 9.0 and (u, v) == (0.25, 0.25)


def _scene(tmp_scene_dir, name, p, n, f, max_prims=4):
    return _reference_scene(scenes.write_obj(os.path.join(tmp_scene_dir, name), p, n, f), max_prims)


def _emu_matches_oracle(tris, nodes, q, lb_sample=400):
    st = pq.emu_build(tris, nodes)
    want = pq.oracle_closest_point(tris, q)
    s = pq.ol.EmuStats()
    same(pq.emu_closest_point(q, stats=s), want)
    assert s.overflow == 0 and s.max_stack < st.stack_bound
    sub = q[np.linspace(0, q.shape[0] - 1, min(lb_sample, q.shape[0])).astype(np.int64)]
    violations, children = pq.emu_lb_check(sub)
    assert children > 0 and violations == 0
    return st, want


def _icosphere(subdiv):
    p, f = scenes.icosphere(subdiv)
    return p.astype(np.float32), (p / np.linalg.norm(p, axis=1, keepdims=True)).astype(np.float32), f


def test_emu_icosphere_and_displaced_sphere(tmp_scene_dir, bumpy_ref):
    tris, nodes, _ = _scene(tmp_scene_dir, "pico.obj", *_icosphere(3))
    _, want = _emu_matches_oracle(tris, nodes, query_sets(positions(tris), 11))
    assert (want["tri"] != MISS).mean() > 0.5
    tris, nodes, _ = bumpy_ref
    _emu_matches_oracle(tris, nodes, query_sets(positions(tris), 12)[::4], lb_sample=60)


def test_emu_scattered_triangles(tmp_scene_dir):
    tris, nodes, _ = _scene(tmp_scene_dir, "pscatter.obj", *scenes.scattered_triangles(3000))
    _emu_matches_oracle(tris, nodes, query_sets(positions(tris), 13))


def test_emu_tie_grid_index_tie_break(tmp_scene_dir):
    """Coincident lattices: many triangles in different leaves at the same d2; the smallest index must win."""
    tris, nodes, _ = _scene(tmp_scene_dir, "pties.obj", *scenes.tie_grid(16, layers=3))
    p = positions(tris)
    rng = np.random.default_rng(14)
    lattice = np.stack(np.meshgrid(np.arange(0, 16.5, 0.5), np.arange(0, 16.5, 0.5), [0.0, 0.5, -0.5, 3.0], indexing="ij"), -1)
    q = np.concatenate([pq.queries(lattice.reshape(-1, 3)), query_sets(p, 15)])
    st, want = _emu_matches_oracle(tris, nodes, q)
    assert st.n_leaf_blocks > 1
    # ties really occur: several triangles reach the winning d2
    sub = q[:300]
    d2 = np.array([[pq.oracle_on_triangle(np.array([s["x"], s["y"], s["z"]], dtype=np.float32), *t)[0] for t in p[:400]] for s in sub[:40]])
    assert ((d2 == d2.min(1, keepdims=True)).sum(1) > 1).mean() > 0.5


def test_emu_fuzz(tmp_scene_dir):
    host = load_product().host
    rng = np.random.default_rng(16)
    for case in range(8):
        pos, faces = scenes.fuzz_scene(case, rng)
        nrm = np.tile(np.array([[0.0, 0.0, 1.0]], dtype=np.float32), (pos.shape[0], 1))
        path = scenes.write_obj(os.path.join(tmp_scene_dir, "pfuzz%d.obj" % case), pos, nrm, faces)
        tris, nodes, _ = host.load_scene(path, int(rng.choice([1, 2, 4, 8])))
        _emu_matches_oracle(tris, nodes, query_sets(positions(tris), 100 + case))


@pytest.mark.parametrize("depth", [31, 32, 63, 64, 127, 128, 255])
def test_emu_deep_chains(tmp_scene_dir, depth):
    tris, nodes, _ = dt.chain(load_product().host, tmp_scene_dir, depth)
    st, _ = _emu_matches_oracle(tris, nodes, query_sets(positions(tris), depth), lb_sample=200)
    assert st.stack_bound == depth + 1


def test_max_d2_and_point_edge_cases(tmp_scene_dir):
    tris, nodes, _ = _scene(tmp_scene_dir, "pedge.obj", *_icosphere(2))
    p = positions(tris)
    pts = np.concatenate([p[:50, 0], p[:50].mean(1) * 1.3, np.zeros((1, 3))]).astype(np.float32)
    cases = []
    for m in (0.0, 1e-6, 0.05, np.inf, -1.0, -0.0, np.nan, -np.inf):
        cases.append(pq.queries(pts, m))
    odd = pq.queries(np.array([[np.nan, 0, 0], [0, np.nan, 0], [0, 0, np.nan], [np.inf, 0, 0], [0, -np.inf, 0],
                               [np.inf, np.inf, -np.inf], [3e38, 0, 0], [1e-40, 0, 1.0]], dtype=np.float32), np.inf)
    odd2 = odd.copy()
    odd2["max_d2"] = 4.0
    q = np.concatenate(cases + [odd, odd2])
    _, want = _emu_matches_oracle(tris, nodes, q)
    miss = want["tri"] == MISS
    md = q["max_d2"]
    assert (miss[~(md >= 0)]).all()                                               # negative / NaN max_d2
    assert np.array_equal(want["d2"][miss].view(np.uint32), md[miss].view(np.uint32))
    assert not want["u"][miss].view(np.uint32).any() and not want["v"][miss].view(np.uint32).any()
    nanpt = np.isnan(q["x"]) | np.isnan(q["y"]) | np.isnan(q["z"])
    assert miss[nanpt].all()
    on_vertex = np.concatenate([np.arange(50) + pts.shape[0] * i for i in range(len(cases))])
    ok = md[on_vertex] >= 0
    assert (want["d2"][on_vertex][ok] == 0).all()                                 # max_d2 = 0 still finds a point on the surface
    inf_pt = np.isinf(q["x"]) | np.isinf(q["y"]) | np.isinf(q["z"])
    assert (want["tri"][inf_pt & (md == np.inf)] == 0).all()                      # every candidate at d2 = inf: the smallest index
    assert miss[inf_pt & (md == 4.0)].all()


# ---- SASS: the lb and d2 sequences are not contracted ---------------------------------------------------------------
PROBE = r"""
#include "point_query.cuh"
using namespace b2rt;
extern "C" __global__ void probe_lb(const uint4* in, float* out) {
    const U4* p = reinterpret_cast<const U4*>(in) + 8 * threadIdx.x;
    float lb[8];
    const float* f = reinterpret_cast<const float*>(in + 8 * threadIdx.x + 5);
    wide_child_lbs(p[0], p[2], p[3], p[4], f[0], f[1], f[2], lb);
    for (int c = 0; c < 8; ++c) out[8 * threadIdx.x + c] = lb[c];
}
extern "C" __global__ void probe_box_d2(const float* in, float* out) {
    const float* f = in + 16 * threadIdx.x;
    out[2 * threadIdx.x] = box_lb(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], f[8]);
    out[2 * threadIdx.x + 1] = dist2(f[0], f[1], f[2], clamp_box(f[9], f[3], f[6]), clamp_box(f[10], f[4], f[7]), clamp_box(f[11], f[5], f[8]));
}
extern "C" __global__ void probe_tri(const float* in, float* out) {
    const float* f = in + 12 * threadIdx.x;
    float d2, u, v;
    closest_on_triangle(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], f[8], f[9], f[10], f[11], d2, u, v);
    out[3 * threadIdx.x] = d2; out[3 * threadIdx.x + 1] = u; out[3 * threadIdx.x + 2] = v;
}
// the seven divisions of closest_on_triangle on their own: their __fdiv_rn expansion is the only FFMA the routine may have
extern "C" __global__ void probe_div(const float* in, float* out) {
    const float* f = in + 14 * threadIdx.x;
    for (int i = 0; i < 7; ++i) out[7 * threadIdx.x + i] = xdiv(f[2 * i], f[2 * i + 1]);
}
"""


def _nvcc_flags():
    spec = importlib.util.spec_from_file_location("_b2rt_build_flags_pq", os.path.join(ROOT, "mini-opencl-raytracer_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.NVCC, [f for f in mod.NVCC_FLAGS if f != "-Xcompiler" and not f.startswith("-fPIC")]


def _opcodes(sass, kernel):
    body = re.split(r"\n\s*Function : ", sass)
    text = next(b for b in body if b.split("\n", 1)[0].strip() == kernel)
    ops = collections.Counter()
    for line in text.splitlines():
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_]+)", line)
        if m:
            ops[m.group(1)] += 1
    return ops


def test_lb_and_d2_sequences_are_not_contracted(tmp_path):
    nvcc, flags = _nvcc_flags()
    if not (os.path.exists(nvcc) or shutil.which(nvcc)) or shutil.which("cuobjdump") is None:
        pytest.skip("needs nvcc and cuobjdump")
    src = tmp_path / "probe.cu"
    src.write_text(PROBE)
    cubin = tmp_path / "probe.cubin"
    subprocess.run([nvcc] + flags + ["-cubin", "-o", str(cubin), str(src)], check=True, capture_output=True, text=True)
    sass = subprocess.run(["cuobjdump", "-sass", str(cubin)], check=True, capture_output=True, text=True).stdout
    lb, box, tri, div = (_opcodes(sass, k) for k in ("probe_lb", "probe_box_d2", "probe_tri", "probe_div"))
    for ops in (lb, box, tri):
        assert ops["FFMA2"] == 0 and ops["FMUL2"] == 0 and ops["FADD2"] == 0, dict(ops)
    assert lb["FFMA"] == 48, "the plane decode is 6 FFMA per child slot, nothing else: %d" % lb["FFMA"]
    assert box["FFMA"] == 0
    assert tri["FFMA"] <= div["FFMA"], "closest_on_triangle has FFMA beyond its divisions (%d > %d)" % (tri["FFMA"], div["FFMA"])
