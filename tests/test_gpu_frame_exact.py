"""-m gpu: the frame path held to the oracle bit for bit.

The reference is the oracle with powf / sinf / cosf evaluated like the kernels' pow_cr / sin_cr / cos_cr (fp64, rounded
once): tests/frame_oracle/oracle_devlibm.c, tied to the glibc oracle by tests/test_frame_oracle_devlibm.py. Every other
operation is the same fp32 arithmetic in the same order on both sides, so frames must agree on every pixel. The
product-against-product frame tests elsewhere cannot see a shading bug, since both sides share csrc/shade.cuh; these
can. The shading functions themselves are compared one by one on edge and random inputs through the device probe
(tests/frame_oracle/shade_probe.cu).

NaN pixels compare as equal whatever their payload (the CPU's default NaN differs from the GPU's)."""
import os

import numpy as np
import pytest

import deep_trees as dt
import frame_oracle_lib as fl
import scenes
from test_frame_oracle_devlibm import check_against_powf, pow_records, special_pow_table, ulp_diff

pytestmark = pytest.mark.gpu
F32 = np.float32
ONE_SEED_COUNT = 24


# ---- the RNG inverted: seeds whose n-th rnd() draw is exactly 0 or 1 ----------------------------------------------------
def _hash_step(x):
    x = np.uint64(x)
    m = np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16); x = (x * np.uint64(0x7feb352d)) & m
    x ^= x >> np.uint64(15); x = (x * np.uint64(0x846ca68b)) & m
    x ^= x >> np.uint64(16)
    return int(x)


def _unhash_step(y):
    y ^= y >> 16
    y = (y * pow(0x846ca68b, -1, 1 << 32)) & 0xFFFFFFFF
    y ^= (y >> 15) ^ (y >> 30)
    y = (y * pow(0x7feb352d, -1, 1 << 32)) & 0xFFFFFFFF
    y ^= y >> 16
    return y


def seeds_drawing_one(draw, first_above_half=None, count=ONE_SEED_COUNT):
    """Seeds whose draw-th rnd() (1-based) is exactly 1.0 (state >= 2^32 - 128 rounds to 2^32); first_above_half
    selects on the first draw (> 0.5: SampleBrdf's specular branch)."""
    out = []
    for t in range(0xFFFFFF80, 0x100000000):
        s = t
        for _ in range(draw):
            s = _unhash_step(s)
        if first_above_half is not None and (_hash_step(s) > 0x80000000) != first_above_half:
            continue
        out.append(s)
        if len(out) == count:
            break
    return out


def test_seed_inversion():
    for draw, first_above_half in ((4, True), (3, False), (1, None)):
        for s in seeds_drawing_one(draw, first_above_half, 4):
            rec = fl.records(1)
            rec[0, 0] = s
            draws = []
            for _ in range(draw):
                out = fl.oracle_run(fl.OP_RND, rec)
                draws.append(float(out[0, :1].view(F32)[0]))
                rec[0, 0] = out[0, 1]
            assert draws[-1] == 1.0
            assert first_above_half is None or (draws[0] > 0.5) == first_above_half


# ---- inputs of the shading functions ----------------------------------------------------------------------------------
def _unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def edge_normals():
    x = [F32(0.001), np.nextafter(F32(0.001), F32(0)), np.nextafter(F32(0.001), F32(1)), F32(-0.001),
         np.nextafter(F32(-0.001), F32(-1))]
    n = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, -1), (0.0, -1.0, 0.0)]
    n += [(float(v), float(np.sqrt(1.0 - float(v) ** 2)), 0.0) for v in x]           # |n.x| on either side of 0.001
    n += [tuple(_unit((1.0, 2.0, -2.0)))]
    return np.array(n, dtype=F32)


def grazing_wo(n):
    """Directions at cos(wo, n) = 1, 0.5, 1e-3, 1e-6 (the rejection threshold of SampleBrdf), 0 and -1e-6."""
    n64 = n.astype(np.float64)
    a = np.array([0.0, 0.0, 1.0]) if abs(n64[2]) < 0.9 else np.array([1.0, 0.0, 0.0])
    t = _unit(np.cross(a, n64))
    return np.array([c * n64 + np.sqrt(1 - c * c) * t for c in (1.0, 0.5, 1e-3, 1e-6, 0.0, -1e-6)], dtype=F32)


ROUGHNESS = [0.0, 1e-20, 0.05, 0.3, 0.7, 0.999, 1.0, float(F32(np.sqrt(2.0))), 92.16, 9999.0]


def brdf_records(rng, n_random):
    rows = []
    seeds = [0, 1, 12345] + seeds_drawing_one(4, True) + seeds_drawing_one(3, False) + seeds_drawing_one(2) + \
        [int(s) for s in rng.integers(0, 1 << 32, 16)]
    for nrm in edge_normals():
        for wo in grazing_wo(nrm):
            for r in ROUGHNESS:
                for spec in (0.0, 0.5):
                    for s in seeds:
                        rows.append((wo, nrm, r, spec, s))
    rec = fl.records(len(rows) + n_random)
    f = rec.view(F32)
    for i, (wo, nrm, r, spec, s) in enumerate(rows):
        f[i, 0:3], f[i, 3:6], f[i, 6] = wo, nrm, r
        f[i, 7:10], f[i, 10:13] = spec, (0.8, 0.5, 0.2)
        rec[i, 13] = s
    k = len(rows)
    nrm = _unit(rng.normal(size=(n_random, 3)))
    wo = _unit(nrm + rng.normal(size=(n_random, 3)) * rng.uniform(0.1, 3.0, (n_random, 1)))
    f[k:, 0:3], f[k:, 3:6] = wo.astype(F32), nrm.astype(F32)
    f[k:, 6] = np.where(rng.random(n_random) < 0.5, rng.uniform(0.0, 1.5, n_random), rng.choice(ROUGHNESS, n_random))
    f[k:, 7:10] = rng.uniform(0, 1, (n_random, 3))
    f[k:, 10:13] = rng.uniform(0, 1, (n_random, 3))
    rec[k:, 13] = rng.integers(0, 1 << 32, n_random, dtype=np.uint64)
    return rec


def pow_edge_and_random(rng, n_random):
    a, b = special_pow_table()
    ra = rng.uniform(0, 1, n_random).astype(F32)
    ra[::7] = rng.uniform(0, 60, ra[::7].shape).astype(F32)
    rb = rng.choice(np.array([2.0, 2.2, 0.45454545, 0.454545], dtype=F32), n_random)
    rb[::3] = (1.0 / (2.0 / rng.uniform(0.0, 1.5, rb[::3].shape) ** 2 - 2.0 + 1.0)).astype(F32)
    return pow_records(np.concatenate([a, ra]), np.concatenate([b, rb])), a.shape[0]


def sincos_records(rng, n_random):
    edge = np.array([0.0, -0.0, 1e-45, 1e-30, 1e-4, np.pi / 2, np.pi, 3 * np.pi / 2, 6.28318530718, 1e4, 1e30, 3e38,
                     -1.0, np.inf, np.nan], dtype=F32)
    rnd = (F32(6.28318530718) * rng.uniform(0, 1, n_random).astype(F32)).astype(F32)
    rec = fl.records(edge.shape[0] + n_random)
    rec.view(F32)[:, 0] = np.concatenate([edge, rnd])
    return rec, edge.shape[0]


def frame_records(rng, n_random):
    rows = []
    for nrm in edge_normals():
        for phi in (0.0, 1e-30, 1.5707964, 3.1415927, 6.28318530718, 1e4, -1.0):
            for st in (0.0, 0.5, 1.0):
                for ct in (1.0, 0.5, 0.0):
                    rows.append(tuple(nrm) + (phi, st, ct))
    rec = fl.records(len(rows) + n_random)
    f = rec.view(F32)
    f[:len(rows), 0:6] = np.array(rows, dtype=F32)
    k = len(rows)
    f[k:, 0:3] = _unit(rng.normal(size=(n_random, 3))).astype(F32)
    f[k:, 3] = F32(6.28318530718) * rng.uniform(0, 1, n_random).astype(F32)
    s2 = rng.uniform(0, 1, n_random).astype(F32)
    f[k:, 4], f[k:, 5] = np.sqrt(s2), np.sqrt(F32(1) - s2)
    return rec, k


def light_records(rng, n_random):
    rows = []
    origins = [(0.0, -25.0, 8.5), (0.0, -5.0, 8.0), (3.0, 1.0, -2.0)]                 # (0, -5, 8): the eye vector is 0
    for o in origins:
        for d in ((0.0, 1.0, 0.0), tuple(_unit((0.3, 0.9, -0.2)))):
            for t in (-1.0, 0.0, 1e-30, 5.0, 1e30, 3e38, np.inf):
                for nrm in edge_normals()[:8]:
                    for lt in (-1, 0, 1, 2, 3):
                        rows.append((o, d, t, nrm, lt))
    rec = fl.records(len(rows) + n_random)
    f = rec.view(F32)
    for i, (o, d, t, nrm, lt) in enumerate(rows):
        f[i, 0:3], f[i, 3:6], f[i, 6], f[i, 7:10] = o, d, t, nrm
        rec[i, 10] = np.uint32(lt & 0xFFFFFFFF)
    k = len(rows)
    f[k:, 0:3] = rng.uniform(-20, 20, (n_random, 3))
    f[k:, 3:6] = _unit(rng.normal(size=(n_random, 3)))
    f[k:, 6] = rng.uniform(-1, 60, n_random)
    f[k:, 7:10] = _unit(rng.normal(size=(n_random, 3)))
    rec[k:, 10] = rng.integers(-1, 4, n_random).astype(np.int64) & 0xFFFFFFFF
    return rec, k


def camera_records(rng, n_random):
    angle = fl.camera_angle()
    rows = []
    cams = [((0.0, 1.0, 0.0), (0.0, 0.0, 1.0)), ((0.0, 0.0, -1.0), (0.0, 1.0, 0.0)), ((1.0, 0.0, 0.0), (0.0, 0.0, 1.0))]
    seeds = [0, 7] + seeds_drawing_one(1, count=2) + seeds_drawing_one(2, count=2)
    for w, h in ((1, 1), (3, 3), (5, 7), (333, 211), (1920, 1080), (65, 49)):
        for gid in sorted({0, (h // 2) * w + w // 2, w * h - 1, w - 1}):
            for s in seeds:
                for front, up in cams:
                    rows.append((w, h, gid, s, front, up))
    rec = fl.records(len(rows) + n_random)
    f = rec.view(F32)
    for i, (w, h, gid, s, front, up) in enumerate(rows):
        rec[i, 0:4] = (w, h, gid, s)
        f[i, 5:8], f[i, 8:11] = front, up
    k = len(rows)
    w = rng.integers(1, 4000, n_random)
    h = rng.integers(1, 3000, n_random)
    rec[k:, 0], rec[k:, 1] = w, h
    rec[k:, 2] = (rng.uniform(0, 1, n_random) * w * h).astype(np.int64)
    rec[k:, 3] = rng.integers(0, 1 << 32, n_random, dtype=np.uint64)
    f[k:, 5:8], f[k:, 8:11] = cams[0]
    f[:, 4] = angle
    return rec, k


def rnd_records(rng, n_random):
    edge = [0, 1, 0xFFFFFFFF, 0x80000000] + seeds_drawing_one(1, count=8)
    rec = fl.records(len(edge) + n_random)
    rec[:len(edge), 0] = edge
    rec[len(edge):, 0] = rng.integers(0, 1 << 32, n_random, dtype=np.uint64)
    return rec, len(edge)


def accumulate_records(rng, n_random):
    olds = [0.0, 1e-45, 1e-40, 0.5, 1.0, 7.5, np.inf, np.nan]
    rads = [0.0, 1e-45, 0.3, 1.0, 50.0, np.inf, np.nan]
    counts = [0, 1, 2, 3, 1 << 24, (1 << 24) + 1, 0xFFFFFFFF]
    rows = [(o, r, c) for o in olds for r in rads for c in counts]
    rec = fl.records(len(rows) + n_random)
    f = rec.view(F32)
    for i, (o, r, c) in enumerate(rows):
        f[i, 0:3], f[i, 4:7] = o, (r, r * 0.5, 0.0)
        rec[i, 7] = c
    k = len(rows)
    f[k:, 0:3] = rng.uniform(0, 2, (n_random, 3))
    f[k:, 4:7] = rng.uniform(0, 4, (n_random, 3))
    rec[k:, 7] = rng.integers(0, 300, n_random)
    return rec, k


def _differing(got, want):
    """Records whose outputs differ in any word (a NaN equals any NaN)."""
    gf, wf = got.view(F32), want.view(F32)
    same = (got == want) | (np.isnan(gf) & np.isnan(wf))
    return ~same.all(axis=1)


CASES = {"pow_cr": (fl.OP_POW, lambda rng, n: pow_edge_and_random(rng, n), 200000),
         "sin_cr/cos_cr": (fl.OP_SINCOS, sincos_records, 200000),
         "frame_sample": (fl.OP_FRAME, frame_records, 100000),
         "sample_brdf": (fl.OP_BRDF, lambda rng, n: (brdf_records(rng, n), None), 250000),
         "light_pixel": (fl.OP_LIGHT, light_records, 100000),
         "camera_dir": (fl.OP_CAMERA, camera_records, 100000),
         "rnd": (fl.OP_RND, rnd_records, 50000),
         "accumulate": (fl.OP_ACCUMULATE, accumulate_records, 100000)}


@pytest.mark.parametrize("name", list(CASES))
def test_shading_function_matches_the_oracle(name):
    """Edge inputs must agree bit for bit. Random inputs may differ only where CUDA's and glibc's fp64 exp2 / log2 / sin /
    cos round to different doubles right at a float rounding boundary: estimated from their error bounds at a few per
    10^9 calls. Measured on a B200: 0 of the 1.1 * 10^6 random records differ; the bound below leaves room for 2 per
    case, each within 2 ulp."""
    op, make, n_random = CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    rec, n_edge = make(rng, n_random)
    if n_edge is None:
        n_edge = rec.shape[0] - n_random
    got, want = fl.probe_run(op, rec), fl.oracle_run(op, rec)
    bad = _differing(got, want)
    edge_bad = np.flatnonzero(bad[:n_edge])
    assert edge_bad.size == 0, (name, [(rec[i].view(F32)[:14].tolist(), got[i].view(F32)[:8].tolist(), want[i].view(F32)[:8].tolist())
                                       for i in edge_bad[:5]])
    rnd_bad = np.flatnonzero(bad[n_edge:]) + n_edge
    print("%s: %d of %d random records differ" % (name, rnd_bad.size, n_random))
    assert rnd_bad.size <= 2, (name, rnd_bad.size)
    for i in rnd_bad:
        assert ulp_diff(got[i].view(F32), want[i].view(F32)).max() <= 2, name


def test_pow_cr_special_values_follow_powf():
    """pow_cr on the device: the special values of C99 powf for the bases and exponents the kernels pass (x^0 = 1 for x = 0,
    inf and NaN; 1^y = 1 for y = +-inf and NaN among them), the rest within 1 ulp of glibc powf."""
    a, b = special_pow_table()
    got = fl.probe_run(fl.OP_POW, pow_records(a, b))[:, 0].view(F32)
    check_against_powf(got, a, b)


def test_pow_sin_cos_within_one_ulp_of_extended_precision():
    """The claim of csrc/shade.cuh: fp64 evaluation rounded once is within 1 ulp of the exact value (long double here)."""
    rng = np.random.default_rng(5)
    n = 200000
    a = rng.uniform(0, 1, n).astype(F32)
    a[::4] = rng.uniform(0, 100, a[::4].shape).astype(F32)
    b = rng.choice(np.array([2.2, 0.45454545, 0.454545], dtype=F32), n)
    b[::3] = rng.uniform(-3, 40, b[::3].shape).astype(F32)
    got = fl.probe_run(fl.OP_POW, pow_records(a, b))[:, 0].view(F32)
    exact = np.power(a.astype(np.longdouble), b.astype(np.longdouble))
    fin = np.isfinite(exact) & (exact < np.longdouble(3e38)) & (exact > np.longdouble(1e-37))
    assert fin.mean() > 0.9
    assert ulp_diff(got[fin], exact[fin].astype(F32)).max() <= 1
    x = (F32(6.28318530718) * rng.uniform(0, 1, n).astype(F32)).astype(F32)
    rec = fl.records(n)
    rec.view(F32)[:, 0] = x
    out = fl.probe_run(fl.OP_SINCOS, rec).view(F32)
    xl = x.astype(np.longdouble)
    assert ulp_diff(out[:, 0], np.sin(xl).astype(F32)).max() <= 1
    assert ulp_diff(out[:, 1], np.cos(xl).astype(F32)).max() <= 1


# ---- whole frames -------------------------------------------------------------------------------------------------------
CAM_B = dict(pos=(0.0, -30.0, 4.0), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0))


def _assert_frame(got, want, what):
    gb, wb = got.view(np.uint32), want.view(np.uint32)
    same = (gb == wb) | (np.isnan(got) & np.isnan(want))
    bad = np.flatnonzero(~same.all(axis=1))
    assert bad.size == 0, "%s: %d pixels differ, first %s: got %s want %s" % (what, bad.size, bad[:4].tolist(),
                                                                             got[bad[:2]].tolist(), want[bad[:2]].tolist())


def _compare(ctx, scene, W, H, frames, bounces, light_type=0, sky=1.0, what="", execute=None, **cam):
    """Render `frames` into a fresh image on the GPU and in the fp64-libm oracle; compare after every frame."""
    tris, nodes, mats = scene
    want = np.zeros((W * H, 4), dtype=F32)
    ctx.resize(W, H)
    for fc in frames:
        ctx.set_frame(fc, bounces, light_type=light_type, sky=sky, **cam)
        if execute is None:
            ctx.execute(W * H)
        else:
            execute(ctx, W, H)
        fl.oracle_render(tris, nodes, mats, want, W, H, fc, bounces, light_type=light_type, sky=sky, **cam)
        _assert_frame(ctx.read_pixels(), want, "%s frame %d (lt %d, sky %g, bounces %d)" % (what, fc, light_type, sky, bounces))
    return want


@pytest.fixture(scope="module")
def cornell_ctx(product, cornell_ref):
    ctx = product.Context(0)
    ctx.upload_scene(*cornell_ref)
    yield ctx
    ctx.close()


def test_cornell_sweep(cornell_ctx, cornell_ref):
    """Light types 0/1/2, sky 0/1/2.5, bounces 0/1/4/9, frame 0 alone and frames 1-3, at an odd size (the centre column
    and row)."""
    for lt in (0, 1, 2):
        for sky in (0.0, 1.0, 2.5):
            for bounces in (0, 1, 4, 9):
                for frames in ((0,), (1, 2, 3)):
                    _compare(cornell_ctx, cornell_ref, 65, 49, frames, bounces, lt, sky, "cornell 65x49")


def test_cornell_full_size_long_runs_and_huge_frame_counts(cornell_ctx, cornell_ref):
    for lt in (0, 1, 2):
        _compare(cornell_ctx, cornell_ref, 256, 256, (1, 2, 3), 4, lt, what="cornell 256^2")
    _compare(cornell_ctx, cornell_ref, 256, 256, (0,), 9, what="cornell 256^2")
    _compare(cornell_ctx, cornell_ref, 33, 17, range(1, 65), 4, 1, what="cornell 64 frames")
    # 2^24 + 1 is not a float: fc rounds to fm1 = 2^24. 2^32 - 1 wraps the seed's hash
    _compare(cornell_ctx, cornell_ref, 64, 63, (1 << 24, (1 << 24) + 1, 0xFFFFFFFF), 4, 2, what="cornell 2^24")


def _material_sweep(mats, tris, rng):
    """Materials for every roughness of ROUGHNESS x specular {0, 0.5} x emission {0, 0.6}, given per triangle."""
    rows = []
    for r in ROUGHNESS:
        for spec in (0.0, 0.5):
            for em in (0.0, 0.6):
                m = np.zeros(16, dtype=F32)
                m[0:3] = rng.uniform(0.1, 0.9, 3)
                m[4:7] = spec
                m[8:11] = em
                m[13], m[14] = r, 1.0
                rows.append(m)
    new_mats = np.ascontiguousarray(np.stack(rows)).view(np.uint8).reshape(-1, 64)
    new_tris = tris.copy()
    new_tris.view(np.uint32).reshape(-1, 64)[:, 60] = rng.integers(0, len(rows), tris.shape[0])
    return new_tris, new_mats


def test_cornell_material_sweep(product, cornell_ref):
    """Cornell's geometry with GGX lobes of every roughness (the glossy branch no loaded test material reaches)."""
    tris, nodes, _ = cornell_ref
    t2, m2 = _material_sweep(cornell_ref[2], tris, np.random.default_rng(17))
    with product.Context(0) as ctx:
        ctx.upload_scene(t2, nodes, m2)
        for lt in (0, 1, 2):
            _compare(ctx, (t2, nodes, m2), 97, 75, (1, 2, 3), 6, lt, what="material sweep")
        _compare(ctx, (t2, nodes, m2), 97, 75, (0,), 9, 1, 2.5, what="material sweep")


def test_execution_paths(product, cornell_ctx, cornell_ref):
    """Render modes 0/1/2, wavefront lanes 2-4, execute_range shards and the reference-layout walk on the material sweep."""
    cap = product.capi
    t2, m2 = _material_sweep(cornell_ref[2], cornell_ref[0], np.random.default_rng(18))
    scene = (t2, cornell_ref[1], m2)
    ctx = cornell_ctx
    ctx.upload_scene(*scene)
    try:
        for mode in (0, 1, 2):
            ctx.set_option(cap.OPT_RENDER_MODE, mode)
            _compare(ctx, scene, 131, 67, range(1, 7), 5, 1, what="render mode %d" % mode)
        ctx.set_option(cap.OPT_RENDER_MODE, 0)
        for lanes in (2, 3, 4):
            ctx.set_option(cap.OPT_WAVEFRONT_LANES, lanes)
            _compare(ctx, scene, 131, 67, (1, 2), 5, 2, what="wavefront lanes %d" % lanes)
        ctx.set_option(cap.OPT_WAVEFRONT_LANES, 0)
        ctx.set_option(cap.OPT_RENDER_MODE, 2)

        def shards(c, W, H):
            for lo in range(0, W * H, 1999):
                c.execute_range(lo, min(lo + 1999, W * H))
        _compare(ctx, scene, 131, 67, (1, 2), 5, 0, execute=shards, what="execute_range shards")
        ctx.set_option(cap.OPT_TRAVERSAL, 1)
        try:
            _compare(ctx, scene, 131, 67, (1, 2), 5, 1, what="reference-layout walk")
        finally:
            ctx.set_option(cap.OPT_TRAVERSAL, 0)
    finally:
        for opt, v in ((cap.OPT_RENDER_MODE, 2), (cap.OPT_WAVEFRONT_LANES, 0)):
            ctx.set_option(opt, v)
        ctx.upload_scene(*cornell_ref)


def test_other_scenes(product, tmp_scene_dir, bumpy_ref):
    """The bumpy sphere, a tie grid (exact t ties across leaves), a deep chain (stack bound 201)."""
    p, n, f = scenes.tie_grid(24, layers=3)
    ties = product.host.load_scene(scenes.write_obj(os.path.join(tmp_scene_dir, "exact_ties.obj"), p, n, f), 4)
    chain = dt.chain(product.host, tmp_scene_dir, 200, axes=(0, 1, 2))
    for name, scene, cam, bounces in (("bumpy", bumpy_ref, CAM_B, 5),
                                      ("tie grid", ties, dict(pos=(12.0, 12.0, 30.0), front=(0.0, 0.0, -1.0), up=(0.0, 1.0, 0.0)), 3),
                                      ("chain", chain, dict(pos=(-10.0, 0.4, 0.6), front=(1.0, 0.0, 0.0), up=(0.0, 0.0, 1.0)), 4)):
        with product.Context(0) as ctx:
            ctx.upload_scene(*scene)
            for mode in (0, 1):
                ctx.set_option(product.capi.OPT_RENDER_MODE, mode)
                _compare(ctx, scene, 161, 121, (1, 2, 3), bounces, 1, what="%s mode %d" % (name, mode), **cam)


def test_device_built_and_refitted_scene(product, tmp_scene_dir):
    import torch
    from test_gpu_device_refit import _dev, _device_build, _load, _refit_device, _to_loader
    from test_gpu_round2 import _deform
    lt, mats = _load(product, tmp_scene_dir, "exact_dev.obj", *scenes.displaced_sphere(4))
    with product.Context(0) as ctx:
        order, d_order = _device_build(ctx, lt, mats)
        tris, nodes = ctx.read_scene()
        _compare(ctx, (tris, nodes, mats), 129, 97, (1, 2), 4, 1, what="device-built", **CAM_B)
        new = _deform(tris, 1.2, 0.7)
        assert _refit_device(ctx, _dev(_to_loader(new, order)), tris.shape[0], d_order) == 0
        _compare(ctx, (new, ctx.read_nodes(), mats), 129, 97, (1, 2), 4, 2, what="refitted", **CAM_B)
        torch.cuda.synchronize()


def test_device_group(product, cornell_ref):
    if product.device_count() < 2:
        pytest.skip("needs two GPUs")
    t2, m2 = _material_sweep(cornell_ref[2], cornell_ref[0], np.random.default_rng(19))
    scene = (t2, cornell_ref[1], m2)
    with product.Context([0, 1]) as grp:
        grp.upload_scene(*scene)
        _compare(grp, scene, 161, 99, (1, 2, 3), 5, 1, what="device group")
