"""The product's host mirror (CLOBJloader + CLBVHScene in host/*.cpp, written from scratch) must
produce the SAME triangle order and node array as the reference's own loader + builder (oracle/_ref,
compiled verbatim), because hit IDs are indices into that array (SURVEY.md 8 a10, Appendix A-14).
cornell.obj is checked against the reference's arrays stored in tests/golden/cornell_scene.npz; other
scenes need oracle/_ref, and where that build is missing the tests check everything else they cover."""
import os

import numpy as np
import pytest

import oracle_lib as ol
import scenes
from conftest import load_product

needs_ref = pytest.mark.skipif(ol.ref() is None, reason="oracle/_ref not built")

TRI_FLOATS = [0, 1, 2, 4, 5, 6, 8, 9, 10, 20, 21, 22, 24, 25, 26, 28, 29, 30, 40, 41, 42, 44, 45, 46, 48, 49, 50]
GOLDEN_TRI_FLOATS = [0, 1, 2, 4, 5, 8, 9, 10, 20, 21, 22, 24, 25, 28, 29, 30, 40, 41, 42, 44, 45, 48, 49, 50]   # tests/golden/make_golden.py
GOLDEN_MAT_FLOATS = [0, 1, 2, 4, 5, 6, 8, 9, 10, 13, 14]


def _same_scene(a, b):
    (ta, na, ma), (tb, nb, mb) = a, b
    assert ta.shape == tb.shape and na.shape == nb.shape and ma.shape == mb.shape
    fa, fb = ta.view(np.float32).reshape(-1, 64), tb.view(np.float32).reshape(-1, 64)
    assert np.array_equal(fa[:, TRI_FLOATS].view(np.uint32), fb[:, TRI_FLOATS].view(np.uint32))     # positions, uvs, normals
    assert np.array_equal(ta.view(np.uint32).reshape(-1, 64)[:, 60], tb.view(np.uint32).reshape(-1, 64)[:, 60])   # mtlIndex
    ba, bb = na.view(np.float32).reshape(-1, 12), nb.view(np.float32).reshape(-1, 12)
    assert np.array_equal(ba[:, [0, 1, 2, 4, 5, 6]].view(np.uint32), bb[:, [0, 1, 2, 4, 5, 6]].view(np.uint32))
    assert np.array_equal(na.view(np.uint32).reshape(-1, 12)[:, 8], nb.view(np.uint32).reshape(-1, 12)[:, 8])      # offset
    pa, pb = na.view(np.uint16).reshape(-1, 24)[:, 18], nb.view(np.uint16).reshape(-1, 24)[:, 18]
    assert np.array_equal(pa, pb)                                                                                     # nPrimitives
    interior = pa == 0
    assert np.array_equal(na[interior, 38], nb[interior, 38])                                                        # axis (garbage in leaves)
    fm, gm = ma.view(np.float32).reshape(-1, 16), mb.view(np.float32).reshape(-1, 16)
    assert np.array_equal(fm[:, [0, 1, 2, 4, 5, 6, 8, 9, 10, 13, 14]].view(np.uint32), gm[:, [0, 1, 2, 4, 5, 6, 8, 9, 10, 13, 14]].view(np.uint32))


def test_cornell_matches_reference_and_golden(cornell_ref):
    prod = load_product()
    mine = prod.host.load_scene(scenes.CORNELL, 4)
    _same_scene(mine, cornell_ref)
    g = np.load(os.path.join(scenes.GOLDEN, "cornell_scene.npz"))     # written by the reference's own loader + builder
    tris, nodes, mats = mine
    assert np.array_equal(nodes.view(np.uint32).reshape(-1, 12)[:, 8], g["node_offset"])
    assert np.array_equal(tris.view(np.uint32).reshape(-1, 64)[:, 60], g["tri_mtl"])
    assert np.array_equal(tris.view(np.float32).reshape(-1, 64)[:, GOLDEN_TRI_FLOATS].view(np.uint32), g["tri_floats"].view(np.uint32))
    assert np.array_equal(nodes.view(np.float32).reshape(-1, 12)[:, [0, 1, 2, 4, 5, 6]].view(np.uint32), g["node_bounds"].view(np.uint32))
    nprims = nodes.view(np.uint16).reshape(-1, 24)[:, 18]
    assert np.array_equal(nprims, g["node_nprims"])
    assert np.array_equal(np.where(nprims == 0, nodes[:, 38], 255), g["node_axis"])                                  # axis (garbage in leaves)
    assert np.array_equal(mats.view(np.float32).reshape(-1, 16)[:, GOLDEN_MAT_FLOATS].view(np.uint32), g["mat_floats"].view(np.uint32))


@needs_ref
@pytest.mark.parametrize("max_prims", [1, 4, 16])
def test_bumpy_sphere_matches_reference(tmp_scene_dir, max_prims):
    prod = load_product()
    p, n, f = scenes.displaced_sphere(4, amplitude=0.3)
    quads = np.array([[0, 1, 2, 3], [10, 11, 12, 13]])
    path = scenes.write_obj(os.path.join(tmp_scene_dir, "hs%d.obj" % max_prims), p, n, f, quads)
    _same_scene(prod.host.load_scene(path, max_prims), ol.ref_load_scene(path, max_prims))


def test_scattered_and_generated_scenes_match_reference(tmp_scene_dir):
    prod = load_product()
    path = os.path.join(tmp_scene_dir, "scatter.obj")
    assert prod.host.write_scattered_obj(path, 20000, seed=3) == 20000
    a = prod.host.load_scene(path, 4)
    assert a[0].shape[0] == 40000
    if ol.ref() is not None:
        _same_scene(a, ol.ref_load_scene(path, 4))
    path = os.path.join(tmp_scene_dir, "geo.obj")
    assert prod.host.write_icosphere_obj(path, 24, amplitude=0.1) == 20 * 24 * 24
    a = prod.host.load_scene(path, 4)
    if ol.ref() is not None:
        _same_scene(a, ol.ref_load_scene(path, 4))
    # closed, outward-facing mesh: every outside-in ray hits a front face
    rays = scenes.shell_rays(4000, 8.0, seed=9)
    h = ol.oracle_closest(a[0], a[1], rays)
    assert (h["tri"] != 0xFFFFFFFF).mean() > 0.99
    # paths longer than the reference loader's 80-byte buffer are written and read like any other
    deep = os.path.join(tmp_scene_dir, "d" * 80)
    os.makedirs(deep, exist_ok=True)
    for name, write in (("s.obj", lambda p: prod.host.write_scattered_obj(p, 100, seed=3)), ("g.obj", lambda p: prod.host.write_icosphere_obj(p, 2))):
        assert write(os.path.join(deep, name)) > 0
        assert prod.host.load_scene(os.path.join(deep, name), 4)[0].shape[0] > 0


def test_loader_quirks(tmp_scene_dir):
    """Comment words, unknown usemtl, ignored one-character tokens, malformed faces."""
    prod = load_product()
    base = os.path.join(tmp_scene_dir, "quirk")
    with open(base + ".mtl", "w") as f:
        f.write("# comment\nnewmtl a\n# Kd 9 9 9 (comment words are parsed like statements)\nKd 1 0 0\nNs 10\nnewmtl b\nKe 2 2 2\nNi 1.5\n")
    with open(base + ".obj", "w") as f:
        f.write("# a comment\nmtllib quirk.mtl\no thing\nv 0 0 0\nv 1 0 0\nv 0 1 0\nv 1 1 0\nvt 0 0\nvn 0 0 1\ns off\n"
                "usemtl b\nf 1/1/1 2/1/1 3/1/1 \nusemtl nosuch\nf 2/1/1 4/1/1 3/1/1\n")
    mine = prod.host.load_scene(base + ".obj", 4)
    if ol.ref() is not None:
        _same_scene(mine, ol.ref_load_scene(base + ".obj", 4))
    assert mine[0].shape[0] == 4 and set(mine[0].view(np.uint32).reshape(-1, 64)[:, 60]) == {1}
    with open(base + "2.mtl", "w") as f:
        f.write("newmtl a\n")
    with open(base + "2.obj", "w") as f:
        f.write("v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvn 0 0 1\nf 1 2 3\n")      # no v/vt/vn triplets
    with pytest.raises(prod.host.HostError):
        prod.host.load_scene(base + "2.obj", 4)                                  # one-character tokens are ignored -> no faces
    with open(base + "3.obj", "w") as f:
        f.write("v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvn 0 0 1\nf 1//1 2//1 9//1\n")
    with open(base + "3.mtl", "w") as f:
        f.write("newmtl a\n")
    with pytest.raises(prod.host.HostError):
        prod.host.load_scene(base + "3.obj", 4)                                  # the reference reads out of bounds here
    with pytest.raises(prod.host.HostError):
        prod.host.load_scene(os.path.join(tmp_scene_dir, "missing.obj"), 4)


def test_scene_cache_round_trip_and_invalidation(tmp_scene_dir):
    """SURVEY.md 8f-3: the binary cache must return byte-identical arrays (same triangle order = same hit IDs) and must
    be ignored when the source, maxPrimitivesInNode or the file itself changed."""
    import time
    prod = load_product()
    p, n, f = scenes.displaced_sphere(4, amplitude=0.3)
    path = scenes.write_obj(os.path.join(tmp_scene_dir, "cache.obj"), p, n, f)
    plain = prod.host.load_scene(path, 4)
    t1, n1, m1, hit = prod.host.load_scene(path, 4, cache=True)
    assert not hit and os.path.exists(path + ".p4.b2rtscn")
    t2, n2, m2, hit = prod.host.load_scene(path, 4, cache=True)
    assert hit
    for a, b in ((plain[0], t2), (plain[1], n2), (plain[2], m2), (t1, t2), (n1, n2)):
        assert np.array_equal(a, b)                                        # whole records, padding included
    if ol.ref() is not None:
        _same_scene((t2, n2, m2), ol.ref_load_scene(path, 4))
    # another maxPrimitivesInNode is another cache file; an explicit cache path works too
    assert not prod.host.load_scene(path, 2, cache=True)[3]
    other = os.path.join(tmp_scene_dir, "elsewhere.bin")
    assert not prod.host.load_scene(path, 4, cache=other)[3]
    assert prod.host.load_scene(path, 4, cache=other)[3]
    # corrupt payload -> checksum mismatch -> miss (and the cache is rewritten)
    with open(other, "r+b") as fh:
        fh.seek(4096)
        fh.write(b"\xff\xff\xff\xff")
    assert not prod.host.load_scene(path, 4, cache=other)[3]
    assert prod.host.load_scene(path, 4, cache=other)[3]
    # truncated file -> miss
    with open(other, "r+b") as fh:
        fh.truncate(os.path.getsize(other) - 16)
    assert not prod.host.load_scene(path, 4, cache=other)[3]
    # the source changes (new mtime) -> stale -> miss, and the new content is what comes back
    time.sleep(0.01)
    p2 = p * np.float32(1.5)
    scenes.write_obj(path, p2, n, f)
    t3, n3, m3, hit = prod.host.load_scene(path, 4, cache=True)
    assert not hit and not np.array_equal(t3, t2)
    assert prod.host.load_scene(path, 4, cache=True)[3]


def test_parallel_build_is_identical_to_the_reference_build(tmp_scene_dir, monkeypatch):
    """Scenes of >= 65536 triangles are built by a team of threads (host/scene_build.cpp); topology, node numbering and
    the triangle order (= hit IDs) must not depend on the thread count and must equal the reference's recursion
    (without oracle/_ref: the one-thread build, which runs that recursion alone)."""
    prod = load_product()

    def reference(path, max_prims):
        if ol.ref() is not None:
            return ol.ref_load_scene(path, max_prims)
        monkeypatch.setenv("B2RT_BUILD_THREADS", "1")
        return prod.host.load_scene(path, max_prims)
    path = os.path.join(tmp_scene_dir, "par.obj")
    assert prod.host.write_scattered_obj(path, 50000, extent=30.0, edge_min=0.2, edge_max=1.0, seed=9) == 50000
    want = reference(path, 4)
    assert want[0].shape[0] == 100000
    for threads in ("1", "3", "8"):
        monkeypatch.setenv("B2RT_BUILD_THREADS", threads)
        got = prod.host.load_scene(path, 4)
        _same_scene(got, want)
    p, n, f = scenes.displaced_sphere(6, amplitude=0.2)          # 81920 faces -> 163840 triangles, shared vertices
    path = scenes.write_obj(os.path.join(tmp_scene_dir, "par_sphere.obj"), p, n, f)
    want = reference(path, 2)
    monkeypatch.setenv("B2RT_BUILD_THREADS", "5")
    _same_scene(prod.host.load_scene(path, 2), want)


def test_number_parsing_equals_strtof():
    """The loader's decimal fast path must return bit-for-bit what strtof (the engine behind the reference's
    fscanf("%f"), CLOBJloader.cpp:47-62) returns, including float rounding boundaries, long digit strings, exponents,
    signs, leading zeros, hex floats and inf/nan."""
    import ctypes
    prod = load_product()
    libc = ctypes.CDLL("libc.so.6")
    libc.strtof.restype = ctypes.c_float
    libc.strtof.argtypes = [ctypes.c_char_p, ctypes.c_void_p]
    rng = np.random.default_rng(123)
    words = ["0", "-0", "+0.0", "1", "-1.5", ".5", "-.25", "5.", "1e5", "1E-5", "1.25e+3", "007.500", "0.000001", "123456.789",
             "16777217", "16777216.5", "0.1", "0.3", "1e22", "1e23", "1e-22", "1e-45", "3.4028235e38", "3.5e38", "1e-38", "1.17549435e-38",
             "0x10", "0x1.8p1", "inf", "-inf", "nan", "1e", "2e+", "3.e2", "123456789012345", "1234567890123456", "0.1234567890123456789",
             "8388608.5", "8388609.5", "4194304.25", "1.00000005960464477539", "1.000000059604644775390625", "0.50000002980232238769531250"]
    for _ in range(60000):
        kind = rng.integers(0, 5)
        if kind == 0:
            words.append("%.6f" % rng.uniform(-100, 100))
        elif kind == 1:
            words.append(repr(float(np.float32(rng.standard_normal() * 10.0 ** int(rng.integers(-6, 7))))))
        elif kind == 2:
            words.append("%.*e" % (int(rng.integers(0, 17)), rng.standard_normal() * 10.0 ** int(rng.integers(-20, 21))))
        elif kind == 3:                                          # exact float midpoints and their neighbours, printed in full
            f = np.float32(rng.uniform(0.5, 2.0) * 2.0 ** int(rng.integers(-10, 11)))
            mid = (float(f) + float(np.nextafter(f, np.float32(np.inf)))) / 2.0
            words.append("%.40g" % mid)
            words.append("%.17g" % np.nextafter(mid, np.inf))
        else:
            words.append("%d.%0*d" % (rng.integers(0, 1000), int(rng.integers(1, 12)), rng.integers(0, 10 ** 9)))
    got = ol.parse_numbers(" ".join(w for w in words if w not in ("1e", "2e+")), len(words) + 8)
    want = np.array([libc.strtof(w.encode(), None) for w in words if w not in ("1e", "2e+")], dtype=np.float32)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # a number with a dangling exponent marker stops where strtof stops: "1e" is 1, then the word "e" is not a number
    assert np.array_equal(ol.parse_numbers("1e 7"), np.array([1.0], dtype=np.float32))


def test_face_token_scanner_equals_sscanf():
    """`f` vertices are read with sscanf("%d/%d/%d") by the reference (CLOBJloader.cpp:96); the loader's own scanner must
    give the same three values for well-formed and malformed tokens alike."""
    import ctypes
    prod = load_product()
    libc = ctypes.CDLL("libc.so.6")
    rng = np.random.default_rng(5)
    tokens = ["1/2/3", "12/34/56", "1//3", "1/2", "7", "/2/3", "-1/2/3", "+5/6/7", "1/-2/3", "12abc/3/4", "1/2/3/4", "1/2/3x", "0/0/0",
              "2147483647/1/1", "99999999999/1/1", "1/ 2/3", " 1/2/3", "1 /2/3", "a/b/c", "", "-", "1/", "1/2/", "//", "1/+2/-3", "007/08/09"]
    for _ in range(3000):
        parts = [str(int(rng.integers(-50, 5_000_000))) if rng.random() < 0.9 else "" for _ in range(int(rng.integers(1, 5)))]
        tokens.append("/".join(parts))
    for tok in tokens:
        a, b, c = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
        libc.sscanf(tok.encode(), b"%d/%d/%d", ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        want = tuple(v.value & 0xFFFFFFFF for v in (a, b, c))
        assert ol.scan_triplet(tok) == want, tok
