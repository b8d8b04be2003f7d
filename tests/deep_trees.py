"""Deep BVHs for the traversal tests (numpy + the product's OBJ loader).

Every traversal kernel sizes its stack from the tree: 32, 64, 128 or 256 entries (pick_cap, csrc/kernels.cu), a
tail-kernel frontier of max(256, 4 (bound + 8)) words and a tail record of bound + 8 stack words. The scenes the other
tests use are shallow (stack bound <= 43), so these helpers build trees of a known, exact depth:

  chain(D)        D + 1 loader pairs hung off a spine: binary depth D, stack bound D + 1
  spine(D, s)     the same spine with a balanced subtree of s leaves at every level (wide frontiers)
  geometric(K)    K faces in geometric progression through the loader and the SAH builder: deep without a caller tree

The caller-built trees are CLLinearBVHNode arrays in pre-order with exact union boxes, uploaded as they are
(b2rt_upload_scene takes caller-supplied trees)."""
import os

import numpy as np

import scenes

# the triangle of face k of a chain: (x_k, 0, 0) (x_k + .8, 0, 0) (x_k, .8, .3), i.e. the plane z = 0.375 y, front
# faces for rays going down in z
_EDGE_X, _EDGE_Y, _EDGE_Z = 0.8, 0.8, 0.3


def _loader_faces(host, path, xs):
    """One small triangle per x in `xs`, written as an OBJ and read by the product's loader: every face becomes the
    loader's duplicated pair. Returns (tris, mats, positions (2 len(xs), 3, 3))."""
    p = np.zeros((len(xs), 3, 3))
    p[:, :, 0] = np.asarray(xs, dtype=np.float64)[:, None]
    p[:, 1, 0] += _EDGE_X
    p[:, 2, 1], p[:, 2, 2] = _EDGE_Y, _EDGE_Z
    p = p.reshape(-1, 3).astype(np.float32)
    nrm = np.tile(np.array([[0.0, -0.35, 0.94]], dtype=np.float32), (p.shape[0], 1))
    scenes.write_obj(path, p, nrm, np.arange(p.shape[0]).reshape(-1, 3))
    tris, mats = host.load_triangles(path)
    assert tris.shape[0] == 2 * len(xs)                        # every face is one duplicated pair, in file order
    pos = tris.view(np.float32).reshape(-1, 64)[:, [0, 1, 2, 20, 21, 22, 40, 41, 42]].reshape(-1, 3, 3)
    return tris, mats, pos


def _nodes(records):
    """records: pre-order list of (lo, hi, offset, n_prims, axis) -> (n, 48) uint8 CLLinearBVHNode array."""
    nodes = np.zeros((len(records), 48), dtype=np.uint8)
    f = nodes.view(np.float32).reshape(-1, 12)
    u = nodes.view(np.uint32).reshape(-1, 12)
    h = nodes.view(np.uint16).reshape(-1, 24)
    for i, (lo, hi, off, n_prims, axis) in enumerate(records):
        f[i, 0:3], f[i, 4:7] = lo, hi
        u[i, 8] = off
        h[i, 18] = n_prims
        nodes[i, 38] = axis
    return nodes


def _spine_tree(pos, depth, side, axes):
    """Pre-order records of a spine of `depth` interior levels: level j's first child is a balanced subtree over leaves
    [j side, (j + 1) side), its second child is level j + 1; the spine ends in leaf depth * side. Leaf k holds the
    loader pair 2k, 2k + 1. Level j's split axis is axes[j % len(axes)]; subtree nodes split on x."""
    recs = []

    def leaf(k):
        p = pos[2 * k:2 * k + 2].reshape(-1, 3)
        recs.append((p.min(0), p.max(0), 2 * k, 2, 0))
        return len(recs) - 1

    def balanced(lo, hi):
        if hi - lo == 1:
            return leaf(lo)
        i = len(recs)
        recs.append(None)
        a = balanced(lo, (lo + hi) // 2)
        b = balanced((lo + hi) // 2, hi)
        recs[i] = (np.minimum(recs[a][0], recs[b][0]), np.maximum(recs[a][1], recs[b][1]), b, 0, 0)
        return i

    # the spine in a loop (no recursion as deep as the tree): level j, then its subtree, then level j + 1
    levels = []
    for j in range(depth):
        levels.append(len(recs))
        recs.append(None)
        balanced(j * side, (j + 1) * side)
    levels.append(leaf(depth * side))
    for j in range(depth - 1, -1, -1):
        i, a, b = levels[j], levels[j] + 1, levels[j + 1]
        recs[i] = (np.minimum(recs[a][0], recs[b][0]), np.maximum(recs[a][1], recs[b][1]), b, 0, axes[j % len(axes)])
    return _nodes(recs)


def chain(host, directory, depth, axes=(0,), direction=1):
    """Chain tree of binary depth `depth` (stack bound depth + 1): faces at x = direction * k, k = 0 .. depth; interior
    node 2j has leaf j at 2j + 1 as its first child and the rest of the chain at 2j + 2 as its second. Returns
    (tris, nodes, mats)."""
    path = os.path.join(directory, "chain%d_%s_%d.obj" % (depth, "".join(map(str, axes)), direction))
    tris, mats, pos = _loader_faces(host, path, direction * np.arange(depth + 1))
    return tris, _spine_tree(pos, depth, 1, axes), mats


def spine(host, directory, depth, side, axes=(0,)):
    """Spine of `depth` levels with a balanced subtree of `side` leaves (a power of two) at each: faces at x = k,
    k = 0 .. depth * side. Returns (tris, nodes, mats)."""
    path = os.path.join(directory, "spine%d_%d.obj" % (depth, side))
    tris, mats, pos = _loader_faces(host, path, np.arange(depth * side + 1))
    return tris, _spine_tree(pos, depth, side, axes), mats


def grazing_rays(n_faces, n, seed, direction=1, y_jitter=0.0):
    """Rays along a row of chain faces (x = direction * k, k < n_faces), half from beyond each end. Each is aimed at a
    point of a random face k and descends so gently that it passes over every face in front of k while it stays
    inside every box: the walk has to go through the whole row. y_jitter > 0 tilts the rays sideways (either sign),
    which changes the visiting order at nodes that split on y."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, n_faces, n)
    ty = 0.267 + rng.normal(0.0, 0.02, n)
    tgt = np.stack([direction * k + 0.267 + rng.normal(0.0, 0.02, n), ty, 0.375 * ty], 1)
    far = direction * (n_faces + 4.0)
    near = -direction * 5.0
    o = np.stack([np.where(np.arange(n) % 2 == 0, far, near), ty + rng.normal(0.0, y_jitter, n) if y_jitter else ty,
                  np.full(n, 0.29)], 1)
    return scenes.pack_rays(o, tgt - o)


def chain_rays(n_faces, n, seed, direction=1):
    """Grazing rays (straight and tilted), rays from anywhere around the row, and a share cut short by tmax."""
    lo = np.array([min(0.0, direction * n_faces) - 2.0, -1.0, -1.0])
    hi = np.array([max(0.0, direction * n_faces) + 2.0, 2.0, 2.0])
    rays = np.concatenate([grazing_rays(n_faces, n // 2, seed, direction), grazing_rays(n_faces, n // 4, seed + 1, direction, 0.003),
                           scenes.box_rays(n - n // 2 - n // 4, lo, hi, seed=seed + 2)])
    rays["tmax"][::7] = np.random.default_rng(seed + 3).uniform(0.5, n_faces + 8.0, rays["tmax"][::7].shape).astype(np.float32)
    return rays


def geometric_positions(count=600, ratio=1.1):
    """Face k: a right triangle of legs 0.3 s_k at distance ~s_k from the origin, s_k = ratio^k, on axis k mod 3 (with
    half of that on the next axis). Every face is a step further out than all before it, so a SAH builder nests them."""
    s = ratio ** np.arange(count)
    p = np.zeros((count, 3, 3))
    for k in range(count):
        c = np.zeros(3)
        c[k % 3], c[(k + 1) % 3] = s[k], 0.5 * s[k]
        p[k] = [c, c + [0.3 * s[k], 0.0, 0.0], c + [0.0, 0.3 * s[k], 0.0]]
    return p.astype(np.float32)


def geometric(host, directory, count=600, ratio=1.1):
    """The geometric-progression OBJ through the product's loader and SAH builder (4 primitives per leaf). Returns
    (tris, nodes, mats, positions (count, 3, 3))."""
    p = geometric_positions(count, ratio)
    nrm = np.tile(np.array([[0.0, 0.0, 1.0]], dtype=np.float32), (3 * count, 1))
    path = scenes.write_obj(os.path.join(directory, "geometric%d.obj" % count), p.reshape(-1, 3), nrm, np.arange(3 * count).reshape(count, 3))
    tris, nodes, mats = host.load_scene(path, 4)
    return tris, nodes, mats, p


def geometric_rays(p, n, seed):
    """Rays at the centroids of random faces of every scale, half from the far side of the origin and half from
    further out than the face. The scene spans ~1e25, so tmax is unlimited except on every fifth ray, which stops
    between 0.3 and 1.2 times the distance to its target."""
    rng = np.random.default_rng(seed)
    tgt = p[rng.integers(0, p.shape[0], n)].mean(1).astype(np.float64)
    half = n // 2
    o = np.concatenate([-0.5 * np.abs(tgt[:half]).max(1, keepdims=True) * np.ones((1, 3)), 3.0 * tgt[half:] + 1.0])
    rays = scenes.pack_rays(o, tgt - o, np.finfo(np.float32).max)
    dist = np.linalg.norm(tgt - o, axis=1)[::5]
    rays["tmax"][::5] = (dist * rng.uniform(0.3, 1.2, dist.shape)).astype(np.float32)
    return rays
