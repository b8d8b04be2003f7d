"""numpy views of the reference's POD layouts (CLshared_structs.hpp:13-88) and of the
ray-stream records of include/b2rt.h. Sizes/offsets: SURVEY.md 8a."""
import numpy as np

TRI_BYTES, NODE_BYTES, MAT_BYTES = 256, 48, 64

RAY_DTYPE = np.dtype([("ox", "<f4"), ("oy", "<f4"), ("oz", "<f4"), ("tmin", "<f4"),
                      ("dx", "<f4"), ("dy", "<f4"), ("dz", "<f4"), ("tmax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("tri", "<u4")])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 16
# b2rt_closest_point records: a query point with its search radius squared, and the nearest surface point found
POINT_QUERY_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("max_d2", "<f4")])
POINT_HIT_DTYPE = np.dtype([("d2", "<f4"), ("u", "<f4"), ("v", "<f4"), ("tri", "<u4")])
assert POINT_QUERY_DTYPE.itemsize == 16 and POINT_HIT_DTYPE.itemsize == 16
# b2rt_trace_radiance record: the path's radiance and the RNG state after it
RADIANCE_DTYPE = np.dtype([("r", "<f4"), ("g", "<f4"), ("b", "<f4"), ("seed", "<u4")])
assert RADIANCE_DTYPE.itemsize == 16

# CLLinearBVHNode, 48 B
NODE_DTYPE = np.dtype({"names": ["bmin", "bmax", "offset", "nPrimitives", "axis"],
                       "formats": [("<f4", 3), ("<f4", 3), "<u4", "<u2", "u1"],
                       "offsets": [0, 16, 32, 36, 38], "itemsize": NODE_BYTES})
# CLTriangle, 256 B: three 80-byte CLVertex {position, uv, normal, tangent_s, tangent_t} + mtlIndex
TRI_DTYPE = np.dtype({"names": ["p1", "uv1", "n1", "p2", "uv2", "n2", "p3", "uv3", "n3", "mtlIndex"],
                      "formats": [("<f4", 3)] * 9 + ["<u4"],
                      "offsets": [0, 16, 32, 80, 96, 112, 160, 176, 192, 240], "itemsize": TRI_BYTES})
# CLMaterial, 64 B
MAT_DTYPE = np.dtype({"names": ["diffuse", "specular", "emission", "type", "roughness", "ior"],
                      "formats": [("<f4", 3), ("<f4", 3), ("<f4", 3), "<u4", "<f4", "<f4"],
                      "offsets": [0, 16, 32, 48, 52, 56], "itemsize": MAT_BYTES})


def make_rays(origins, dirs, tmax=100000.0):
    """Pack (n,3) origins and directions into b2rt_ray records."""
    o = np.asarray(origins, dtype=np.float32)
    d = np.asarray(dirs, dtype=np.float32)
    r = np.zeros(o.shape[0], dtype=RAY_DTYPE)
    r["ox"], r["oy"], r["oz"] = o[:, 0], o[:, 1], o[:, 2]
    r["dx"], r["dy"], r["dz"] = d[:, 0], d[:, 1], d[:, 2]
    r["tmax"] = tmax
    return r
