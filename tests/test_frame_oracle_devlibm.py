"""The fp64-libm oracle (tests/frame_oracle/oracle_devlibm.c), which the GPU frames are held to bit for bit, tied to the
glibc oracle that is pinned against the reference build (tests/test_oracle.py): it is the same C with powf / sinf / cosf
evaluated in fp64 and rounded once, so it may differ only where glibc's float functions round the other way -- by a few
ulp on a few pixels, with no path taking another branch."""
import ctypes as C

import numpy as np

import frame_oracle_lib as fl
import oracle_lib as ol

F32 = np.float32


def ordered(x):
    """float32 -> int64 on which the distance of two values is their distance in ulp (-0 and +0 coincide)."""
    b = np.asarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.where(b < 0, -(b & 0x7FFFFFFF), b)


def ulp_diff(a, b):
    return np.abs(ordered(a) - ordered(b))


def glibc_powf(a, b):
    libm = C.CDLL("libm.so.6")
    libm.powf.argtypes = [C.c_float, C.c_float]
    libm.powf.restype = C.c_float
    return np.array([libm.powf(float(x), float(y)) for x, y in zip(a, b)], dtype=np.float32)


# bases the frame kernels pass to pow_cr (rnd() in [0, 1], pixel values >= 0 or NaN, squares of any sign), crossed with
# the exponents they use (2, 2.2, 0.4545.., 1/(alpha+1) of any value including 0, +-inf and NaN)
SPECIAL_BASES = [0.0, 1e-45, 1.1754942e-38, 1e-30, 0.25, 0.5, 1 - 2.0 ** -24, 1.0, 1 + 2.0 ** -23, 2.0, 1e30, 3.4028235e38,
                 np.inf, np.nan]
SPECIAL_EXPONENTS = [0.0, -0.0, 2.0, 2.2, 0.45454545, 0.454545, 1.0, -1.0, 0.5, 1e-30, -1e-30, 40.0, -40.0, 3e38, -3e38,
                     np.inf, -np.inf, np.nan]
SQUARE_BASES = [-0.0, -1e-45, -0.5, -1.0, -3.0, -1e20, -np.inf]


def special_pow_table():
    a = [x for x in SPECIAL_BASES for _ in SPECIAL_EXPONENTS] + SQUARE_BASES
    b = [y for _ in SPECIAL_BASES for y in SPECIAL_EXPONENTS] + [2.0] * len(SQUARE_BASES)
    return np.array(a, dtype=np.float32), np.array(b, dtype=np.float32)


def pow_records(a, b):
    rec = fl.records(a.shape[0])
    rec.view(np.float32)[:, 0], rec.view(np.float32)[:, 1] = a, b
    return rec


def check_against_powf(got, a, b):
    """Results glibc gives as 0, 1, inf or NaN must be exactly that; all others within 1 ulp of glibc."""
    want = glibc_powf(a, b)
    special = np.isnan(want) | np.isinf(want) | (want == 0) | (want == 1)
    same = (got == want) | (np.isnan(got) & np.isnan(want))
    bad = np.flatnonzero(special & ~same)
    assert bad.size == 0, ["pow(%r, %r) = %r, powf gives %r" % (a[i], b[i], got[i], want[i]) for i in bad]
    assert not np.isnan(got[~special]).any()
    assert ulp_diff(got[~special], want[~special]).max(initial=0) <= 1


def test_variant_pow_special_values_follow_glibc_powf():
    a, b = special_pow_table()
    got = fl.oracle_run(fl.OP_POW, pow_records(a, b))[:, 0].view(np.float32)
    check_against_powf(got, a, b)
    assert (got[(b == 0) | (a == 1)] == 1).all()


def test_variant_differs_from_glibc_oracle_by_a_few_ulp(cornell_ref):
    """Cornell at 256^2, 4 bounces, frames 1-3, light types 0/1/2 (and 9 bounces at frame 0): measured at most 3 ulp on
    0.17-0.42 % of the pixels (bound asserted: 4 ulp, 1 %); a path taking another branch would differ far more."""
    tris, nodes, mats = cornell_ref
    W = H = 256
    for lt, frames, bounces in ((0, (1, 2, 3), 4), (1, (1, 2, 3), 4), (2, (1, 2, 3), 4), (0, (0,), 9)):
        glibc = np.zeros((W * H, 4), dtype=np.float32)
        fp64 = np.zeros((W * H, 4), dtype=np.float32)
        for fc in frames:
            ol.oracle_render(tris, nodes, mats, glibc, W, H, fc, bounces, light_type=lt)
            fl.oracle_render(tris, nodes, mats, fp64, W, H, fc, bounces, light_type=lt)
        assert np.array_equal(np.isnan(glibc), np.isnan(fp64)), lt
        d = ulp_diff(np.nan_to_num(glibc), np.nan_to_num(fp64))
        differ = (d != 0).any(axis=1)
        assert d.max() <= 4, (lt, int(d.max()))
        assert 0 < differ.mean() < 0.01, (lt, differ.mean())
