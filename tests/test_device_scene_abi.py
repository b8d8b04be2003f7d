"""b2rt_build_scene_device without a CUDA device: it fails loudly, there is no host fallback."""
import ctypes

import numpy as np
import pytest

from conftest import load_product


def test_device_scene_build_fails_without_a_gpu():
    prod = load_product()
    if prod.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(prod.B2RTError) as e:
        prod.Context(0)
    assert e.value.status == -1                                          # CL_DEVICE_NOT_FOUND
    L = prod.lib()
    tris = np.zeros((4, 256), dtype=np.uint8)
    out = [ctypes.c_uint64(0) for _ in range(3)]
    st = L.b2rt_build_scene_device(None, ctypes.c_void_p(tris.ctypes.data), 4, None, *[ctypes.byref(o) for o in out], None)
    assert st == -34                                                     # CL_INVALID_CONTEXT
    assert [o.value for o in out] == [0, 0, 0]
