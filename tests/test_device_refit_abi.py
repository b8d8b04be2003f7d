"""b2rt_refit_scene_device without a CUDA device: it fails loudly, there is no host fallback."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_product


def test_device_refit_fails_without_a_gpu():
    prod = load_product()
    if prod.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(prod.B2RTError) as e:
        prod.Context(0)
    assert e.value.status == -1                                          # CL_DEVICE_NOT_FOUND
    L = prod.lib()
    tris = np.zeros((4, 256), dtype=np.uint8)
    status = np.zeros(1, dtype=np.uint32)
    st = L.b2rt_refit_scene_device(None, ctypes.c_void_p(tris.ctypes.data), 4, None, ctypes.c_void_p(status.ctypes.data), None)
    assert st == -34                                                     # CL_INVALID_CONTEXT
    assert status[0] == 0


def test_status_bits_are_the_header_values():
    with open(os.path.join(ROOT, "include", "b2rt.h")) as f:
        header = dict((k, int(v)) for k, v in re.findall(r"\bB2RT_REFIT_([A-Z_]+)\s*=\s*(\d+)", f.read()))
    cap = load_product().capi
    assert header == {k: getattr(cap, "REFIT_" + k) for k in ("NONFINITE", "DUPLICATE", "RANGE", "LEAF_BOX", "ORDER")}
    assert header == {"NONFINITE": 1, "DUPLICATE": 2, "RANGE": 4, "LEAF_BOX": 8, "ORDER": 16}
