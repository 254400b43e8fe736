"""Argument checks of the strip cluster labelling (include/spgg.h: spgg_strip_clusters) that need no GPU."""
import ctypes as C

import numpy as np
import pytest


def test_strip_cluster_entry_points_reject_a_null_handle_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    rec = np.zeros(64, np.uint8)
    n, first, total = C.c_int64(-7), C.c_int64(-7), C.c_int64(-7)
    for rc in (lib.spgg_strip_cluster_record_bytes(None),
               lib.spgg_strip_clusters(None, 0, 0, rec.ctypes.data),
               lib.spgg_strip_clusters_resolve(None, 1, 0, rec.ctypes.data, C.byref(n), C.byref(first),
                                               C.byref(total))):
        assert rc == _lib.E_INVALID
        with pytest.raises(ValueError):
            _lib.check(rc)
    assert n.value == first.value == total.value == -7


def test_strip_engine_checks_of_before_the_library():
    import spgg_b200
    from spgg_b200 import strips
    se = strips.StripEngine.__new__(strips.StripEngine)
    se.lib, se.h, se._open = spgg_b200.load(), C.c_void_p(), 0
    for of in ("X", 2, None, True):
        with pytest.raises(ValueError, match="of must be"):
            se.cluster_sizes(of=of)
        with pytest.raises(ValueError, match="of must be"):
            se.cluster_labels(of=of, periodic=True)
    with pytest.raises(ValueError):      # a valid `of` reaches the library, which refuses the null handle
        se.cluster_sizes(of="D")
