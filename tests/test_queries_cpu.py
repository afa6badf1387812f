"""rcd_set_queries without a GPU: a call on a NULL handle is refused, whatever the list."""
import numpy as np


def test_set_queries_on_a_null_handle_is_einval():
    from rcd_b200.host import _native as N
    lib = N.load()
    slots = np.arange(4, dtype=np.uint32)
    assert lib.rcd_set_queries(None, 4, slots.ctypes.data, N.SRC_HOST) == N.RCD_EINVAL
    assert lib.rcd_set_queries(None, 0, None, N.SRC_HOST) == N.RCD_EINVAL
    assert lib.rcd_set_queries(None, 4, slots.ctypes.data, N.SRC_DEVICE) == N.RCD_EINVAL
