"""rcd_reserve and rcd_alerts_reserve refuse a NULL handle with a return code (no device needed)."""


def test_reserve_calls_refuse_a_null_handle():
    from rcd_b200.host import _native as N
    lib = N.load()
    assert lib.rcd_reserve(None, 1 << 20, 1 << 20) == N.RCD_EINVAL
    assert lib.rcd_alerts_reserve(None, 1 << 20) == N.RCD_EINVAL
