"""Slot release in the ingest id table (rcd_ingest_release, csrc/rcd_ingest.hpp): freed slots are handed to new
vehicle ids lowest first, the id limit counts live ids, and bad calls change nothing.  Host code; no GPU."""
import ctypes

import numpy as np
import pytest

from tests import ingest_cases as C


def _msgs(ids, t=1.0):
    import random
    rng = random.Random(7)
    return "\n".join(C.reference_message(rng, 0, t, vid=v) for v in ids)


def _table(g):
    return {g.id_of(k): k for k in range(g.n_objects) if _live(g, k)}


def _live(g, slot):
    from rcd_b200.host import _native as N
    try:
        g.id_of(slot)
        return True
    except N.NativeError as e:
        assert e.code == N.RCD_EINVAL
        return False


def test_new_ids_take_freed_slots_lowest_first_then_fresh_ones():
    from rcd_b200.host.ingest import VehicleIngest
    with VehicleIngest(threads=1) as g:
        rec, _ = g.decode(_msgs([f"v{k}" for k in range(10)]))
        assert rec["slot"].tolist() == list(range(10))
        assert g.release(np.array([7, 2, 5], np.uint32)) == 7
        assert g.n_objects == 10  # slots handed out: the frame size does not shrink
        # known ids keep their slots; new ids take 2, 5, 7 in arrival order, then fresh slots; a released id comes back anew
        rec, _ = g.decode(_msgs(["v3", "new-a", "v2", "new-b", "v9", "new-c", "new-d", "new-e"]))
        assert rec["slot"].tolist() == [3, 2, 5, 7, 9, 10, 11, 12]
        assert [g.id_of(int(s)) for s in rec["slot"]] == ["v3", "new-a", "v2", "new-b", "v9", "new-c", "new-d", "new-e"]
        assert g.n_objects == 13
        assert g.slot_of("v7") is None and g.slot_of("v5") is None
        assert g.slot_of("v2") == 5


def test_same_batch_repeats_of_a_new_id_share_the_reused_slot():
    from rcd_b200.host.ingest import VehicleIngest
    with VehicleIngest(threads=1) as g:
        g.decode(_msgs(["a", "b", "c"]))
        g.release([1])
        rec, max_seq = g.decode(_msgs(["x", "x", "y"]))
        assert rec["slot"].tolist() == [1, 1, 3] and rec["seq"].tolist() == [0, 1, 0] and max_seq == 1


def test_releasing_k_at_a_full_limit_lets_exactly_k_new_vehicles_in():
    from rcd_b200.host.ingest import VehicleIngest
    with VehicleIngest(threads=1) as g:
        g.set_limit(8)
        rec, _ = g.decode(_msgs([f"v{k}" for k in range(8)]))
        assert len(rec) == 8 and g.rejected == 0
        rec, _ = g.decode(_msgs(["late"]))
        assert len(rec) == 0 and g.rejected == 1
        assert g.release([0, 6, 3]) == 5
        rec, _ = g.decode(_msgs(["n1", "n2", "n3", "n4", "v1"]))
        assert sorted(rec["slot"].tolist()) == [0, 1, 3, 6]  # n4 is rejected, known v1 is served
        assert g.slot_of("n4") is None and g.rejected == 2
        assert g.n_objects == 8  # the frame never grows past the limit


def test_bad_release_returns_einval_and_changes_nothing():
    from rcd_b200.host import _native as N
    from rcd_b200.host.ingest import VehicleIngest
    with VehicleIngest(threads=1) as g:
        g.decode(_msgs([f"v{k}" for k in range(6)]))
        assert g.release([4]) == 5
        before = (_table(g), g.n_objects)
        for bad in ([4], [1, 4], [6], [1, 100], [2, 2], [1, 3, 1]):  # free, free, out of range, out of range, repeats
            with pytest.raises(N.NativeError) as e:
                g.release(np.array(bad, np.uint32))
            assert e.value.code == N.RCD_EINVAL
            assert (_table(g), g.n_objects) == before
        # lookup of a released id: RCD_ESTATE; id_name of a free slot: RCD_EINVAL
        lib = N.load()
        s = ctypes.c_uint32()
        assert lib.rcd_ingest_lookup(g._g, b"v4", 2, ctypes.byref(s)) == N.RCD_ESTATE
        p, ln = ctypes.c_char_p(), ctypes.c_uint32()
        assert lib.rcd_ingest_id_name(g._g, 4, ctypes.byref(p), ctypes.byref(ln)) == N.RCD_EINVAL
        assert lib.rcd_ingest_id_name(g._g, 3, ctypes.byref(p), ctypes.byref(ln)) == N.RCD_OK
        # an empty release is fine and reports the live count
        live = ctypes.c_uint64()
        assert lib.rcd_ingest_release(g._g, 0, None, ctypes.byref(live)) == N.RCD_OK and live.value == 5
