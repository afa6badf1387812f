"""k_narrow runs its per-offset phases on groups of 32 predict pairs gathered over several queue batches.
These frames put the group boundaries where they matter, through the bench's frame variant (fused detect +
predict, no candidate counts, profiling off), and check the records against the CPU oracle.

How the pairs reach the groups:
  * k_pairs appends the survivors of a chunk of 32 neighbours for its 32 queries lane by lane: a query that sees
    all 32 neighbours of a chunk fills a run of 32 queue entries, its own self pair included, and in a tile where
    every query sees the whole chunk these runs line up with the 32-entry batches of k_narrow.
  * A warp of k_narrow takes batches w, w + W, w + 2W, ... with W = 4 * (2 * tiles + 1) warps on frames this
    small, so a warp usually takes several batches of the same tile.  Only pairs whose querying object has a
    history have offsets to look at; in the small frames below that is one object, H.  So the warp that takes
    H's batch holds exactly H's surviving pairs when its batches run out, however many empty batches it took.
"""
import numpy as np
import pytest

from tests.gpu_helpers import compare_pairs
from tests.helpers import f64_frame

pytestmark = pytest.mark.gpu


def _oracle():
    from oracle import oracle as O
    return O


def _check_fused(e, frame, pat, query_stride=None):
    """One fused frame against the oracle (queries i with i % query_stride == 0 only, if given)."""
    from rcd_b200.host import _native as N
    O = _oracle()
    e.upload(frame)
    e.set_patterns(pat)
    e.step(N.MODE_PREDICT, with_detect=True)
    got = e.download()
    c = e.counts()
    assert c["n_fallback"] == 0
    kw = {} if query_stride is None else {"want_potentials": False, "query_stride": query_stride}
    f64 = f64_frame(frame)
    d = O.frame_A(f64, "detect", **kw)["risks"]
    p = O.frame_A(f64, "predict", pattern_codes=pat, **kw)["risks"]
    det = np.sort(np.concatenate([d, p[p["offset"] < 0]]), order=["i", "j"])  # no history: predict falls back to detect
    if query_stride is not None:
        got = got[got["i"] % query_stride == 0]
    else:
        assert c["n_pairs"] == len(det) + (p["offset"] >= 0).sum()
    compare_pairs(got[got["predicted"] == 0], det, "detect")
    compare_pairs(got[got["predicted"] == 1], p[p["offset"] >= 0], "predict")
    return got


def _stack_frame(k):
    """k - 1 stationary objects without history stacked on the z axis (z in [0, 30]) and, last, H: the only object
    with a history, 60 m above them and falling through all of them at 20 m/s.  Every object is within 100 m of
    every other one, so every query sees all k objects; each pair (H, j) has offsets to look at (H passes through
    j), every other pair has none.  In the grid of the bounds below H's cell key is the largest (the z layer is
    the slowest-varying part of the key), so H comes last in cell order."""
    from rcd_b200.host import workloads as W
    f = W.empty_frame(k)
    f["pz"][: k - 1] = np.linspace(0.0, 30.0, k - 1, dtype=np.float32)
    f["pz"][k - 1] = 60.0
    f["vz"][k - 1] = -20.0
    f["size"][:] = 2.0
    f["type"][:] = 4
    pat = np.full(k, 3, np.uint8)  # RCD_PAT_NO_HISTORY
    pat[k - 1] = 2                 # RCD_PAT_ACCELERATING (a = 0)
    return f, pat


# k = 1 : H alone: its self pair only, 0 pairs pending, no group runs.
# k = 2 : one 4-entry batch with one pair (H, j): the warp ends with 1 pending pair.
# k = 32: one tile whose single chunk holds all 32 objects: H's run is one whole batch with its self pair in it,
#         31 pending pairs at the end of that warp's batches.
# k = 33: two tiles; chunk 0 of each holds the first 32 objects in cell order, i.e. everything but H, so H's run
#         in chunk 0 is one whole batch of 32 pairs, none of them its self pair: exactly one full group runs
#         between batches and the warp ends with 0 pending.  Chunk 1 holds H alone (self pairs only).
@pytest.mark.parametrize("k", [1, 2, 32, 33])
def test_group_boundaries_small_frames(k):
    from rcd_b200.host.engine import FrameEngine
    frame, pat = _stack_frame(k)
    with FrameEngine(k, 1 << 16, world_bounds=((-200.0, -200.0, -50.0), (200.0, 200.0, 150.0))) as e:
        got = _check_fused(e, frame, pat)
    assert (got["predicted"] == 1).sum() == k - 1  # H is predicted to meet every other object


def test_groups_carried_across_batches_100k_clustered():
    """100 k clustered 3-D objects at the density of the bench frame (configs[3] on a 10 km map).  About one pair
    test in 30 of the frame's ~10^8 survives into the queue, so its QA batches far outnumber the 4 * 8 * SMs warps
    of k_narrow: every warp gathers its groups over many batches and carries what is left of one batch into the
    next.  Every 37th object is queried by the oracle against the whole frame."""
    from rcd_b200.host import workloads as W
    from rcd_b200.host.engine import FrameEngine
    n = 100_000
    frame = W.hotspot_frame(n, 2002, 10000.0, 50)
    pat = W.random_patterns(n, 5)
    with FrameEngine(n, 4_000_000, world_bounds=((0, 0, 0), (10000, 10000, 100))) as e:
        got = _check_fused(e, frame, pat, query_stride=37)
        assert e.counts()["n_fallback"] == 0
    assert (got["predicted"] == 1).sum() > 1000
