"""Every BASELINE.json configuration at FULL size against the pinned reference build (oracle/_ref), bit for bit:
configs[2] (dtu_accurate, 1600x1200, 30 views, blocksize 25), configs[3] (templeRing shape, 640x480, 47 views, pin P3 build),
configs[4] (3200x2400, 64 views, pin P3 build) and north_star's 60-view job.  configs[1] is covered by
test_gpu_live_reference.py::test_baseline_config2_full_size_bit_exact_vs_live_reference.

configs[2] needs care: with 1200 rows and blocksize 25 the reference's tile loader leaves the bottom of the last block row's
shared-memory window unloaded (threads outside the image return first, gipuma.cu:1488-1491 vs 1510-1525; SURVEY.md §7), so
its pixels in rows >= 1189 read stale shared memory.  The damage travels upwards by at most 6 rows per colour pass
(close + far propagation) = 96 rows in 8 iterations, so rows < 1088 must still be identical; and the same job at 1600 x 1216
(whole tile rows, no undefined behaviour in the reference) must be identical everywhere.

The reference's outputs and times are digests recorded on a B200 (tests/golden/reference_outputs.json, oracle/recorded.py);
GIPUMA_RECORD_REFERENCE records them again from the live build."""
import os

import pytest

from oracle import recorded

pytestmark = pytest.mark.gpu
WORKERS = max(1, min(32, len(os.sched_getaffinity(0))))


def _both(node, sc, safe=None):
    """Our run and the reference's recorded outputs; with `safe`, the reference's rows [:safe] and the costs below."""
    from gipuma_b200 import api

    def run():
        from oracle import pyref
        r_n4, r_c, printed_s, _ = pyref.Harness("ref64" if sc.n_views > 32 else "ref").run(sc)
        if safe is None:
            return {"norm4": r_n4, "cost": r_c, "printed_s": printed_s}
        return {"norm4_above": r_n4[:safe], "cost_above": r_c[:safe], "cost_below": r_c[safe:], "printed_s": printed_s}

    ref = recorded.reference(node, run)
    ls, ms, _ = api.runcuda(sc)
    return ls, ref, ms / 1e3


def test_config3_dtu_accurate_full_size_tile_aligned_bit_exact(request):
    from gipuma_b200 import scene as S
    sc = S.make_config(3, rows=1216, cols=1600, workers=WORKERS)          # 38 whole tile rows: the reference loads every window
    ls, ref, ours_s = _both(request.node, sc)
    assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0
    assert ours_s < ref["printed_s"]


def test_config3_dtu_accurate_full_size_as_specified(request):
    from gipuma_b200 import scene as S
    sc = S.make_config(3, workers=WORKERS)                                 # 1600 x 1200: reference UB in the last block row
    safe = 1189 - 6 * 2 * sc.params.iterations - 5
    ls, ref, ours_s = _both(request.node, sc, safe)
    assert ref.bits_differ("norm4_above", ls.norm4[:safe]) == 0 and ref.bits_differ("cost_above", ls.c[:safe]) == 0
    # below that line only pixels reached by the reference's stale shared memory may differ: a small minority (estimated
    # on the recorded sample of those costs)
    diff = ref.fraction_differing("cost_below", ls.c[safe:])
    assert diff < 0.5
    assert ours_s < ref["printed_s"]


def test_config4_temple_ring_full_size_bit_exact(request):
    from gipuma_b200 import scene as S
    sc = S.make_config(4, workers=WORKERS)                                 # 640 x 480, 47 views, blocksize 11
    ls, ref, ours_s = _both(request.node, sc)
    assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0
    assert ours_s < ref["printed_s"]


def test_northstar_60_view_job_full_size_bit_exact(request):
    from gipuma_b200 import scene as S
    sc = S.make_config(6, workers=WORKERS)                                 # 1600 x 1200, 60 views, dtu_fast parameters
    ls, ref, ours_s = _both(request.node, sc)
    assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0
    assert ours_s < ref["printed_s"]


def test_config5_3200x2400_64_views_full_size_bit_exact(request):
    from gipuma_b200 import scene as S
    sc = S.make_config(5, workers=WORKERS)
    ls, ref, ours_s = _both(request.node, sc)
    assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0
    assert ours_s < ref["printed_s"]
