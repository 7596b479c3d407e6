"""The reference's fused 20-neighbour sweep (gipuma_black_cu / gipuma_red_cu, gipuma.cu:1122-1351, 1714-1725, 1770-1781) —
what `runcuda` launches when the reference is built without SMALLKERNEL (gipuma.cu:1913-1940) — selected here with
gpm_set_option("neighbours", 20).  Bar: bit-exact, against committed golden outputs of the pinned reference build and
against outputs of the reference build recorded on a B200 (oracle/recorded.py)."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, bits_equal

pytestmark = pytest.mark.gpu

FUSED = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "fused_*.npz")))


def _load(name):
    from gipuma_b200.golden import scene_from_arrays
    z = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    return scene_from_arrays(name, z), z


@pytest.mark.parametrize("name", FUSED)
def test_fused_kernels_match_golden(name):
    from gipuma_b200 import api
    sc, z = _load(name)
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.set_option("neighbours", 20)
        ctx.load_scene(sc, seed=int(z["seed"]))
        ctx.init()
        n4, c = ctx.get_state()
        assert bits_equal(n4, z["init_norm4"]) == 0 and bits_equal(c, z["init_cost"]) == 0
        ctx.phase(0, 7)                                   # gipuma_black_cu: 20 candidates + refinement, one launch
        n4, c = ctx.get_state()
        assert bits_equal(n4, z["black_norm4"]) == 0 and bits_equal(c, z["black_cost"]) == 0
        ctx.phase(1, 7)                                   # gipuma_red_cu
        n4, c = ctx.get_state()
        assert bits_equal(n4, z["iter1_norm4"]) == 0 and bits_equal(c, z["iter1_cost"]) == 0


@pytest.mark.parametrize("name", FUSED)
@pytest.mark.parametrize("opts", [{}, {"memo": 0}, {"memo": 0, "prune": 0, "dedupe": 0}])
def test_fused_full_run_matches_golden(name, opts):
    from gipuma_b200 import api
    sc, z = _load(name)
    o = dict(opts, neighbours=20)
    ls, ms, st = api.runcuda(sc, seed=int(z["seed"]), options=o)
    assert bits_equal(ls.norm4, z["final_norm4"]) == 0
    assert bits_equal(ls.c, z["final_cost"]) == 0
    assert st["launches"] == 2 + 2 * sc.params.iterations + 1


LIVE = [
    # rows, cols, views, iters, box, n_best, comb, colour, seed
    (96, 128, 5, 3, 11, 3, 1, False, 5),
    (64, 96, 2, 2, 15, 2, 1, False, 6),
    (64, 96, 6, 2, 7, 3, 3, False, 7),                 # COMB_GOOD
    (64, 64, 4, 3, 21, 3, 1, False, 8),                # border-heavy: every guard of the 20 candidates is exercised
    (96, 128, 4, 3, 9, 3, 1, True, 9),                 # float4
    (64, 96, 33, 1, 5, 3, 1, True, 10),                # float4, > 32 views (pin P3 build)
]


@pytest.mark.parametrize("rows,cols,views,iters,box,nbest,comb,colour,seed", LIVE)
def test_fused_full_run_bit_exact_vs_live_reference(request, rows, cols, views, iters, box, nbest, comb, colour, seed):
    """Against the reference's outputs as recorded on a B200 (oracle/recorded.py)."""
    from gipuma_b200 import api, scene as S
    from oracle import recorded
    sc = S.make_config(4 if views > 10 else 2, rows=rows, cols=cols, n_views=views, iterations=iters, seed=3000 + seed)
    sc.params.box_hsize = sc.params.box_vsize = box
    sc.params.n_best = nbest
    sc.params.cost_comb = comb
    if colour:
        sc = S.colorize(sc)

    def run():
        from oracle import pyref
        r_n4, r_c, _ = pyref.Harness("ref64" if views > 32 else "ref").run_fused(sc, seed=seed)
        return {"norm4": r_n4, "cost": r_c}

    ref = recorded.reference(request.node, run)
    for opts in ({}, {"memo": 0, "prune": 0, "dedupe": 0}):
        ls, _, _ = api.runcuda(sc, seed=seed, options=dict(opts, neighbours=20))
        assert ref.bits_differ("norm4", ls.norm4) == 0
        assert ref.bits_differ("cost", ls.c) == 0


def test_fused_mode_through_the_runcuda_adapter(monkeypatch):
    """GIPUMA_B200_NEIGHBOURS=20 makes the drop-in runcuda() behave like a reference built without SMALLKERNEL."""
    from gipuma_b200 import scene as S
    from oracle import pyref
    if not os.path.exists(os.path.join(pyref.REF_DIR, "libhx_dropin.so")):
        pytest.skip("oracle/_ref/libhx_dropin.so not built (needs the reference headers)")
    if not FUSED:
        pytest.skip("no fused golden fixtures")
    sc, z = _load(FUSED[0])
    monkeypatch.setenv("GIPUMA_B200_NEIGHBOURS", "20")
    n4, c, _, _ = pyref.Harness("dropin").run(sc, seed=int(z["seed"]))
    assert bits_equal(n4, z["final_norm4"]) == 0 and bits_equal(c, z["final_cost"]) == 0


def test_view_shard_refuses_the_fused_sweep():
    import torch
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=64, cols=96, n_views=3, iterations=1, seed=1)
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.set_option("neighbours", 20)
        ctx.load_scene(sc)
        ctx.init_planes()
        buf = torch.empty(ctx.shard_stage_floats(0), dtype=torch.float32, device="cuda")
        with pytest.raises(api.GipumaError):
            ctx.shard_stage(0, 0, None, 1, buf)
        with pytest.raises(api.GipumaError):
            ctx.set_option("neighbours", 12)
