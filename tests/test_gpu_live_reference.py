"""GPU parity against the pinned reference build (oracle/_ref/libhx_ref*.so) on fresh seeds, sizes and parameter corners
that the committed golden fixtures do not cover.  The reference's outputs are digests recorded on a B200
(tests/golden/reference_outputs.json, oracle/recorded.py); GIPUMA_RECORD_REFERENCE records them again from the live build."""
import numpy as np
import pytest

from oracle import recorded

pytestmark = pytest.mark.gpu


def _ref(n_views):
    from oracle import pyref
    return pyref.Harness("ref64" if n_views > 32 else "ref")


def _run(sc, seed):
    def run():
        r_n4, r_c, printed_s, _ = _ref(sc.n_views).run(sc, seed=seed)
        return {"norm4": r_n4, "cost": r_c, "printed_s": printed_s}
    return run


def _every_kernel(sc, seed):
    """Init, the six kernels of one iteration (each from the reference's own previous state) and the final kernel."""
    def run():
        from oracle import pyref
        ref = _ref(sc.n_views)
        out = {}
        n4, c, _ = ref.steps(sc, [pyref.STEP_INIT], seed=seed)
        out["init_norm4"], out["init_cost"] = n4, c
        for step in range(1, 7):
            n4, c, _ = ref.steps(sc, [step], norm4=n4, cost=c, seed=seed)
            out["step%d_norm4" % step], out["step%d_cost" % step] = n4, c
        out["final_norm4"] = ref.steps(sc, [pyref.STEP_COMPUTE_DISP], norm4=n4, cost=c)[0]
        return out
    return run


def reference_tile_fully_loaded(rows, cols, box):
    """True iff the reference's shared-memory loader (gipuma.cu:1510-1525) defines every tile element an in-image
    pixel reads.  Threads outside the image return before loading their 7-8 elements (gipuma.cu:1488-1491), so a
    partial last block column/row leaves holes (SURVEY.md §7, "Reference UB")."""
    if cols % 32:
        return False
    r = rows % 32
    if r == 0:
        return True
    R = (box + 1) // 2
    tw = 32 + 2 * R
    loaded_rows = (224 * ((r + 1) // 2) + 1) // tw
    return r + 2 * R <= loaded_rows


CASES = [
    # cfg, rows, cols, views, iters, box, n_best, cost_comb, seed
    (1, 240, 320, 2, 3, 15, 2, 1, 0xC0FFEE),          # BASELINE config 1 as specified
    (2, 96, 160, 10, 2, 15, 3, 1, 12345),             # dtu_fast parameters, other seed
    (2, 64, 96, 1, 2, 7, 1, 1, 99),                   # single source view
    (2, 64, 96, 6, 2, 11, 8, 1, 5),                   # n_best > number of views
    (2, 64, 96, 6, 2, 11, 3, 0, 5),                   # COMB_ALL
    (2, 64, 96, 6, 2, 11, 3, 3, 5),                   # COMB_GOOD
    (4, 64, 96, 33, 1, 5, 3, 1, 3),                   # 33 views: second view per lane, pin P3 build
    (5, 64, 96, 64, 1, 5, 3, 1, 8),                   # GPM_MAX_VIEWS = 64 source views
    (3, 96, 96, 8, 1, 25, 3, 1, 11),                  # largest window (six 32-sample rounds)
    (2, 64, 96, 5, 2, 3, 2, 1, 1),                    # smallest window
]


@pytest.mark.parametrize("cfg,rows,cols,views,iters,box,nbest,comb,seed", CASES)
def test_full_run_bit_exact_vs_live_reference(request, cfg, rows, cols, views, iters, box, nbest, comb, seed):
    from gipuma_b200 import api, scene as S
    sc = S.make_config(cfg, rows=rows, cols=cols, n_views=views, iterations=iters, seed=1000 + seed)
    sc.params.box_hsize = sc.params.box_vsize = box
    sc.params.n_best = nbest
    sc.params.cost_comb = comb
    assert reference_tile_fully_loaded(rows, cols, box)
    ref = recorded.reference(request.node, _run(sc, seed))
    ls, _, _ = api.runcuda(sc, seed=seed)
    assert ref.bits_differ("norm4", ls.norm4) == 0
    assert ref.bits_differ("cost", ls.c) == 0


COLOR_CASES = [
    # rows, cols, views, iters, box, n_best, cost_comb, seed      (float4 tile of box > 21 exceeds the reference's 48 KB)
    (96, 128, 5, 2, 11, 3, 1, 31337),
    (64, 96, 3, 2, 19, 2, 1, 7),
    (64, 96, 6, 2, 7, 3, 3, 11),                      # COMB_GOOD
    (64, 96, 6, 1, 5, 8, 0, 12),                      # COMB_ALL
    (64, 64, 4, 3, 21, 3, 1, 123),                    # border-heavy, largest float4 window the reference can launch
    (64, 96, 33, 1, 5, 3, 1, 3),                      # > 32 views
]


@pytest.mark.parametrize("rows,cols,views,iters,box,nbest,comb,seed", COLOR_CASES)
def test_color_processing_full_run_bit_exact_vs_live_reference(request, rows, cols, views, iters, box, nbest, comb, seed):
    """-color_processing: float4 images, runcuda<float4> (gipuma.cu:1965-1966)."""
    from gipuma_b200 import api, scene as S
    sc = S.colorize(S.make_config(4 if views > 10 else 2, rows=rows, cols=cols, n_views=views, iterations=iters,
                                  seed=2000 + seed))
    sc.params.box_hsize = sc.params.box_vsize = box
    sc.params.n_best = nbest
    sc.params.cost_comb = comb
    assert reference_tile_fully_loaded(rows, cols, box)
    ref = recorded.reference(request.node, _run(sc, seed))
    for opts in ({}, {"memo": 0, "prune": 0, "dedupe": 0}):
        ls, _, _ = api.runcuda(sc, seed=seed, options=opts)
        assert ref.bits_differ("norm4", ls.norm4) == 0
        assert ref.bits_differ("cost", ls.c) == 0


def test_color_every_kernel_of_one_iteration_vs_live_reference(request):
    from gipuma_b200 import api, scene as S
    sc = S.colorize(S.make_config(2, rows=96, cols=128, n_views=6, iterations=1, seed=4243))
    sc.params.box_hsize = sc.params.box_vsize = 13
    ref = recorded.reference(request.node, _every_kernel(sc, 99))
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.load_scene(sc, seed=99)
        ctx.init()
        m4, mc = ctx.get_state()
        assert ref.bits_differ("init_norm4", m4) == 0 and ref.bits_differ("init_cost", mc) == 0
        ctx.set_option("cost_variant", 3)                 # the initialisation kernel's rounding, on its own planes
        assert ref.bits_differ("init_cost", ctx.cost_eval(m4)) == 0
        for step, (colour, mask) in zip(range(1, 7), [(0, 1), (0, 2), (0, 4), (1, 1), (1, 2), (1, 4)]):
            ctx.phase(colour, mask)
            m4, mc = ctx.get_state()
            assert ref.bits_differ("step%d_norm4" % step, m4) == 0, "planes differ after reference kernel %d" % step
            assert ref.bits_differ("step%d_cost" % step, mc) == 0, "costs differ after reference kernel %d" % step
        ctx.finalize()
        m4, mc = ctx.get_state()
        assert ref.bits_differ("final_norm4", m4) == 0


def test_color_and_gray_images_cannot_be_mixed():
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=64, cols=96, n_views=2, iterations=1, seed=1)
    cs = S.colorize(sc)
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.set_params(sc.params)
        ctx.set_reference(np.ascontiguousarray(cs.images[0]), cs.cameras[0])
        with pytest.raises(api.GipumaError):
            ctx.set_view(0, np.ascontiguousarray(sc.images[1]), sc.cameras[1])


def test_ragged_image_size_init_and_cost_bit_exact(request):
    """75 x 53 (no multiple of 32 or 16, narrower than two tiles).  The reference's sweep kernels read unloaded
    shared memory for such shapes, so only the stages that do not depend on its tile loader are compared:
    initialisation (texture path) and the cost function on identical planes (harness kernel, whole tile loaded)."""
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=53, cols=75, n_views=4, iterations=2, seed=77)
    sc.params.box_hsize = sc.params.box_vsize = 9

    def run():
        from oracle import pyref
        ref = _ref(sc.n_views)
        n4, c, _ = ref.steps(sc, [pyref.STEP_INIT], seed=5)
        return {"init_norm4": n4, "init_cost": c, "sweep_cost": ref.cost_eval(sc, n4)}

    ref = recorded.reference(request.node, run)
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.load_scene(sc, seed=5)
        ctx.init()
        m4, mc = ctx.get_state()
        assert ref.bits_differ("init_norm4", m4) == 0 and ref.bits_differ("init_cost", mc) == 0
        assert ref.bits_differ("sweep_cost", ctx.cost_eval(m4)) == 0
        ctx.sweep(2)
        ctx.finalize()
        o4, oc = ctx.get_state()
    assert np.isfinite(o4).all() and np.isfinite(oc).all()


def test_every_kernel_of_one_iteration_vs_live_reference(request):
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=96, cols=128, n_views=7, iterations=1, seed=4242)
    ref = recorded.reference(request.node, _every_kernel(sc, 31337))
    with api.Context(sc.cols, sc.rows, sc.n_views) as ctx:
        ctx.load_scene(sc, seed=31337)
        ctx.init()
        m4, mc = ctx.get_state()
        assert ref.bits_differ("init_norm4", m4) == 0 and ref.bits_differ("init_cost", mc) == 0
        for step, (colour, mask) in zip(range(1, 7), [(0, 1), (0, 2), (0, 4), (1, 1), (1, 2), (1, 4)]):
            ctx.phase(colour, mask)
            m4, mc = ctx.get_state()
            assert ref.bits_differ("step%d_norm4" % step, m4) == 0, "planes differ after reference kernel %d" % step
            assert ref.bits_differ("step%d_cost" % step, mc) == 0, "costs differ after reference kernel %d" % step
        ctx.finalize()
        m4, mc = ctx.get_state()
        assert ref.bits_differ("final_norm4", m4) == 0


def test_non_8bit_images_stay_exact(request):
    """Arbitrary (non-8-bit) float images."""
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=96, cols=128, n_views=5, iterations=2, seed=2024)
    rng = np.random.default_rng(9)
    sc.images = (sc.images * 0.731 + rng.uniform(0, 3, size=sc.images.shape)).astype(np.float32)      # not integers
    ref = recorded.reference(request.node, _run(sc, 77))
    ls, _, _ = api.runcuda(sc, seed=77)
    assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0


def test_border_heavy_scene(request):
    """Small image, large window, strongly tilted random planes: many samples project onto or beyond the image border."""
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2, rows=64, cols=64, n_views=4, iterations=3, seed=31)
    sc.params.box_hsize = sc.params.box_vsize = 21
    ref = recorded.reference(request.node, _run(sc, 123))
    for opts in ({}, {"memo": 0}):
        ls, _, _ = api.runcuda(sc, seed=123, options=opts)
        assert ref.bits_differ("norm4", ls.norm4) == 0 and ref.bits_differ("cost", ls.c) == 0


def test_baseline_config2_full_size_bit_exact_vs_live_reference(request):
    """BASELINE configs[1] as benchmarked: 1600 x 1200, 10 source views, 8 iterations, blocksize 15 — all 9.6 M output
    floats identical to the reference's."""
    from gipuma_b200 import api, scene as S
    sc = S.make_config(2)
    assert reference_tile_fully_loaded(sc.rows, sc.cols, sc.params.box_hsize)
    ref = recorded.reference(request.node, _run(sc, 0xC0FFEE))
    ls, ms, st = api.runcuda(sc)
    assert ref.bits_differ("norm4", ls.norm4) == 0
    assert ref.bits_differ("cost", ls.c) == 0
    assert ms / 1e3 < ref["printed_s"]   # and faster than the reference over the same span (its time recorded on a B200)
