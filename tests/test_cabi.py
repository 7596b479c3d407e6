"""The drop-in boundary: libgipuma_b200.so loads on a CPU-only box, exports every symbol include/gipuma_b200.h
declares, and refuses to compute without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gipuma_b200.h")


def declared_symbols():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gpm_[a-z_0-9]+)\s*\(", txt)))


def test_header_declares_the_documented_surface():
    syms = declared_symbols()
    for s in ("gpm_create", "gpm_destroy", "gpm_set_params", "gpm_set_reference", "gpm_set_view", "gpm_set_rng",
              "gpm_init", "gpm_sweep", "gpm_phase", "gpm_finalize", "gpm_run", "gpm_get_state", "gpm_set_state",
              "gpm_cost_eval", "gpm_last_error"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    from gipuma_b200 import api
    lib = api.load_library()
    for s in declared_symbols():
        assert hasattr(lib, s), "libgipuma_b200.so does not export %s" % s


def test_header_is_plain_c(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "gipuma_b200.h"\nint main(void){ gpm_params p; gpm_camera c; (void)p; (void)c; return sizeof(p) > 0 ? 0 : 1; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "t.o")])


def test_struct_layouts_match_ctypes():
    from gipuma_b200 import api
    code = r'''
#include <stdio.h>
#include "gipuma_b200.h"
int main(void){ printf("%zu %zu\n", sizeof(gpm_params), sizeof(gpm_camera)); return 0; }
'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(code)
        subprocess.check_call(["gcc", "-I" + os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        a, b = map(int, subprocess.check_output([os.path.join(d, "s")]).split())
    assert a == ctypes.sizeof(api.GpmParams) and b == ctypes.sizeof(api.GpmCamera)


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    from gipuma_b200 import api
    with pytest.raises(api.GipumaError) as e:
        api.Context(64, 64, 2)
    assert "CUDA" in str(e.value) or "device" in str(e.value)


def test_missing_library_fails_loudly():
    env = dict(os.environ, GIPUMA_B200_LIB="/nonexistent/libgipuma_b200.so", PYTHONPATH=ROOT)
    code = "from gipuma_b200 import api\ntry:\n    api.load_library()\nexcept api.GipumaError as e:\n    print('LOUD', e)\n"
    out = subprocess.check_output([sys.executable, "-c", code], env=env).decode()
    assert out.startswith("LOUD") and "no CPU fallback" in out


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gipuma_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in txt and "from oracle" not in txt and "gipuma_oracle" not in txt, f


def test_python_binding_refuses_buffers_it_would_reinterpret():
    """api._ptr hands raw addresses to the C-ABI, which reads float32 row-major memory: other dtypes / strided views are refused
    (images are converted, outputs must be right)."""
    import numpy as np
    from gipuma_b200 import api
    with pytest.raises(TypeError):
        api._ptr(np.zeros((4, 4), np.float64))
    with pytest.raises(TypeError):
        api._ptr(np.zeros((4, 8), np.float32)[:, ::2])
    img = api._image(np.arange(12, dtype=np.uint8).reshape(3, 4))
    assert img.dtype == np.float32 and img.flags["C_CONTIGUOUS"] and img[2, 3] == 11.0


def test_bench_arms_describe_the_same_workload():
    """The driver compares the two arms' `config` objects: they must be identical for every mode (VERDICT r1: same_config)."""
    import argparse
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for world, mode in ((1, "auto"), (2, "auto"), (8, "auto"), (4, "batch"), (8, "hybrid")):
        args = argparse.Namespace(mode=mode, config=0, shard=0, color=False, neighbours=8, scene="smooth")
        m, cfg, shard = bench.resolve(args, world)
        a = bench.config_dict(args, m, cfg, shard, world, "scene", 1600, 1200, 60, 8, 15, 3)
        b = bench.config_dict(args, m, cfg, shard, world, "scene", 1600, 1200, 60, 8, 15, 3)
        assert a == b and a["mode"] == m
        if world == 1:
            assert m == "single" and cfg == 2
        if mode == "auto" and world > 1:
            assert m == "view_shard" and cfg == 6 and shard == world


def test_bench_dump_outputs_stays_within_64_mb_with_a_fixed_sample(tmp_path):
    """bench.py --dump-outputs: whole outputs when they fit, else the same seeded pixel sample on every run."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(3)
    small = rng.standard_normal((120, 160, 4)).astype(np.float32), rng.standard_normal((120, 160)).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "small"), *small)
    assert sorted(os.listdir(tmp_path / "small")) == ["cost.npy", "norm4.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "norm4.npy"), small[0])
    assert np.array_equal(np.load(tmp_path / "small" / "cost.npy"), small[1])
    H, W = 2400, 3200                                         # BASELINE configs[4]: 154 MB of outputs
    norm4 = np.broadcast_to(np.arange(H * W, dtype=np.float32).reshape(H, W, 1), (H, W, 4))
    cost = -np.arange(H * W, dtype=np.float32).reshape(H, W)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), norm4, cost)
        files = [tmp_path / run / f for f in ("norm4.npy", "cost.npy", "pixel_index.npy")]
        assert sum(os.path.getsize(f) for f in files) <= 64 * 10 ** 6
        idx = np.load(files[2])
        assert idx.dtype == np.float64 and len(np.unique(idx)) == idx.size
        assert np.array_equal(np.load(files[0])[:, 0], idx.astype(np.float32))
        assert np.array_equal(np.load(files[1]), -idx.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "pixel_index.npy"), np.load(tmp_path / "b" / "pixel_index.npy"))


def test_batch_driver_validates_arguments_and_has_no_cpu_fallback():
    """gpm_batch_run (host C++): bad descriptors are refused before any CUDA call; without a device the workers fail loudly
    (no CPU path), with the reason in gpm_batch_last_error()."""
    import numpy as np
    from gipuma_b200 import api, scene as S
    params = S.AlgorithmParameters(box_hsize=9, box_vsize=9, iterations=1, n_best=2, cost_comb=S.COMB_BEST_N)
    params.depthMin, params.depthMax = 300.0, 800.0
    P = [S.load_dtu_projections()[i] for i in range(3)]
    imgs = np.zeros((3, 64, 96), np.float32)
    with pytest.raises(api.GipumaError, match="bad arguments"):
        api.batch_run(imgs[:1], P[:1], params, [0])                       # a reference view needs at least one source view
    with pytest.raises(api.GipumaError, match="bad arguments"):
        api.batch_run(imgs, P, params, [0], max_views=0)
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:      # noqa: BLE001
        has_gpu = False
    if not has_gpu:
        with pytest.raises(api.GipumaError, match="CUDA"):
            api.batch_run(imgs, P, params, [0], cam_scale=1600.0 / 96)


def test_cpp_host_example_builds_and_fails_loudly_without_a_device(tmp_path):
    """examples/shard_host.cpp links against the C-ABI with plain g++ (no CUDA headers); without a GPU it must exit non-zero
    with the library's "no CUDA device" message — there is no CPU path to fall back to."""
    from gipuma_b200 import build, scene as S
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import dump_scene
    exe = build.build_examples()
    assert os.path.exists(exe)
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present: covered by tests/test_gpu_cpp_host.py")
    except ImportError:
        pass
    sc = S.make_config(1, rows=64, cols=96)
    scene_file = str(tmp_path / "scene.bin")
    dump_scene.dump(sc, scene_file)
    p = subprocess.run([exe, scene_file, str(tmp_path / "out.bin"), "1"], capture_output=True, text=True, timeout=120)
    assert p.returncode != 0 and "CUDA" in p.stderr
