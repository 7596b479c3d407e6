#!/usr/bin/env python
"""bench.py — headline benchmark of the PatchMatch hot path (BASELINE.json metric: Mpixel-iters/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode auto|single|batch|view_shard|hybrid]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one complete pass of the hot path over one reference view: random initialisation, `iterations` red/black
sweeps, final depth/normal kernel (what the reference's runcuda() does once per process).

Workloads (synthetic 8-bit images rendered from a textured height field, real DTU camera geometry; `--scene hard` adds
occluding blocks, a texture-less band and sensor noise):
  N = 1 (mode single)      BASELINE.json configs[1]: 'dtu_fast' parameters, 1600x1200, 10 source views, 8 iterations.
  N > 1 (mode view_shard)  north_star's strong-scaling job: ONE 1600x1200 reference view with 60 source views (dtu_fast
                           parameters) whose source views are sharded over the N ranks; after every exchange stage the ranks'
                           local top-n_best view costs are all-gathered over NCCL/NVLink (gpm_shard_run, behind the C-ABI)
                           and combined exactly as pmCostMultiview_cu does (gipuma.cu:742-806).  "scaling": "strong".
                           Default exchange: one ncclAllGather per stage (measured 4-6 % faster than the fused peer-memory
                           kernel, DESIGN.md §9); --exchange p2p selects the fused kernel.
                           Rank 0 also runs the same job unsharded and reports whether the outputs are bit-identical.
  --mode batch             every rank its own reference view (scripts/dtu_fast.sh:30-55), no collective, weak scaling.
  --mode hybrid --shard G  BASELINE configs[4]: N/G groups, each one 3200x2400 / 64-view reference view sharded G ways.

Printed JSON (one line, rank 0):
  value        Mpixel-iters/s = jobs * W*H*iterations / 1e6 / t, t = device time from the first sweep kernel to the end of the
               final kernel (the reference's own timed span, gipuma.cu:1908-1952; init excluded), inputs resident in HBM;
               summed over the K timed steps, max over ranks.
  ms_per_step  full device time of a step INCLUDING initialisation.
  e2e          same metric through the public API with HOST buffers: per step the images are uploaded from pinned host
               memory (H2D), the job runs, and planes+costs are read back (D2H); wall clock around the call.
  roofline     HBM line of the dominant kernel from SURVEY.md §8(d)'s algorithmic bytes (164 + 12 V per pixel-iteration,
               the unfused three-phase formula) and its live CUDA-event duration; `binding_unit` is the texture unit:
               filtered fetches per second achieved (live counters) over the ceiling measured in this process.
  cpu_baseline the single-thread C restatement (oracle/gipuma_oracle.c) on a FIXED band of rows of the N = 1 workload.
--dump-outputs DIR writes what rank 0's last timed step computed (see dump_outputs); the inputs of a workload are the same
in every run, so two builds can be compared output for output.
--impl reference times the reference's own implementation of the path — gipuma.cu compiled unmodified for sm_100a
(oracle/_ref, pins P1/P2 by macro, P3 for > 32 views) — on the same workload, same metric, on one GPU.  (The reference
has no CPU implementation of this path; its CUDA kernels are "the reference's own implementation", DESIGN.md §7.)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mpixel-iters/s (ref-view PatchMatch sweep)"
UNIT = "Mpixel-iters/s"
FETCHES_PER_PAIR = 5          # bilinear fetches per (view, sample): centre, x+-1, y+-1 (gipuma.cu:251-253)
DUMP_BYTES = 64 * 10 ** 6     # --dump-outputs: at most this much in all ...
DUMP_PIXELS = 1 << 21         # ... else this many sampled pixels (20 B of outputs + 8 B of index each)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([t.strip() for t in out.split(",")])
            except Exception:      # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def finish(self) -> dict:
        self._halt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 3 + i and r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


# ---------------------------------------------------------------------------------------------------------------------
# workload definition — shared by both arms so that their `config` objects are identical
# ---------------------------------------------------------------------------------------------------------------------

def resolve(args, world):
    mode = args.mode
    if mode == "auto":
        mode = "single" if world == 1 else "view_shard"
    if mode == "single" and world > 1:
        mode = "batch"
    config = args.config if args.config else {"single": 2, "batch": 2, "view_shard": 6, "hybrid": 5}[mode]
    shard = world
    if mode == "hybrid":
        shard = args.shard if args.shard else max(1, world // 2)
        if world % shard:
            raise SystemExit("--shard must divide the number of GPUs")
    return mode, config, shard


def workers_for(world):
    n = len(os.sched_getaffinity(0)) // max(1, world)
    return max(1, min(32, n))


def make_scene(args, config, seed_rank, world, positions=None):
    from gipuma_b200 import scene as S
    sc = S.make_config(config, seed=1234 + 17 * seed_rank, hard=(args.scene == "hard"), workers=workers_for(world),
                       render_positions=positions)
    return S.colorize(sc) if args.color else sc


def config_label(config):
    return {1: "BASELINE configs[0]", 2: "BASELINE configs[1]", 3: "BASELINE configs[2]", 4: "BASELINE configs[3]",
            5: "BASELINE configs[4]", 6: "north_star 60-view job"}[config]


def config_dict(args, mode, config, shard, world, sc_name, W, H, V, iters, box, n_best):
    suffix = ""
    if args.color:
        suffix += ", -color_processing (float4 images)"
    if args.neighbours == 20:
        suffix += ", fused 20-neighbour sweep (reference built without SMALLKERNEL)"
    if args.scene == "hard":
        suffix += ", hard scene (occluders, texture-less band, sensor noise)"
    par = {"single": "one reference view on one GPU",
           "batch": "reference-view batch: one independent reference view per GPU, no collective",
           "view_shard": "one reference view, source views sharded over the GPUs; per exchange stage every rank's local top-n_best view costs reach all ranks (NCCL all-gather over NVLink behind the C-ABI; --exchange p2p: fused peer-memory exchange)",
           "hybrid": "groups of %d GPUs shard the source views of their group's reference view; groups are independent" % shard}[mode]
    return {"workload": "%s: %s, %dx%d, %d source views, %d iterations, blocksize %d, n_best %d" % (config_label(config), sc_name, W, H, V, iters, box, n_best) + suffix,
            "mode": mode, "parallelism": par,
            "timed_span": "first sweep kernel .. end of final depth/normal kernel (the reference's own span, gipuma.cu:1908-1952; init excluded)",
            "l2": "flushed between timed steps (256 MiB write)",
            "rng": "seed 0xC0FFEE, reference zero-state refinement RNG (pins P1/P2)"}


def hbm_algorithmic_bytes_per_pixel_iter(V):
    """SURVEY.md §8(d): 3 phases x (own state r+w 40 B + reference 4 B + 4 V B of source images) + 32 B neighbour planes."""
    return 164 + 12 * V


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:      # noqa: BLE001
        return {}


def load_traffic(key):
    """dram__bytes_read + write per launch of the dominant kernel from this round's committed ncu capture, or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        return t.get(key)
    except Exception:      # noqa: BLE001
        return None


def dump_outputs(path, norm4, cost):
    """The outputs of a run as the caller receives them: planes [H, W, 4] (world normal xyz, depth) as DIR/norm4.npy and
    costs [H, W] as DIR/cost.npy, float32.  Above DUMP_BYTES the same fixed, seeded sample of DUMP_PIXELS pixels is
    written for every run of the workload ([P, 4] and [P]), with their flat pixel indices as DIR/pixel_index.npy."""
    os.makedirs(path, exist_ok=True)
    norm4 = np.ascontiguousarray(norm4, dtype=np.float32)
    cost = np.ascontiguousarray(cost, dtype=np.float32)
    if norm4.nbytes + cost.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(cost.size, DUMP_PIXELS, replace=False))
        norm4, cost = norm4.reshape(-1, 4)[idx], cost.reshape(-1)[idx]
        np.save(os.path.join(path, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "norm4.npy"), norm4)
    np.save(os.path.join(path, "cost.npy"), cost)


def cpu_baseline(sc, neighbours: int = 8) -> dict:
    """Single-thread C restatement on a fixed band: one iteration over rows [H/2, H/2 + 8) of the workload; then the same
    code with every host thread on rows [H/2, H/2 + 2 * threads) (reported separately)."""
    from oracle import pyoracle
    o = pyoracle.Oracle(sc)
    rng = np.random.default_rng(0)
    H, W = sc.rows, sc.cols

    def band(rows, threads):
        n = o.set_threads(threads)
        pl = np.zeros((H, W, 4), np.float32)
        pl[..., 2] = -1.0
        pl[..., 3] = sc.gt_depth * rng.uniform(0.9, 1.1, size=(H, W)).astype(np.float32)
        y0 = H // 2
        cost = np.full((H, W), 50.0, np.float32)
        cost[y0:y0 + rows] = o.cost_eval(pl, y0, y0 + rows)[y0:y0 + rows]
        t0 = time.perf_counter()
        if neighbours == 20:                                         # fused kernel: 20 candidates + refinement per colour
            for colour in (0, 1):
                pl, cost = o.phase(pl, cost, colour, 8 | 4, y0, y0 + rows)
        else:
            o.sweep(pl, cost, 1, y0, y0 + rows)
        dt = time.perf_counter() - t0
        return rows * W / 1e6 / dt, dt, n, y0

    v1, dt1, _, y0 = band(8, 1)
    all_threads = len(os.sched_getaffinity(0))
    out = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
           "sample": "1 iteration over the fixed rows [%d,%d) of the same %dx%d / %d-view workload, 1 thread: %.1f s (host has %d cores)"
                     % (y0, y0 + 8, W, H, sc.n_views, dt1, os.cpu_count() or 0)}
    if all_threads > 1:
        vm, dtm, n, _ = band(min(H // 2, 2 * all_threads), all_threads)
        out["all_threads"] = {"value": vm, "cores": n, "sample": "rows [%d,%d), %.1f s" % (y0, y0 + min(H // 2, 2 * all_threads), dtm)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------

def roofline_block(W, H, V, iters, sweep_ms_per_step, launches_per_step, pairs_per_step, fetch_peak, kernel, traffic, fetches_per_pair):
    peaks = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    avg_launch_ms = sweep_ms_per_step / launches_per_step
    alg_bytes = hbm_algorithmic_bytes_per_pixel_iter(V) * W * H * iters / launches_per_step
    achieved = alg_bytes / 1e9 / (avg_launch_ms / 1e3)
    gfetch = pairs_per_step * fetches_per_pair / 1e9 / (sweep_ms_per_step / 1e3)
    r = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
         "traffic": traffic["bytes_per_launch"] if traffic else None,
         "traffic_source": traffic["source"] if traffic else None,
         "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
         "kernel": kernel, "avg_launch_ms": avg_launch_ms, "launches_per_step": launches_per_step,
         "algorithmic_bytes_per_launch": alg_bytes,
         "algorithmic_bytes_formula": "SURVEY.md §8(d): (164 + 12 V) B per pixel-iteration (unfused 3-phase formula), V = %d; "
                                      "the fused colour launch's own floor is (40+4+4V)+32 = %d B" % (V, 76 + 4 * V),
         "binding_unit": {"name": "texture unit (L1TEX data pipe): filtered R32F fetches",
                          "achieved": gfetch, "peak": fetch_peak, "unit": "Gfetch/s",
                          "frac": (gfetch / fetch_peak) if fetch_peak else None,
                          "how": "achieved = (view,sample) pairs evaluated (device counters of the timed steps) x %d fetches / sweep time; "
                                 "peak = gpm_measure_fetch_peak in this process (dense 8x4-texel footprints on the same texture)" % fetches_per_pair},
         "note": "this path is a gather: each evaluated hypothesis does ~3200 bilinear fetches against a few hundred compulsory HBM "
                 "bytes (SURVEY.md 'Read this first' #4), so the HBM fraction is << 1 % by construction; the texture unit is the roof"}
    return r


def run_ours_single_or_batch(args, mode, config, rank, world, local, sc):
    import torch
    from gipuma_b200 import api
    torch.cuda.set_device(local)
    W, H, V, iters = sc.cols, sc.rows, sc.n_views, sc.params.iterations
    pinned = torch.from_numpy(np.ascontiguousarray(sc.images)).pin_memory()
    out4 = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
    outc = torch.empty((H, W), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")          # > 126 MB L2
    ctx = api.Context(W, H, V, device=local)
    if args.neighbours != 8:
        ctx.set_option("neighbours", args.neighbours)
    imgs = [pinned[i] for i in range(pinned.shape[0])]

    def upload():
        ctx.load_scene(sc, images=imgs)                                       # H2D from pinned host memory

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    upload()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.ExternalStream(ctx.stream)
    for _ in range(args.warmup):
        ctx.run()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # ---- device-resident timing -----------------------------------------------------------------------------
    barrier()
    sweep_ms = step_ms = 0.0
    launches = 0
    pairs = hyp = skipped = pruned = 0
    for _ in range(args.steps):
        flush.fill_(1)                                                        # L2 flush between timed iterations
        torch.cuda.synchronize()
        e0.record(stream)
        sweep_ms += ctx.run()                                                 # the library's own CUDA-event span
        e1.record(stream)
        e1.synchronize()
        step_ms += e0.elapsed_time(e1)
        st = ctx.stats()
        launches += st["launches"]
        pairs += st["pairs"];  hyp += st["hypotheses"];  skipped += st["skipped"];  pruned += st["pruned"]
    barrier()
    outputs = ctx.get_state() if args.dump_outputs and rank == 0 else None    # the last timed step's result
    # ---- end to end through the public API, host buffers ------------------------------------------------------
    e2e_s = 0.0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        upload()
        ctx.run()
        ctx.get_state_into(out4, outc)                                        # D2H of planes + costs
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
    barrier()
    clocks = sampler.finish() if sampler else None
    t = torch.tensor([sweep_ms, step_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)    # max over ranks
    sweep_ms, step_ms, e2e_ms = [float(v) for v in t.tolist()]
    line = None
    if rank == 0:
        fetch_peak = ctx.measure_fetch_peak()
        ablation = {}
        if world == 1 and not args.no_ablation:   # how much of the speed is skipped work: the same job without the exact shortcuts
            for name, opts in (("value_memo_off", {"memo": 0}), ("value_prune_off", {"prune": 0}),
                               ("value_memo_prune_dedupe_off", {"memo": 0, "prune": 0, "dedupe": 0}), ("value_quadperm_off", {"quadperm": 0})):
                for k, v in opts.items():
                    ctx.set_option(k, v)
                ctx.run()
                ms = ctx.run()
                ablation[name] = W * H * iters / 1e3 / ms
                for k in opts:
                    ctx.set_option(k, 1)
        units = world * args.steps * W * H * iters / 1e6
        cfg = config_dict(args, mode, config, world, world, sc.name, W, H, V, iters, sc.params.box_hsize, sc.params.n_best)
        tkey = "cfg%d%s%s" % (config, "_color" if args.color else "", "_n20" if args.neighbours == 20 else "")
        line = {
            "metric": METRIC, "value": units / (sweep_ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "value_incl_init": units / (step_ms / 1e3),
            "e2e": {"value": units / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(pinned.numel() * 4),
                    "d2h_bytes_per_step": int(W * H * 20), "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches),
            "roofline": roofline_block(W, H, V, iters, sweep_ms / args.steps, 2 * iters, pairs / args.steps, fetch_peak, "gpm::k_sweep",
                                       load_traffic(tkey), FETCHES_PER_PAIR * (3 if args.color else 1)),
            "work": dict({"hypotheses_evaluated": hyp // args.steps, "hypotheses_skipped_exact": skipped // args.steps,
                          "hypotheses_pruned_exact": pruned // args.steps, "view_samples": pairs // args.steps}, **ablation),
            "clocks": clocks,
        }
        if world == 1:                                            # the CPU baseline is timed at N = 1 only
            try:
                line["cpu_baseline"] = cpu_baseline(sc, neighbours=args.neighbours)
            except Exception as e:      # noqa: BLE001
                line["cpu_baseline"] = {"error": repr(e)}
        else:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "timed at N = 1 only"}
    ctx.close()
    if outputs is not None:
        dump_outputs(args.dump_outputs, *outputs)
    return line


def sharded_layout(args, config, shard, rank, world):
    from gipuma_b200 import multigpu as M
    group_of, rank_in, members = M.hybrid_layout(world, shard)
    nviews = {1: 2, 2: 10, 3: 30, 4: 47, 5: 64, 6: 60}[config]
    mine = M.partition_views(nviews, shard)[rank_in[rank]]
    check = rank == 0 and not args.no_check                 # rank 0 also runs the unsharded job: needs every view
    return group_of[rank], rank_in[rank], members, mine, check


def run_ours_sharded(args, mode, config, shard, rank, world, local, sc):
    """view_shard (shard == world) and hybrid (world/shard independent groups)."""
    import torch
    import torch.distributed as dist
    from gipuma_b200 import api, multigpu as M
    my_group, my_rank, members, mine, check = sharded_layout(args, config, shard, rank, world)
    torch.cuda.set_device(local)
    groups = [dist.new_group(ranks=m) if (world > 1 and shard > 1 and len(members) > 1) else None for m in members]
    group = groups[my_group]
    W, H, V, iters = sc.cols, sc.rows, sc.n_views, sc.params.iterations
    used = [0] + [sc.subset[p] for p in mine]
    pinned = {i: torch.from_numpy(np.ascontiguousarray(sc.images[i])).pin_memory() for i in used}
    out4 = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
    outc = torch.empty((H, W), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    runner = M.ViewShardRunner(sc, my_rank, shard, device=local, group=group, exchange=args.exchange)
    ctx = runner.ctx

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.ExternalStream(ctx.stream)
    for _ in range(args.warmup):
        runner.run_timed()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    sweep_ms = step_ms = 0.0
    launches = collectives = pairs = hyp = skipped = 0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=group)
            torch.cuda.synchronize()
        e0.record(stream)
        sweep_ms += runner.run_timed()
        e1.record(stream)
        e1.synchronize()
        step_ms += e0.elapsed_time(e1)
        st = ctx.stats()
        launches += st["launches"];  collectives += st["collectives"];  pairs += st["pairs"];  hyp += st["hypotheses"];  skipped += st["skipped"]
    barrier()
    outputs = ctx.get_state() if args.dump_outputs and rank == 0 else None    # group 0's result of the last timed step
    e2e_s = 0.0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=group)
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        runner.upload(sc, images=pinned)                                      # H2D: reference image + this rank's views
        runner.run_timed()
        if my_rank == 0:
            ctx.get_state_into(out4, outc)                                    # every rank of a group holds the identical result
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
    barrier()
    clocks = sampler.finish() if sampler else None
    h2d = float(len(used) * W * H * 4)
    t = torch.tensor([sweep_ms, step_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(launches), float(pairs), h2d, float(collectives)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    sweep_ms, step_ms, e2e_ms = [float(v) for v in t.tolist()]
    line = None
    if rank == 0:
        n_groups = len(members)
        units = n_groups * args.steps * W * H * iters / 1e6
        fetch_peak = ctx.measure_fetch_peak()
        identical = single_value = None
        if check:
            n4, c = ctx.get_state()
            with api.Context(W, H, V, device=local) as one:
                one.load_scene(sc)
                one.run()
                ms1 = one.run()
                s4, s1 = one.get_state()
            identical = bool(np.array_equal(n4.view(np.uint32), s4.view(np.uint32)) and np.array_equal(c.view(np.uint32), s1.view(np.uint32)))
            single_value = W * H * iters / 1e3 / ms1
        cfg = config_dict(args, mode, config, shard, world, sc.name, W, H, V, iters, sc.params.box_hsize, sc.params.n_best)
        value = units / (sweep_ms / 1e3)
        n_stage_launches = 2 * iters * (gpm_stages := ctx.shard_num_stages())       # per colour: 1 + S evaluations + closing accept
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms / args.steps, "higher_is_better": True, "scaling": "strong" if mode == "view_shard" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "value_incl_init": units / (step_ms / 1e3),
            "e2e": {"value": units / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(cnt[2].item()),
                    "d2h_bytes_per_step": int(n_groups * W * H * 20), "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(cnt[0].item()),
            "collective": {"kind": {"p2p": "fused in the stage kernels: lists stored into every peer's memory over NVLink (CUDA IPC) + per-tile arrival flags, no collective launches (gpm_shard_run / k_shard_fused)",
                                    "nccl": "one ncclAllGather per exchange stage (gpm_shard_run, NCCL loaded behind the C-ABI)", "none": "single rank"}[runner.exchange],
                           "exchange": runner.exchange, "exchanges_per_step_per_rank": int(collectives // max(1, args.steps)),
                           "ranks_per_group": shard, "groups": n_groups},
            "bit_identical_to_single_gpu": identical,
            "strong_scaling": {"single_gpu_value_same_job": single_value, "speedup": (value / n_groups / single_value) if single_value else None,
                               "efficiency": (value / n_groups / single_value / shard) if single_value else None,
                               "note": "same job, all views on one GPU (gpm_run, fused sweep), measured on rank 0 in this run"},
            # per-rank roofline (rank 0): its share of the views, its own counters, one GPU's ceilings
            "roofline": roofline_block(W, H, len(mine), iters, sweep_ms / args.steps, n_stage_launches, pairs / args.steps,
                                       fetch_peak, "gpm::k_shard_stage (rank 0: %d of %d views)" % (len(mine), V), None,
                                       FETCHES_PER_PAIR * (3 if args.color else 1)),
            "work": {"hypotheses_evaluated_rank0": hyp // args.steps, "hypotheses_skipped_exact_rank0": skipped // args.steps,
                     "view_samples_all_ranks": int(cnt[1].item() // args.steps)},
            "clocks": clocks,
            "cpu_baseline": {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "timed at N = 1 only"},
        }
    runner.close()
    if outputs is not None:
        dump_outputs(args.dump_outputs, *outputs)
    return line


# ---------------------------------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------------------------------

def run_reference(args, mode, config, shard, rank, world, local):
    """The reference's own gipuma.cu (oracle/_ref), one reference view on rank 0's GPU."""
    if rank != 0:
        return None
    sc = make_scene(args, config, 0, world)
    import torch
    from oracle import pyref
    if not torch.cuda.is_available():
        return {"impl": "reference", "unavailable": "no CUDA device (the reference's implementation of this path is CUDA only)"}
    torch.cuda.set_device(local)
    W, H, V, iters = sc.cols, sc.rows, sc.n_views, sc.params.iterations
    try:
        h = pyref.Harness("ref64" if V > 32 else "ref")
    except Exception as e:      # noqa: BLE001
        return {"impl": "reference", "unavailable": "pinned reference build missing: %r" % (e,)}
    sampler = ClockSampler(local)

    def run_once():
        """(seconds of the reference's timed span, planes, costs)"""
        if args.neighbours == 20:                     # the kernels a reference built without SMALLKERNEL launches
            n4, c, ms = h.run_fused(sc)
            return ms / 1e3, n4, c
        n4, c, printed_s, _ = h.run(sc)
        return printed_s, n4, c

    for _ in range(args.warmup):
        run_once()
    sampler.start()
    printed = wall = 0.0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        printed_s, n4, c = run_once()
        wall += time.perf_counter() - t0
        printed += printed_s
    clocks = sampler.finish()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n4, c)
    units = args.steps * W * H * iters / 1e6
    value = units / printed
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": printed * 1e3 / args.steps, "higher_is_better": True,
        "scaling": "strong" if mode == "view_shard" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, mode, config, shard, world, sc.name, W, H, V, iters, sc.params.box_hsize, sc.params.n_best),
        "arm": {"runs_on": "1 GPU (rank 0): the reference is single-GPU (main.cpp:658-692)",
                "build": "unmodified gipuma.cu, nvcc 12.9 -O3 --use_fast_math sm_100a, pins P1/P2 by macro%s (oracle/build_ref.sh)"
                         % (", P3 costVector[64]" if V > 32 else ""),
                "span": "the reference's own printed 'Total time needed for computation'"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                         "sample": "whole workload on the GPU: the reference has no CPU implementation of this path"},
        "e2e": {"value": units / wall, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "wall clock around the whole main.cpp stand-in call (GlobalState build, texture upload, runcuda, read-back)"},
        "gpu_launches": args.steps * (1 + 6 * iters + 1), "clocks": clocks,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="auto", choices=["auto", "single", "batch", "view_shard", "hybrid"])
    ap.add_argument("--config", type=int, default=0, help="1-5: BASELINE.json configs; 6: 1600x1200 / 60 views (default of view_shard)")
    ap.add_argument("--shard", type=int, default=0, help="hybrid: GPUs per reference view")
    ap.add_argument("--scene", default="smooth", choices=["smooth", "hard"])
    ap.add_argument("--exchange", default="nccl", choices=["nccl", "p2p"],
                    help="sharded modes: one ncclAllGather per exchange stage (default: measured fastest) or the fused peer-memory exchange")
    ap.add_argument("--no-ablation", action="store_true", help="N = 1: skip the extra runs without memo / lower bound / lane order")
    ap.add_argument("--no-check", action="store_true", help="sharded modes: skip the unsharded comparison run on rank 0")
    ap.add_argument("--color", action="store_true", help="float4 images (the reference's -color_processing)")
    ap.add_argument("--neighbours", type=int, default=8, choices=[8, 20],
                    help="20: the fused sweep of a reference built without SMALLKERNEL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the planes and costs of the last timed step (rank 0's reference view) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    rank, world, local = dist_env()
    mode, config, shard = resolve(args, world)
    if args.impl == "reference":
        # rank 0 alone works; the other ranks leave at once (no process group needed)
        line = run_reference(args, mode, config, shard, rank, world, local)
        if rank == 0 and line is not None:
            print(json.dumps(line))
        return
    # the synthetic scene first: its renderer forks worker processes, which must happen before CUDA / NCCL start threads
    if mode in ("view_shard", "hybrid"):
        my_group, _, _, mine, check = sharded_layout(args, config, shard, rank, world)
        sc = make_scene(args, config, my_group, world, positions=None if check else mine)
    else:
        sc = make_scene(args, config, rank if mode == "batch" else 0, world)
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: gipuma_b200 has no CPU fallback"}))
        sys.exit(1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    if mode in ("view_shard", "hybrid"):
        line = run_ours_sharded(args, mode, config, shard, rank, world, local, sc)
    else:
        line = run_ours_single_or_batch(args, mode, config, rank, world, local, sc)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank == 0 and line is not None:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
