"""Benchmark of the north-star metric: batched RRT* plans/s (512x512 worlds, n=5000, r_rewire=50).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--plans P] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: P independent RRT* plans per GPU (world w
seeded 1000+w, one start/goal pair per world, sample stream of plan p = default_rng(p)), i.e. the
sampler kernel + the persistent plan kernel.  N > 1 is launched by torchrun, one rank per GPU;
plans are independent so every rank runs its own P plans (the headline: weak scaling, no data-path
collective; only per-plan statistics are gathered at the end of each step).  Every timed loop that averages over repeated
launches or calls, in every leg below, runs exactly K of them.

`--dump-outputs DIR` writes what the last timed step of the headline computed (dump_outputs): the inputs are fixed by the
seeds above, so two builds run with the same arguments can be compared output for output.

The JSON line carries, besides the contract keys:
  roofline             plan kernel: algorithmic bytes / CUDA-event time against the shared-memory read bandwidth MEASURED in the
                       run (rrtplanner_b200/peaks.py; SURVEY.md section 8(d) names the bound), plus an HBM view
  e2e                  the same metric through the host-buffer C-ABI call rrtk_ctx_plan_worlds2 -- packed grids, descriptors
                       and PCG64 states up, the path record and statistics of every plan down, all inside the timed region;
                       `trees_mode` beside it is the round-1 form (uint8 grids up, every tree down)
  strong_scaling       BASELINE cfg3 as worded: 4096 plans IN TOTAL sharded over the ranks, every step ending with the gather
                       of all path records to rank 0 over NCCL (inside the timed region), checked against a single-GPU run
  cpu_baseline         the oracle's Python/Numba port of the reference on one core, a bounded sample of the same plans;
                       `matches_oracle`: the trees of that sample equal the GPU's bit for bit
  clocks               nvidia-smi samples during the timed region
and, at N = 1, one object per other BASELINE configuration, each with its own roofline / e2e / cpu_baseline / matches_oracle:
  collision_microbench (cfg2, both collision kernels against the measured L2 read bandwidth), informed_bench (cfg4),
  class_api_bench (cfg1), dubins_bench (cfg5; also at N > 1, every rank its own 1024 plans).

`--impl reference` times the reference's CPU algorithm (oracle/rrt_oracle.py: the numpy/Numba port
with the reference's cost profile -- the Python reference itself cannot travel to the GPU box; BASELINE.md
section 4 calibrates the port against the unmodified reference) on all host cores, one plan per process,
on the same worlds / pairs / streams.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W = H = 512
N_ITER = 5000
R_REWIRE = 50.0
METRIC = "RRT* plans/sec (512x512 grid, n=5000)"
NCU_DRAM_BYTES_PER_PLAN = (97265664.0 + 52136192.0) / 1036          # re-captured whenever the plan kernel changes
NCU_DRAM_SOURCE = "profiles/r2_v5_plan_ncu.txt (plan_grid_kernel): 97.27 MB read + 52.14 MB written for 1036 plans"
NCU_CFD_DRAM_BYTES = 45536256.0 + 416000.0
NCU_CFD16_DRAM_BYTES = 67017472.0 + 3128320.0
NCU_CFD16_DRAM_SOURCE = ("profile constant, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this "
                         "launch (profiles/r2_v5_cfd16_ncu.txt, cold L2 as ncu replays it): 16 MB of segment records + 51 MB of the 64 MB of fields, once")
NCU_CFD_DRAM_SOURCE = ("profile constant, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this "
                       "launch (profiles/r2_v5_cfd_ncu.txt, cold L2 as ncu replays it): 16 MB of segment records + 29.5 MB of the 32 MB of fields, once")
WORKLOAD = "cfg3: batched RRTStar, independent 512x512 value-noise worlds, n=5000, r_rewire=50"


# ------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in timed region"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload definition shared by both arms
# ------------------------------------------------------------------------------------------------
def plan_ids(rank: int, plans_per_gpu: int) -> np.ndarray:
    return np.arange(rank * plans_per_gpu, (rank + 1) * plans_per_gpu)


def host_world_and_pair(pid: int):
    """CPU construction of plan pid's inputs (identical to what the GPU arm builds on the device)."""
    from rrtplanner_b200 import worlds
    og = worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(pid)).astype(np.uint8)
    xs, xg = worlds.start_goal(og, pid)
    return og, xs, xg


# ------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------
def _cpu_one(pid: int):
    from oracle import rrt_oracle as O
    og, xs, xg = host_world_and_pair(pid)
    smp = O.sample_stream(og, N_ITER, pid)
    t = time.perf_counter()
    tree = O.plan_star(og, N_ITER, R_REWIRE, xs, xg, smp)
    return time.perf_counter() - t, tree.j, tree.checks, float(tree.vcosts[tree.vgoal])


def _cpu_warm():
    """JIT-compile the two Numba functions before forking / timing (rrt.py:10,183-184 are JIT'd too)."""
    from oracle import rrt_oracle as O
    og = np.zeros((32, 32), dtype=np.uint8)
    O.plan_star(og, 20, 5.0, [1, 1], [20, 20], O.sample_stream(og, 20, 0))


def cpu_baseline_single(nplans: int = 3, gpu_trees=None):
    """Plans 0..nplans-1 of the workload through the oracle's port, one after the other on one core.  `gpu_trees`
    (pts, cost, parent, stats of the timed GPU batch, host arrays) makes the headline self-certifying: the trees the CPU leg
    computes anyway are compared with them bit for bit (`matches_oracle`)."""
    from oracle import rrt_oracle as O
    _cpu_warm()
    dt, checks, ok = 0.0, 0, True
    for pid in range(nplans):
        og, xs, xg = host_world_and_pair(pid)
        smp = O.sample_stream(og, N_ITER, pid)
        t0 = time.perf_counter()
        tree = O.plan_star(og, N_ITER, R_REWIRE, xs, xg, smp)
        dt += time.perf_counter() - t0
        checks += tree.checks
        if gpu_trees is not None:
            pts, cost, parent, stats = gpu_trees
            top = tree.j + (1 if tree.found else 0)
            ok = ok and int(stats[pid, 0]) == tree.j and bool(stats[pid, 2]) == bool(tree.found) and \
                np.array_equal(pts[pid, :tree.j].astype(np.int64), tree.points[:tree.j]) and \
                np.array_equal(cost[pid, :tree.j].view(np.int64), tree.vcosts[:tree.j].view(np.int64)) and \
                all(int(parent[pid, v]) == int(tree.parents[v]) for v in range(1, tree.j))
            if tree.found:
                ok = ok and cost[pid, tree.j].view(np.int64) == np.float64(tree.vcosts[tree.vgoal]).view(np.int64) and top == tree.j + 1
    out = {"value": nplans / dt, "unit": "plans/s", "cores": 1, "kind": "port",
           "sample": f"plans 0..{nplans - 1} of the workload run sequentially with oracle/rrt_oracle.py:plan_star "
                     f"(numpy + Numba port with the reference's per-iteration cost profile), {dt:.1f} s",
           "checks_per_s": checks / dt}
    return out, (bool(ok) if gpu_trees is not None else None)


def reference_arm(args):
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    _cpu_warm()                                  # compile before fork so workers inherit the JIT code
    ctx = mp.get_context("fork")
    per_step = cores
    times = []
    with ctx.Pool(cores) as pool:
        for s in range(args.warmup + args.steps):
            ids = [(s * per_step + k) % 4096 for k in range(per_step)]
            t0 = time.perf_counter()
            recs = pool.map(_cpu_one, ids, chunksize=1)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
                checks = sum(r[2] for r in recs)
    total = sum(times)
    value = per_step * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "plans/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "plans_per_step": per_step,
                   "note": "CPU arm: each step is a bounded sample of the workload, one plan per host core"},
        "cpu_baseline": {"value": value, "unit": "plans/s", "cores": cores, "kind": "port",
                         "sample": f"{per_step} plans per step, one per process on {cores} cores, oracle/rrt_oracle.py:plan_star"},
        "e2e": {"value": value, "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "collision_checks_per_s": checks / times[-1], "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# cfg2: collision-check microbenchmark (BASELINE.json configs[1]; the "collision checks/sec" half of the metric)
# ------------------------------------------------------------------------------------------------
CC_SIZE = 2048
CC_NSEG = 1 << 20


def collision_microbench(local: int, steps: int, warmup: int, cpu: bool, sm_mhz: float, peaks: dict):
    """1 Mi segments with iid uniform integer endpoints (default_rng(0)) on one 2048x2048 value-noise world
    (seed 1000), bit-packed = 512 KB: larger than one SM's shared memory, L2-resident.  Timed with CUDA
    events around `steps` launches of rrtk_collision_segments on torch's current stream."""
    import torch

    from rrtplanner_b200 import _lib, batch, worlds
    dev = torch.device("cuda", local)
    db = batch.DeviceBatch("standard", CC_SIZE, CC_SIZE, 8, device=local).gen_worlds([worlds.world_seed(0)])
    L = db.L
    segs_h = np.random.default_rng(0).integers(0, CC_SIZE, size=(CC_NSEG, 4)).astype(np.int32)
    segs = torch.from_numpy(segs_h).to(dev)
    free = torch.empty((CC_NSEG,), dtype=torch.uint8, device=dev)
    cells = torch.empty((CC_NSEG,), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def launch():
        _lib.check(L.rrtk_collision_segments(db.bits.data_ptr(), CC_SIZE, CC_SIZE, segs.data_ptr(), None, CC_NSEG,
                                             free.data_ptr(), cells.data_ptr(), stream.cuda_stream), "collision_segments")

    for _ in range(max(3, warmup)):
        launch()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = steps
    e0.record(stream)
    for _ in range(reps):
        launch()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    ncells = int(cells.sum(dtype=torch.int64).item())
    nfree = int(free.sum(dtype=torch.int64).item())
    alg = 4.0 * ncells                                          # SURVEY.md 8(d): 4 B per cell the reference would test
    achieved = alg / (ms / 1e3) / 1e9
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    l2_peak = float(peaks["l2_read_GBps"])                      # measured on this device in this run (rrtplanner_b200/peaks.py)
    l2_src = ("measured in this run: rrtk_peak_l2_read, every thread streaming a 64 MB L2-resident buffer with 16-byte loads, best of 5 "
              "(%.0f GB/s; the figure assumed in round 1 was 6300 B/clk x SM clock = %.0f GB/s)" % (l2_peak, 6300.0 * sm_mhz * 1e6 / 1e9))

    def roof(kernel, ms_k, traffic, traffic_src):
        return {"kernel": kernel, "bound": "l2", "achieved": alg / (ms_k / 1e3) / 1e9, "peak": l2_peak, "unit": "GB/s",
                "frac": alg / (ms_k / 1e3) / 1e9 / l2_peak, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": alg,
                "bytes_model": "4 B (one grid word) x cells the reference's walk tests (first hit inclusive)", "peak_source": l2_src}

    bit_grid = {
        "kernel": "rrtk::collision_global_kernel (warp per segment on the tiled bit grid)", "segments_per_s": CC_NSEG / (ms / 1e3),
        "cells_per_s": ncells / (ms / 1e3), "ms_per_launch": ms, "gpu_launches": reps,
        "roofline": roof("rrtk::collision_global_kernel", ms, 17309184.0,
                         "profile constant, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of "
                         "this launch (profiles/r2_v5_cc_ncu.txt): 16 MB of segment records + the 512 KB grid, once"),
    }
    # K1 with the grid staged in shared memory (grids up to ~110 KB of bits: the planner-sized worlds), 512x512 here
    S2 = 512
    db2 = batch.DeviceBatch("standard", S2, S2, 8, device=local).gen_worlds([worlds.world_seed(0)])
    segs2_h = np.random.default_rng(1).integers(0, S2, size=(CC_NSEG, 4)).astype(np.int32)
    segs2 = torch.from_numpy(segs2_h).to(dev)
    free_s, cells_s = torch.empty_like(free), torch.empty_like(cells)

    def launch_shared():
        _lib.check(L.rrtk_collision_segments(db2.bits.data_ptr(), S2, S2, segs2.data_ptr(), None, CC_NSEG, free_s.data_ptr(),
                                             cells_s.data_ptr(), stream.cuda_stream), "collision_segments")

    for _ in range(max(3, warmup)):
        launch_shared()
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(reps):
        launch_shared()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_s = e0.elapsed_time(e1) / reps
    ncells_s = int(cells_s.sum(dtype=torch.int64).item())
    smem_peak = float(peaks["smem_read_GBps"])
    shared_grid = {
        "kernel": "rrtk::collision_shared_kernel (warp per segment, the 32 KB bit grid of one 512x512 world staged in shared memory by one "
                  "cp.async.bulk per block)",
        "workload": "%d random segments on one %dx%d world" % (CC_NSEG, S2, S2),
        "segments_per_s": CC_NSEG / (ms_s / 1e3), "cells_per_s": ncells_s / (ms_s / 1e3), "ms_per_launch": ms_s, "gpu_launches": reps,
        "mean_cells_per_segment": ncells_s / CC_NSEG,
        "roofline": {"kernel": "rrtk::collision_shared_kernel", "bound": "smem", "achieved": 4.0 * ncells_s / (ms_s / 1e3) / 1e9, "peak": smem_peak,
                     "unit": "GB/s", "frac": 4.0 * ncells_s / (ms_s / 1e3) / 1e9 / smem_peak, "traffic": None,
                     "bytes_model": "4 B (one grid word) x cells the reference's walk tests", "peak_source": "measured in this run: rrtk_peak_smem_read"},
    }
    if cpu:
        from oracle import c_oracle                            # checker only
        m2 = 1 << 16
        wf2, wc2 = c_oracle.collision_batch(db2.og[0].cpu().numpy(), segs2_h[:m2])
        shared_grid["matches_oracle"] = bool(np.array_equal(free_s[:m2].cpu().numpy().astype(bool), wf2) and np.array_equal(cells_s[:m2].cpu().numpy(), wc2))
    # K1b: same outputs from the clearance field (built once per grid, outside the timed region like the packing)
    cap = 128
    clear = torch.empty((CC_SIZE, CC_SIZE), dtype=torch.uint8, device=dev)
    scratch = torch.empty((2 * db.words,), dtype=torch.int32, device=dev)
    eb0, eb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eb0.record(stream)
    _lib.check(L.rrtk_clearance_field(db.bits.data_ptr(), 1, CC_SIZE, CC_SIZE, cap, clear.data_ptr(), scratch.data_ptr(), stream.cuda_stream), "clearance_field")
    eb1.record(stream)
    free2 = torch.empty_like(free)
    cells2 = torch.empty_like(cells)

    def launch_cf():
        _lib.check(L.rrtk_collision_segments_cf(clear.data_ptr(), CC_SIZE, CC_SIZE, segs.data_ptr(), None, CC_NSEG, free2.data_ptr(),
                                                cells2.data_ptr(), stream.cuda_stream), "collision_segments_cf")

    for _ in range(max(3, warmup)):
        launch_cf()
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(reps):
        launch_cf()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_cf = e0.elapsed_time(e1) / reps
    iso_field = {
        "kernel": "rrtk::collision_cf_kernel (thread per segment on one uint8 Chebyshev clearance field, cap %d; rrtk_collision_segments_cf)" % cap,
        "segments_per_s": CC_NSEG / (ms_cf / 1e3), "cells_per_s": ncells / (ms_cf / 1e3), "ms_per_launch": ms_cf, "gpu_launches": reps,
        "field_build_ms": eb0.elapsed_time(eb1), "field_bytes": CC_SIZE * CC_SIZE,
        "same_outputs_as_bit_grid_kernel": bool(torch.equal(free, free2) and torch.equal(cells, cells2)),
        "roofline": roof("rrtk::collision_cf_kernel", ms_cf, 20984576.0,
                         "profile constant, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this "
                         "launch (profiles/r2_v5_cf_ncu.txt): 16 MB of segment records + the 4 MB field, once (the 5 MB of results stay in L2)"),
    }
    # K1b on directional fields: one field per octant of the walk (8 bytes per cell), about half the reads per segment
    cap8 = 255
    clear8 = torch.empty((8, CC_SIZE, CC_SIZE), dtype=torch.uint8, device=dev)
    eb0.record(stream)
    _lib.check(L.rrtk_clearance_field_dir(db.bits.data_ptr(), 1, CC_SIZE, CC_SIZE, cap8, clear8.data_ptr(), stream.cuda_stream), "clearance_field_dir")
    eb1.record(stream)
    free3 = torch.empty_like(free)
    cells3 = torch.empty_like(cells)

    def launch_cfd():
        _lib.check(L.rrtk_collision_segments_cfd(clear8.data_ptr(), CC_SIZE, CC_SIZE, segs.data_ptr(), None, CC_NSEG, free3.data_ptr(),
                                                 cells3.data_ptr(), stream.cuda_stream), "collision_segments_cfd")

    for _ in range(max(3, warmup)):
        launch_cfd()
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(reps):
        launch_cfd()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_cfd = e0.elapsed_time(e1) / reps
    # the same with every octant split at slope 1/2: sixteen fields (16 bytes per cell), longer steps again
    clear16 = torch.empty((16, CC_SIZE, CC_SIZE), dtype=torch.uint8, device=dev)
    eb2, eb3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eb2.record(stream)
    _lib.check(L.rrtk_clearance_field_dir16(db.bits.data_ptr(), 1, CC_SIZE, CC_SIZE, cap8, clear16.data_ptr(), stream.cuda_stream), "clearance_field_dir16")
    eb3.record(stream)
    free4 = torch.empty_like(free)
    cells4 = torch.empty_like(cells)

    def launch_cfd16():
        _lib.check(L.rrtk_collision_segments_cfd16(clear16.data_ptr(), CC_SIZE, CC_SIZE, segs.data_ptr(), None, CC_NSEG, free4.data_ptr(),
                                                   cells4.data_ptr(), stream.cuda_stream), "collision_segments_cfd16")

    for _ in range(max(3, warmup)):
        launch_cfd16()
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(reps):
        launch_cfd16()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_cfd16 = e0.elapsed_time(e1) / reps
    octants = {
        "kernel": "rrtk::collision_cf_kernel on eight directional uint8 clearance fields, one per octant of the walk (rrtk_clearance_field_dir + "
                  "rrtk_collision_segments_cfd), cap %d" % cap8,
        "segments_per_s": CC_NSEG / (ms_cfd / 1e3), "cells_per_s": ncells / (ms_cfd / 1e3), "ms_per_launch": ms_cfd, "gpu_launches": reps,
        "field_build_ms": eb0.elapsed_time(eb1), "field_bytes": 8 * CC_SIZE * CC_SIZE,
        "same_outputs_as_bit_grid_kernel": bool(torch.equal(free, free3) and torch.equal(cells, cells3)),
        "roofline": roof("rrtk::collision_cf_kernel", ms_cfd, NCU_CFD_DRAM_BYTES, NCU_CFD_DRAM_SOURCE),
    }
    out = {
        "workload": "cfg2: %d random segments on one %dx%d bit-packed world (512 KB, L2-resident)" % (CC_NSEG, CC_SIZE, CC_SIZE),
        "mean_cells_per_segment": ncells / CC_NSEG, "free_fraction": nfree / CC_NSEG,
        "obstacle_fraction": float(db.og.float().mean().item()),
        # the fastest of the kernels carries the leg's headline numbers; each is listed with its own roofline object
        "kernel": "rrtk::collision_cf_kernel (thread per segment on sixteen directional uint8 clearance fields: the octants of the walk split at "
                  "slope 1/2, cap %d; rrtk_clearance_field_dir16 + rrtk_collision_segments_cfd16)" % cap8,
        "segments_per_s": CC_NSEG / (ms_cfd16 / 1e3), "cells_per_s": ncells / (ms_cfd16 / 1e3), "ms_per_launch": ms_cfd16, "gpu_launches": reps,
        "field_build_ms": eb2.elapsed_time(eb3), "field_bytes": 16 * CC_SIZE * CC_SIZE,
        "same_outputs_as_bit_grid_kernel": bool(torch.equal(free, free4) and torch.equal(cells, cells4)),
        "roofline": roof("rrtk::collision_cf_kernel", ms_cfd16, NCU_CFD16_DRAM_BYTES, NCU_CFD16_DRAM_SOURCE),
        "note": "a clearance-field walk skips the cells the field proves free, so it reads far fewer bytes than the algorithmic 4 B x cells the "
                "reference would test (about 4 scattered byte reads per segment here, 5 on the eight octant fields, 10 on the isotropic field); "
                "what bounds it is the rate of scattered L1 reads (~1.08 cycles per lane-load per SM, scripts/micro/scatter.cu) and the slowest "
                "lane of each warp",
        "octant_fields_kernel": octants,
        "isotropic_field_kernel": iso_field,
        "bit_grid_kernel": bit_grid,
        "shared_grid_kernel": shared_grid,
    }
    if cpu:
        from oracle import c_oracle                            # checker + CPU baseline only
        m = 1 << 17
        og_h = db.og[0].cpu().numpy()
        c_oracle.collision_batch(og_h, segs_h[:1024])
        t0 = time.perf_counter()
        wf, wc = c_oracle.collision_batch(og_h, segs_h[:m])
        dt = time.perf_counter() - t0
        out["matches_oracle"] = bool(np.array_equal(free[:m].cpu().numpy().astype(bool), wf) and np.array_equal(cells[:m].cpu().numpy(), wc))
        out["cpu_baseline"] = {"value": m / dt, "unit": "segments/s", "cores": 1, "kind": "port",
                               "sample": "first %d segments through oracle/rrt_oracle.c:orc_collision_batch (compiled C walk of "
                                         "rrt.py:183-229 on the uint8 grid), %.3f s" % (m, dt)}
    return out


# ------------------------------------------------------------------------------------------------
# cfg4: RRTStarInformed, 1024 start/goal pairs on one 1024x1024 world, n=20000 (BASELINE.json configs[3])
# ------------------------------------------------------------------------------------------------
INF_SIZE, INF_PLANS, INF_N, INF_RGOAL = 1024, 1024, 20000, 5.0


def informed_bench(local: int, steps: int, cpu: bool, peaks: dict, plans: int = INF_PLANS):
    """One 1024x1024 value-noise world (seed 1000), `plans` start/goal pairs (device sampler, seed 2000+p), n = 20000,
    r_rewire = 50, r_goal = 5; free-space stream of plan p = default_rng(p); the unit-disc points of the ellipse phase are
    pre-generated per plan (default_rng(7).uniform, SURVEY.md 8(d)) and the rotations come from the reference's own numpy
    construction (rrt.py:601-613).  Device arm with CUDA events, end to end through rrtk_ctx_plan_worlds2 (bit grid, states and
    unit-disc streams up; path records down), two plans against the C oracle."""
    import torch

    from rrtplanner_b200 import _lib, batch, worlds
    from rrtplanner_b200.rrt import RRTStarInformed
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)
    S, n, P = INF_SIZE, INF_N, plans
    db = batch.DeviceBatch("informed", S, S, n, R_REWIRE, INF_RGOAL, device=local).gen_worlds([worlds.world_seed(0)])
    pair = batch.DeviceBatch("star", S, S, 8, device=local)
    pair.bits, pair.rowcum = db.bits, db.rowcum
    pair.set_plans(batch.make_desc(np.zeros(P, int), np.zeros((P, 2)), np.zeros((P, 2))))
    pair.seed_samples(2000 + np.arange(P))
    d = pair.samples.cpu().numpy().astype(np.int64)
    starts = d[:, 0]
    differs = (d[:, 1:] != starts[:, None]).any(axis=2)
    goals = d[np.arange(P), 1 + differs.argmax(axis=1)]
    og = db.og[0].cpu().numpy()
    helper = RRTStarInformed(og, 8, R_REWIRE, INF_RGOAL, pbar=False)
    rots = np.stack([np.asarray(helper.rotation_to_world_frame(a, b), dtype=np.float64) for a, b in zip(starts, goals)])
    desc = batch.make_desc(np.zeros(P, int), starts, goals, rots)
    db.set_plans(desc)
    db.seed_samples(np.arange(P))
    u = np.random.default_rng(7).uniform(0, 1, size=(P, n, 2))
    balls = np.stack([np.sqrt(u[..., 0]) * np.cos(2 * np.pi * u[..., 1]), np.sqrt(u[..., 0]) * np.sin(2 * np.pi * u[..., 1])], axis=-1)
    db.set_balls_host(balls)
    for _ in range(2):
        db.run()
    torch.cuda.synchronize(dev)
    reps = steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        db.run()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    st = db.out["stats"].cpu().numpy()
    Sx = {nm: st[:, i].astype(np.float64) for i, nm in enumerate(_lib.STAT_NAMES)}
    alg = 8.0 * Sx["nn_pairs"].sum() + 8.0 * Sx["ring_members"].sum() + 4.0 * Sx["cells"].sum()
    smem_b, blocks = db.footprint()
    out = {"workload": "cfg4: RRTStarInformed, one %dx%d world, %d start/goal pairs, n=%d, r_rewire=%g, r_goal=%g" % (S, S, P, n, R_REWIRE, INF_RGOAL),
           "plans_per_s": P / (ms / 1e3), "ms_per_launch": ms, "gpu_launches": reps, "goal_found_frac": float(st[:, 2].mean()),
           "solution_found_frac": float((st[:, 5] >= 0).mean()),
           "mean_first_solution_iter": float(st[st[:, 5] >= 0, 5].mean()) if (st[:, 5] >= 0).any() else None,
           "ellipse_iter_frac": float(st[:, 6].mean() / n), "mean_vertices": float(st[:, 0].mean()),
           "kernel": "rrtk::plan_scan_kernel<RRTK_INFORMED, K=8, T=256>", "blocks_per_sm": blocks, "smem_bytes_per_block": smem_b,
           "roofline": {"bound": "smem", "achieved": alg / (ms / 1e3) / 1e9, "peak": peaks["smem_read_GBps"], "unit": "GB/s",
                        "frac": alg / (ms / 1e3) / 1e9 / peaks["smem_read_GBps"], "traffic": None,
                        "algorithmic_bytes_per_launch": alg, "peak_source": "measured in this run (rrtk_peak_smem_read)",
                        "bytes_model": "8 B x (iteration, filled vertex) pairs + 8 B x radius-set members + 4 B x grid cells tested"}}
    # end to end: one packed grid, descriptors, PCG64 states and the unit-disc streams up; path records + statistics down
    ctx = _lib.Context()
    bits_host = _lib.pack_grids_host(og[None])
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()          # noqa: E731
    balls_pin, states = pin(balls), batch.seed_states(np.arange(P))
    best = None
    for rep in range(2):
        t0 = time.perf_counter()
        got = ctx.plan_worlds2(_lib.KIND_INFORMED, bits_host, S, S, desc, n, R_REWIRE, INF_RGOAL, states=states, balls=balls_pin, bits=True,
                               trees=False, paths=True, path_cap=PATH_CAP)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    ctx.close()
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    out["e2e"] = {"value": P / best, "unit": "plans/s", "h2d_bytes_per_step": int(bits_host.nbytes + P * (64 + 32 + n * 16)),
                  "d2h_bytes_per_step": int(P * (PATH_CAP * 8 + 12 + _lib.STAT_COUNT * 8)),
                  "api": "rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS), seed mode + unit-disc streams from pinned host memory",
                  "matches_device_arm": bool(np.array_equal(got["stats"][:, keep], st[:, keep]))}
    if cpu:
        from oracle import c_oracle                            # checker + CPU baseline only
        res = db.download()
        smp = db.samples.cpu().numpy()
        ok, dt, m = True, 0.0, 2
        for p in range(m):
            t0 = time.perf_counter()
            wp, wc, wpar, wst, _ = c_oracle.plan_raw("informed", og, n, starts[p], goals[p], smp[p], R_REWIRE, INF_RGOAL, balls[p], rots[p])
            dt += time.perf_counter() - t0
            top = wst["j"] + (1 if wst["found"] else 0)
            ok = ok and int(res.stats[p, 0]) == wst["j"] and np.array_equal(res.pts[p, :top], wp[:top]) and \
                np.array_equal(res.parent[p, :top], wpar[:top]) and np.array_equal(res.cost[p, :top].view(np.int64), wc[:top].view(np.int64))
        out["matches_oracle"] = bool(ok)
        out["cpu_baseline"] = {"value": m / dt, "unit": "plans/s", "cores": 1, "kind": "port",
                               "sample": "plans 0..%d of the workload through oracle/rrt_oracle.c:orc_plan (compiled C restatement of rrt.py:690-748; "
                                         "far faster than the Python reference), %.2f s" % (m - 1, dt)}
    return out


# ------------------------------------------------------------------------------------------------
# cfg1: one RRTStar plan through the drop-in class (BASELINE.json configs[0], the reference's own CPU-runnable case)
# ------------------------------------------------------------------------------------------------
def class_api_bench(steps: int, cpu: bool):
    """RRTStar(og, n=1000, r_rewire=50, seed=0).plan() on a 256x256 world, `steps` calls timed around the public call including
    the networkx graph it returns -- the latency a user of the reference's API sees (the reference: about 0.6 s, SURVEY.md 6)."""
    from rrtplanner_b200 import rrt, worlds
    og = worlds.perlin_occupancygrid(256, 256, seed=worlds.world_seed(0))
    xs, xg = worlds.start_goal(og, 0)
    pl = rrt.RRTStar(og, 1000, 50.0, pbar=False, seed=0)
    pl.plan(xs, xg)
    reps = steps
    t0 = time.perf_counter()
    for _ in range(reps):
        pl = rrt.RRTStar(og, 1000, 50.0, pbar=False, seed=0)
        T, gv = pl.plan(xs, xg)
    dt = (time.perf_counter() - t0) / reps
    out = {"workload": "cfg1: RRTStar(og 256x256, n=1000, r_rewire=50, seed=0).plan(), class API incl. set-up of the grid on the device and "
                       "the networkx graph", "s_per_plan": dt, "plans_per_s": 1 / dt, "nodes": T.number_of_nodes(), "gpu_launches": 3 * reps,
           "e2e": {"value": 1 / dt, "unit": "plans/s", "h2d_bytes_per_step": int(256 * 256 + 64 + 1000 * 4),
                   "d2h_bytes_per_step": int(1001 * 16 + 96), "api": "rrtplanner_b200.RRTStar(...).plan(xstart, xgoal)"}}
    if cpu:
        from oracle import rrt_oracle as O                     # checker + CPU baseline only
        _cpu_warm()
        smp = O.sample_stream(og, 1000, 0)
        t0 = time.perf_counter()
        tree = O.plan_star(og, 1000, 50.0, xs, xg, smp)
        dtc = time.perf_counter() - t0
        pts = np.stack([np.asarray(T.nodes[v]["pt"]) for v in range(tree.j)])
        par = {int(b): int(a) for a, b in T.edges}
        ok = int(gv) == int(tree.vgoal) and np.array_equal(pts, tree.points[: tree.j]) and \
            all(par[v] == int(tree.parents[v]) for v in range(1, tree.j)) and \
            all(T.edges[par[v], v]["cost"] == tree.vcosts[v] for v in range(1, tree.j))
        out["matches_oracle"] = bool(ok)
        out["cpu_baseline"] = {"value": 1 / dtc, "unit": "plans/s", "cores": 1, "kind": "port",
                               "sample": "the same plan through oracle/rrt_oracle.py:plan_star (numpy + Numba port), %.2f s" % dtc}
    return out


# ------------------------------------------------------------------------------------------------
# cfg5: Dubins-vehicle RRT* (BASELINE.json configs[4]); no reference code exists for it -- parity UNPINNED
# ------------------------------------------------------------------------------------------------
DUB_PLANS, DUB_NH, DUB_RHO, DUB_DS = 1024, 16, 6.0, 1.0


def dubins_bench(local: int, steps: int, cpu: bool, plans: int = DUB_PLANS, threads: int = 0, rank: int = 0, world: int = 1):
    """1024 Dubins RRT* plans (rewire on) on independent 512x512 worlds, n=5000, r=50, 16 headings, rho=6, ds=1;
    sample cells from the device PCG64 stream of plan p, headings = default_rng(7000+p).integers(0, 16, n) (host).
    Also times the same shape with the Euclidean model + rewire (the RRT* the reference's rewire block intends).
    With world > 1 every rank runs its own `plans` plans (ids rank * plans ...: weak scaling, no collective in the path);
    the time is the maximum over the ranks and only the device arm is measured."""
    import torch

    from rrtplanner_b200 import _lib, batch, worlds
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)
    ids = rank * plans + np.arange(plans)
    out = {"workload": "cfg5: %d Dubins RRT* plans (choose-parent + rewire), independent %dx%d worlds, n=%d, r_rewire=%g, "
                       "%d headings, rho=%g cells, ds=%g" % (plans, W, H, N_ITER, R_REWIRE, DUB_NH, DUB_RHO, DUB_DS),
           "parity": "UNPINNED: the reference ships no Dubins code; bit-exact against this project's specification oracle/rewire_oracle.c"}
    keep = {}
    for model in ("dubins", "euclid"):
        db = batch.DeviceBatch2(model, W, H, N_ITER, r_rewire=R_REWIRE, nheadings=DUB_NH, rho=DUB_RHO, ds=DUB_DS, device=local,
                                threads=threads)
        db.gen_worlds([worlds.world_seed(int(p)) for p in ids])
        pair_db = batch.DeviceBatch("star", W, H, 8, device=local)
        pair_db.bits, pair_db.rowcum = db.bits, db.rowcum
        pair_db.set_plans(batch.make_desc(np.arange(plans), np.zeros((plans, 2)), np.zeros((plans, 2))))
        pair_db.seed_samples(2000 + ids)
        draws = pair_db.samples.cpu().numpy().astype(np.int64)
        starts = draws[:, 0]
        differs = (draws[:, 1:] != starts[:, None]).any(axis=2)
        goals = draws[np.arange(plans), 1 + differs.argmax(axis=1)]
        hs = np.random.default_rng(6000).integers(0, DUB_NH, size=(plans, 2))
        db.set_plans(batch.make_desc2(np.arange(plans), np.concatenate([starts, hs[:, :1]], axis=1),
                                      np.concatenate([goals, hs[:, 1:]], axis=1)))
        db.seed_samples(ids)
        if model == "dubins":
            db.seed_heads(7000 + ids)
        for _ in range(2):
            db.run()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = steps
        e0.record(stream)
        for _ in range(reps):
            db.run()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / reps
        if world > 1:
            import torch.distributed as dist
            tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
        st = db.out["stats"].cpu().numpy()
        smem, blocks = db.footprint()
        rec = {"plans_per_s": plans * world / (ms / 1e3), "n_gpus": world, "plans_per_gpu": plans, "ms_per_launch": ms, "gpu_launches": reps, "mean_vertices": float(st[:, 0].mean()),
               "goal_found_frac": float(st[:, 2].mean()), "rewires_per_plan": float(st[:, 5].mean()),
               "edge_length_evals_per_s": float(st[:, 8].sum()) / (ms / 1e3), "edge_tests_per_s": float(st[:, 3].sum()) / (ms / 1e3),
               "smem_bytes_per_block": smem, "blocks_per_sm": blocks, "overflow": int(st[:, 9].sum()),
               "kernel": "rrtk::plan_rewire_kernel<%s, T=%d>" % (model.upper(), threads or 256)}
        if world > 1:
            out["dubins_rrtstar" if model == "dubins" else "euclid_rrtstar_with_rewire"] = rec
            continue
        # end to end through the host-buffer C ABI: grids, descriptors, PCG64 states and headings up, every tree down
        ctx = _lib.Context()
        og_pin = torch.empty(tuple(db.og.shape), dtype=torch.uint8, pin_memory=True)
        og_pin.copy_(db.og)
        torch.cuda.synchronize(dev)
        og_host = og_pin.numpy()
        out_pin = tuple(torch.empty(shape, dtype=dt, pin_memory=True).numpy() for shape, dt in (
            ((plans, N_ITER + 1, 2), torch.int16), ((plans, N_ITER + 1), torch.uint8), ((plans, N_ITER + 1), torch.float64),
            ((plans, N_ITER + 1), torch.float64), ((plans, N_ITER + 1), torch.int32), ((plans, _lib.STAT_COUNT), torch.int64)))
        desc_h = batch.make_desc2(np.arange(plans), np.concatenate([starts, hs[:, :1]], axis=1), np.concatenate([goals, hs[:, 1:]], axis=1))
        heads_h = db.heads.cpu().numpy() if model == "dubins" else None
        t_best = None
        for rep in range(2):
            t0 = time.perf_counter()
            ctx.set_grids(og_host)
            r_host = ctx.plan2(db.cfg, desc_h, N_ITER, states=batch.seed_states(ids), heads=heads_h, out=out_pin)
            dt = time.perf_counter() - t0
            t_best = dt if t_best is None else min(t_best, dt)
        # the pipelined form: packed grids, descriptors, PCG64 states and headings up; path records + statistics down
        cap = PATH_CAP
        bits_pin = torch.empty(tuple(db.bits.shape), dtype=db.bits.dtype, pin_memory=True)
        bits_pin.copy_(db.bits)
        torch.cuda.synchronize(dev)
        bits_host = bits_pin.numpy().view(np.uint32).reshape(plans, -1)
        out2 = {k: torch.empty(shape, dtype=dt, pin_memory=True).numpy() for k, shape, dt in (
            ("stats", (plans, _lib.STAT_COUNT), torch.int64), ("path", (plans, cap), torch.int32), ("xy", (plans, cap, 2), torch.int16),
            ("path_head", (plans, cap), torch.uint8), ("len", (plans,), torch.int32), ("path_cost", (plans,), torch.float64))}
        states_h = batch.seed_states(ids)
        t_pipe = None
        for rep in range(3):
            t0 = time.perf_counter()
            r2 = ctx.plan2_worlds(db.cfg, bits_host, W, H, desc_h, N_ITER, states=states_h, heads=heads_h, bits=True, trees=False, paths=True,
                                  path_cap=cap, out=out2)
            dt = time.perf_counter() - t0
            t_pipe = dt if t_pipe is None or rep == 1 else min(t_pipe, dt)        # the first call allocates the pipeline's buffers
        ctx.close()
        st_dev = db.out["stats"].cpu().numpy()
        rec["e2e"] = {"value": plans / t_pipe, "unit": "plans/s",
                      "api": "rrtk_ctx_plan2_worlds (packed grids in, seed mode, path records out; chunks of one plan per SM, five plan streams), pinned host buffers",
                      "h2d_bytes_per_step": int(plans * (bits_host.shape[1] * 4 + 64 + 32 + (N_ITER if model == "dubins" else 0))),
                      "d2h_bytes_per_step": int(plans * (cap * 9 + 12 + _lib.STAT_COUNT * 8)),
                      "matches_device_arm": bool(np.array_equal(r2["stats"][:, :3], st_dev[:, :3])),
                      "trees_mode": {"value": plans / t_best, "unit": "plans/s",
                                     "api": "rrtk_ctx_set_grids + rrtk_ctx_plan2 (uint8 grids up, every tree down), not pipelined",
                                     "h2d_bytes_per_step": int(plans * (W * H + 64 + 32 + (N_ITER if model == "dubins" else 0))),
                                     "d2h_bytes_per_step": int(plans * ((N_ITER + 1) * 25 + _lib.STAT_COUNT * 8)),
                                     "matches_device_arm": bool(np.array_equal(r_host[4], db.out["parent"].cpu().numpy()))}}
        out["dubins_rrtstar" if model == "dubins" else "euclid_rrtstar_with_rewire"] = rec
        keep[model] = (db, starts, goals, hs)
    if cpu and world == 1:
        from oracle import rewire_oracle as O2                # checker + CPU baseline only
        for model, key in (("dubins", "dubins_rrtstar"), ("euclid", "euclid_rrtstar_with_rewire")):
            db, starts, goals, hs = keep[model]
            res = db.download()
            ok, dt, m = True, 0.0, 4
            for p in range(m):
                og = db.og[p].cpu().numpy()
                smp = db.samples[p].cpu().numpy().astype(np.int64)
                hd = db.heads[p].cpu().numpy().astype(np.int64) if model == "dubins" else np.zeros(N_ITER, dtype=np.int64)
                t0 = time.perf_counter()
                want = O2.plan(model, og, N_ITER, [*starts[p], hs[p, 0]], [*goals[p], hs[p, 1]], np.concatenate([smp, hd[:, None]], axis=1),
                               star=True, rewire=True, r_rewire=R_REWIRE, nh=DUB_NH, rho=DUB_RHO, ds=DUB_DS)
                dt += time.perf_counter() - t0
                top = want["stats"]["j"] + want["stats"]["found"]
                ok = ok and np.array_equal(res.parent[p, :top], want["parent"][:top]) and \
                    np.array_equal(res.cost[p, :top].view(np.int64), want["cost"][:top].view(np.int64))
            out[key]["matches_oracle"] = bool(ok)
            out[key]["cpu_baseline"] = {"value": m / dt, "unit": "plans/s", "cores": 1, "kind": "port",
                                        "sample": "plans 0..%d of the workload through oracle/rewire_oracle.c (compiled C), %.2f s" % (m - 1, dt)}
    return out


# ------------------------------------------------------------------------------------------------
# shared set-up of a cfg3 batch: worlds made on the device, start/goal pairs from the device sampler
# ------------------------------------------------------------------------------------------------
def cfg3_batch(local: int, ids: np.ndarray, threads: int = 0):
    """DeviceBatch with world / pair / descriptor of the plans `ids` resident in HBM.  World of plan p = seed 1000+p;
    start/goal of plan p = first two distinct draws of free[default_rng(2000+p).integers(nfree)] (worlds.start_goal),
    produced with the device sampler so no grid has to visit the host."""
    import torch

    from rrtplanner_b200 import batch, worlds
    P = len(ids)
    db = batch.DeviceBatch("star", W, H, N_ITER, R_REWIRE, device=local, threads=threads)
    db.gen_worlds([worlds.world_seed(int(p)) for p in ids])
    pair_db = batch.DeviceBatch("star", W, H, 8, device=local)
    pair_db.bits, pair_db.rowcum = db.bits, db.rowcum
    pair_db.set_plans(batch.make_desc(np.arange(P), np.zeros((P, 2)), np.zeros((P, 2))))
    pair_db.seed_samples(2000 + ids)
    draws = pair_db.samples.cpu().numpy().astype(np.int64)
    starts = draws[:, 0]
    differs = (draws[:, 1:] != starts[:, None]).any(axis=2)
    goals = draws[np.arange(P), 1 + differs.argmax(axis=1)]
    desc = batch.make_desc(np.arange(P), starts, goals)
    db.set_plans(desc)
    dev = torch.device("cuda", local)
    states = torch.from_numpy(batch.seed_states(ids).view(np.int64)).to(dev)
    db.samples = torch.empty((P, N_ITER, 2), dtype=torch.int16, device=dev)
    return db, desc, states, starts, goals


# ------------------------------------------------------------------------------------------------
# strong scaling: BASELINE cfg3 as worded -- 4096 worlds in total, sharded over the ranks, paths gathered
# ------------------------------------------------------------------------------------------------
STRONG_PLANS, PATH_CAP = 4096, 256


def strong_leg(local: int, rank: int, world: int, steps: int, warmup: int, barrier, total: int = STRONG_PLANS):
    """Fixed total work: `total` plans, rank r runs batch.shard(total, r, world); every step ends with the final gather
    the north star names -- the path record of every plan (vertex ids, points, length, cost: what route2gv /
    vertices_as_ndarray give the reference's caller, rrt.py:87-129) and its statistics row -- to rank 0 with one
    torch.distributed.gather per field on the device (NCCL over NVLink), inside the timed region.  Rank 0 then re-runs
    all `total` plans alone (untimed) and checks that the gathered records are the ones a single GPU computes."""
    import torch
    import torch.distributed as dist

    from rrtplanner_b200 import _lib, batch, multigpu
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)
    ids = np.asarray(list(batch.shard(total, rank, world)), dtype=np.int64)
    db, _, states, _, _ = cfg3_batch(local, ids)
    L, P = db.L, len(ids)

    def step():
        _lib.check(L.rrtk_sample_streams(db.bits.data_ptr(), db.rowcum.data_ptr(), W, H, db.desc.data_ptr(), P, states.data_ptr(),
                                         N_ITER, db.samples.data_ptr(), stream.cuda_stream), "sample_streams")
        db.run()
        rec = db.path_records(PATH_CAP)
        return multigpu.gather_tensors(rec, total, dst=0) if world > 1 else rec

    for _ in range(max(1, warmup)):
        got = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        got = step()
    e1.record(stream)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    if rank != 0:
        return None
    rec_bytes = PATH_CAP * 4 + PATH_CAP * 4 + 4 + 8 + _lib.STAT_COUNT * 8
    out = {"scaling": "strong", "plans_total": total, "plans_per_gpu": int(np.ceil(total / world)), "value": total / (ms / 1e3),
           "unit": "plans/s", "ms_per_step": ms,
           "gather": {"what": "path vertex ids + points (cap %d), path length, path cost, statistics row of every plan" % PATH_CAP,
                      "bytes_per_plan": rec_bytes, "bytes_to_rank0_per_step": int(rec_bytes * (total - P)),
                      "transport": "torch.distributed.gather on device tensors (NCCL)" if world > 1 else "none (one rank)",
                      "inside_timed_region": True},
           "long_paths": int((got["len"] > PATH_CAP).sum().item())}
    if world > 1:
        # the same `total` plans on this GPU alone: the gathered records must be bit-identical
        full, _, fstates, _, _ = cfg3_batch(local, np.arange(total, dtype=np.int64))
        _lib.check(L.rrtk_sample_streams(full.bits.data_ptr(), full.rowcum.data_ptr(), W, H, full.desc.data_ptr(), total, fstates.data_ptr(),
                                         N_ITER, full.samples.data_ptr(), stream.cuda_stream), "sample_streams")
        full.run()
        want = full.path_records(PATH_CAP)
        # rows longer than the cap are left unwritten by design: compare the defined part
        # (the two walk counters of the statistics row depend on how the warps of a block interleave in the goal search -- a shared
        #  bound prunes candidates -- and are left out, as in the parity tests)
        keep = torch.tensor([i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")], device=dev)
        ok = all(bool(torch.equal(got[k], want[k])) for k in ("len", "path_cost")) and bool(torch.equal(got["stats"][:, keep], want["stats"][:, keep]))
        short = want["len"] <= PATH_CAP
        ok = ok and bool(torch.equal(got["path"][short], want["path"][short])) and bool(torch.equal(got["xy"][short], want["xy"][short]))
        out["gathered_equals_single_gpu_run"] = ok
    else:
        out["gathered_equals_single_gpu_run"] = True     # one rank: the records are the single-GPU run
    return out


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed, for comparing two builds output for output
# ------------------------------------------------------------------------------------------------
DUMP_PLANS = 256          # trees of 256 plans at n = 5000: 25.6 MB
# statistics that are results of a plan; checks / cells depend on how the warps of a block interleave in the goal search and
# nn_pairs on which form of the plan kernel answers the nearest query, so they are left out
DUMP_STATS = ("j", "vgoal", "found", "first_solution_iter", "ellipse_iters", "accepted", "ring_members")


def dump_outputs(out_dir: str, out: dict):
    """Write the trees of a fixed sample of plans (default_rng(0), at most DUMP_PLANS, ascending plan index) and the result
    statistics of every plan as DIR/<name>.npy: plan_index, pts (float32), cost (float64), parent (float32; ids < 2**24),
    stat_<name> (float64).  Every value written is finite: the unfilled rows of a tree (row >= j + found) keep the fill values
    of pts (-32768) and parent (-1), and their cost, inf in the library's layout, is written as -1 (a real cost is >= 0)."""
    import torch

    from rrtplanner_b200 import _lib
    P = out["stats"].shape[0]
    sel = np.sort(np.random.default_rng(0).choice(P, size=min(P, DUMP_PLANS), replace=False))
    idx = torch.from_numpy(sel).to(out["pts"].device)
    stats = out["stats"].cpu().numpy()
    cost = out["cost"].index_select(0, idx).cpu().numpy()
    top = stats[sel, _lib.STAT_NAMES.index("j")] + (stats[sel, _lib.STAT_NAMES.index("found")] != 0)
    cost[np.arange(cost.shape[1])[None, :] >= top[:, None]] = -1.0
    arrays = {"plan_index": sel.astype(np.float64),
              "pts": out["pts"].index_select(0, idx).cpu().numpy().astype(np.float32),
              "cost": cost,
              "parent": out["parent"].index_select(0, idx).cpu().numpy().astype(np.float32)}
    for name in DUMP_STATS:
        arrays["stat_" + name] = stats[:, _lib.STAT_NAMES.index(name)].astype(np.float64)
    for name, a in arrays.items():
        if not np.isfinite(a).all():
            raise RuntimeError(f"--dump-outputs: {name} of the last timed step holds a non-finite value")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def gpu_arm(args):
    import torch
    import torch.distributed as dist

    from rrtplanner_b200 import _lib, batch, worlds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if _lib.lib().rrtk_device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    P = args.plans
    ids = plan_ids(rank, P)

    # ---- setup (untimed): worlds, pairs, descriptors resident in HBM -------------------------
    db, desc, states, starts, goals = cfg3_batch(local, ids, args.threads)
    L = db.L
    stream = torch.cuda.current_stream(dev)

    def step():
        _lib.check(L.rrtk_sample_streams(db.bits.data_ptr(), db.rowcum.data_ptr(), W, H, db.desc.data_ptr(), P, states.data_ptr(),
                                         N_ITER, db.samples.data_ptr(), stream.cuda_stream), "sample_streams")
        db.run()

    gathered = [torch.empty_like(db.out["stats"]) for _ in range(world)] if (world > 1 and rank == 0) else None

    def gather_stats():
        if world > 1:
            dist.gather(db.out["stats"], gathered, dst=0)

    for _ in range(args.warmup):
        step()
        gather_stats()
    barrier()

    # ---- timed region: exactly K steps, CUDA events on the launching stream -----------------
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_begin.record(stream)
    for k in range(args.steps):
        ev[k][0].record(stream)
        _lib.check(L.rrtk_sample_streams(db.bits.data_ptr(), db.rowcum.data_ptr(), W, H, db.desc.data_ptr(), P, states.data_ptr(),
                                         N_ITER, db.samples.data_ptr(), stream.cuda_stream), "sample_streams")
        ev[k][1].record(stream)
        db.run()
        ev[k][2].record(stream)
        gather_stats()
    e_end.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    clocks = sampler.stop(t_wall0, t_wall1)
    ms_total = e_begin.elapsed_time(e_end)
    ms_sampler = float(np.mean([ev[k][0].elapsed_time(ev[k][1]) for k in range(args.steps)]))
    ms_plan = float(np.mean([ev[k][1].elapsed_time(ev[k][2]) for k in range(args.steps)]))
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())

    stats = db.out["stats"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, db.out)
    S = {n: stats[:, i] for i, n in enumerate(_lib.STAT_NAMES)}
    if world > 1 and rank == 0:
        all_stats = torch.stack(gathered).cpu().numpy().reshape(-1, _lib.STAT_COUNT)
    else:
        all_stats = stats

    # ---- the same K steps issued on two alternating streams with their own sample / output buffers ----
    # A batch of 4096 plans occupies 1036 plan slots 3.95 times over; while its last plans finish, the slots that are already free
    # wait for the next launch (the headline above: one stream, ~16 % of the slot-time idle in that ramp-down).  A caller that
    # plans batch after batch can let the next batch start in that shadow.  Reported beside the headline, not instead of it.
    overlapped = None
    if not args.plan_only:
        import copy as _copy
        sides = []
        for i in range(2):
            d2 = _copy.copy(db)                       # shares worlds, bit grids, descriptors; own samples and outputs
            d2.samples = torch.empty_like(db.samples)
            d2.out = {k: (torch.empty_like(v) if v is not None else None) for k, v in db.out.items()}
            sides.append((d2, torch.cuda.Stream(device=dev)))

        def ov_step(i):
            d2, st2 = sides[i & 1]
            with torch.cuda.stream(st2):
                _lib.check(L.rrtk_sample_streams(d2.bits.data_ptr(), d2.rowcum.data_ptr(), W, H, d2.desc.data_ptr(), P, states.data_ptr(),
                                                 N_ITER, d2.samples.data_ptr(), st2.cuda_stream), "sample_streams")
                d2.run()

        for i in range(4):
            ov_step(i)
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record(stream)
        for _, st2 in sides:
            st2.wait_stream(stream)
        for i in range(args.steps):
            ov_step(i)
        for _, st2 in sides:
            stream.wait_stream(st2)
        o1.record(stream)
        barrier()
        tov = torch.tensor([o0.elapsed_time(o1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tov, op=dist.ReduceOp.MAX)
        same_ov = all(bool(torch.equal(sides[i][0].out["parent"], db.out["parent"])) for i in range(2))
        overlapped = {"value": P * world * args.steps / (float(tov.item()) / 1e3), "unit": "plans/s", "ms_per_step": float(tov.item()) / args.steps,
                      "how": "the same %d steps on two alternating CUDA streams, each with its own sample and output buffers, so that the ramp-down "
                             "of one batch overlaps the start of the next; every step still plans all %d plans of the batch" % (args.steps, P),
                      "matches_single_stream_steps": same_ov}

    # ---- end-to-end through the host-buffer C ABI (what a Python caller of plan_batch gets) ----
    # Headline form: the caller keeps its worlds packed (rrtk_pack_grid_host, once per set_og) and asks for what the reference's
    # caller keeps of a plan -- the path (ids, points, cost) and the statistics; beside it the round-1 form (uint8 grids in,
    # every tree out).  Both move everything through pinned host buffers inside the timed region.
    e2e = None
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    if not args.no_e2e:
        Pe = min(P, args.e2e_plans)
        og_pinned = torch.empty((Pe, W, H), dtype=torch.uint8, pin_memory=True)
        og_pinned.copy_(db.og[:Pe])
        bits_pinned = torch.empty((Pe, db.words), dtype=torch.int32, pin_memory=True)
        bits_pinned.copy_(db.bits[:Pe])
        torch.cuda.synchronize(dev)
        og_host = og_pinned.numpy()
        bits_host = bits_pinned.numpy().view(np.uint32)
        packer_ok = bool(np.array_equal(_lib.pack_grids_host(og_host[:4]), bits_host[:4]))     # the host packer makes the same words
        pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()          # noqa: E731
        out_paths = {"stats": pin((Pe, _lib.STAT_COUNT), torch.int64), "path": pin((Pe, PATH_CAP), torch.int32),
                     "xy": pin((Pe, PATH_CAP, 2), torch.int16), "len": pin((Pe,), torch.int32), "path_cost": pin((Pe,), torch.float64)}
        out_trees = {"stats": pin((Pe, _lib.STAT_COUNT), torch.int64), "pts": pin((Pe, N_ITER + 1, 2), torch.int16),
                     "cost": pin((Pe, N_ITER + 1), torch.float64), "parent": pin((Pe, N_ITER + 1), torch.int32)}
        ctx = _lib.Context()
        desc_e = desc[:Pe]

        def e2e_step(mode):
            st = batch.seed_states(ids[:Pe])                         # seeds -> PCG64 states (host)
            # chunked pipeline: H2D grids, (K0) + free index, sampler, K7, (path extraction), D2H
            if mode == "paths":
                ctx.plan_worlds2(_lib.KIND_STAR, bits_host, W, H, desc_e, N_ITER, R_REWIRE, states=st, bits=True, trees=False, paths=True,
                                 path_cap=PATH_CAP, out=out_paths, chunk=args.e2e_chunk)
            else:
                ctx.plan_worlds2(_lib.KIND_STAR, og_host, W, H, desc_e, N_ITER, R_REWIRE, states=st, bits=False, trees=True, paths=False,
                                 out=out_trees, chunk=args.e2e_chunk)

        def timed(mode):
            for _ in range(max(1, args.warmup - 1)):
                e2e_step(mode)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                e2e_step(mode)
            barrier()
            tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        dt_paths, dt_trees = timed("paths"), timed("trees")
        rec = db.path_records(PATH_CAP)
        torch.cuda.synchronize(dev)
        short = out_paths["len"] <= PATH_CAP
        same_paths = (np.array_equal(out_paths["stats"][:, :3], stats[:Pe, :3]) and np.array_equal(out_paths["len"], rec["len"][:Pe].cpu().numpy())
                      and np.array_equal(out_paths["path_cost"].view(np.int64), rec["path_cost"][:Pe].cpu().numpy().view(np.int64))
                      and np.array_equal(out_paths["xy"][short], rec["xy"][:Pe].cpu().numpy()[short]))
        same_trees = np.array_equal(out_trees["stats"][:, :3], stats[:Pe, :3]) and np.array_equal(out_trees["cost"], db.out["cost"][:Pe].cpu().numpy())
        rec_bytes = PATH_CAP * 8 + 4 + 8 + _lib.STAT_COUNT * 8
        e2e = {"value": Pe * world * args.steps / dt_paths, "unit": "plans/s",
               "h2d_bytes_per_step": int(Pe * (db.words * 4 + 64 + 32)),
               "d2h_bytes_per_step": int(Pe * rec_bytes),
               "plans_per_step_per_gpu": Pe, "ms_per_step": 1000 * dt_paths / args.steps,
               "api": "rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS) via rrtplanner_b200._lib.Context.plan_worlds2: tiled bit grids, plan "
                      "descriptors and PCG64 states up; path record (ids + points, cap %d; length; cost) and statistics of every plan down; "
                      "chunks of %d plans on five plan streams between one preparation and one output stream, pinned host buffers" % (PATH_CAP, args.e2e_chunk or 4 * sms),
               "matches_device_arm": bool(same_paths), "host_packer_matches_device_packer": packer_ok,
               "trees_mode": {"value": Pe * world * args.steps / dt_trees, "unit": "plans/s", "ms_per_step": 1000 * dt_trees / args.steps,
                              "h2d_bytes_per_step": int(Pe * (W * H + 64 + 32)),
                              "d2h_bytes_per_step": int(Pe * ((N_ITER + 1) * 16 + _lib.STAT_COUNT * 8)),
                              "api": "rrtk_ctx_plan_worlds2(RRTK_OUT_TREES): uint8 grids up, every tree down (the round-1 call), chunks of %d plans" % (args.e2e_chunk or 2 * sms),
                              "matches_device_arm": bool(same_trees)}}
        ctx.close()

    # ---- strong scaling: the same 4096 plans in total whatever N, with the final gather of the paths ----
    strong = None if args.no_strong else strong_leg(local, rank, world, args.steps, args.warmup, barrier)

    # cfg5 on every rank (weak scaling like the headline; K8 plans shard by index exactly like K7's)
    dub_multi = dubins_bench(local, args.steps, False, rank=rank, world=world) if (world > 1 and not args.no_dubins) else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- derived numbers ------------------------------------------------------------------------
    plans_total = P * world
    value = plans_total * args.steps / (ms_total / 1000.0)
    nn_pairs, ring, cells, checks = (float(S[k].sum()) for k in ("nn_pairs", "ring_members", "cells", "checks"))
    alg_bytes = 8.0 * nn_pairs + 8.0 * ring + 4.0 * cells          # SURVEY.md section 8(d) per-unit figures, one launch
    achieved = alg_bytes / (ms_plan / 1000.0) / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_mhz = clocks.get("sm_mhz") or peaks.get("clocks_under_load", {}).get("sm_mhz_median") or 1965.0
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    from rrtplanner_b200 import peaks as onchip
    measured = onchip.measure(local)                                  # L2 -> SM and shared-memory read bandwidth of this device (csrc/peaks.cu)
    smem_peak = measured["smem_read_GBps"]
    smem_nominal = 128.0 * sms * sm_mhz * 1e6 / 1e9                   # 128 B/clk/SM x SMs x SM clock, for comparison
    hbm_bytes = P * (db.words * 4 + N_ITER * 4 + (N_ITER + 1) * 16 + 64 + _lib.STAT_COUNT * 8)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    smem_b, blocks_per_sm = db.footprint()
    which = db.L.rrtk_plan_kernel(_lib.KIND_STAR, W, H, N_ITER, args.threads).decode()
    plan_kernel_label = {
        "grid": "rrtk::plan_grid_kernel<RRTK_STAR, K=%s samples per round, T=128 threads> (tree in shared memory in bucket order of the samples; "
                "near / within read the buckets around a sample)" % os.environ.get("RRTK_GRID_K", "16"),
        "scan": "rrtk::plan_scan_kernel<RRTK_STAR, K=%s samples per round, T=%s threads> (brute-force packed-key scan)"
                % (os.environ.get("RRTK_PLAN_K", "8"), args.threads or "128 (default)"),
        "wide": "rrtk::plan_wide_kernel<RRTK_STAR>"}.get(which, which)
    roofline = {
        "kernel": plan_kernel_label, "bound": "smem", "achieved": achieved, "peak": smem_peak,
        "unit": "GB/s", "frac": achieved / smem_peak, "traffic": NCU_DRAM_BYTES_PER_PLAN * P,
        "traffic_source": "profile constant, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture "
                          "(" + NCU_DRAM_SOURCE + "), scaled to the plans of this launch; the tree, grid and sample stream of a plan cross HBM once",
        "peak_source": "measured in this run: rrtk_peak_smem_read (one block per SM reading its shared memory with conflict-free 16-byte loads, "
                       f"best of 5); nominal 128 B/clk/SM x {sms} SMs x {sm_mhz:.0f} MHz = {smem_nominal:.0f} GB/s",
        "measured_peaks": measured,
        "algorithmic_bytes_per_launch": alg_bytes,
        "bytes_model": "8 B x (iteration, filled vertex) pairs + 8 B x radius-set members + 4 B x grid cells tested: what the reference's loop "
                       "touches (SURVEY 8(d)), whichever kernel runs -- the bucket kernel answers near / within from ~1/13 of the tree, so like "
                       "the clearance-field walk of cfg2 it moves fewer bytes than it is credited with",
        "kernel_ms": ms_plan,
        "smem_bytes_actually_read_per_launch": (4.0 * nn_pairs + 4.0 * ring + 4.0 * cells) if which != "grid" else None,
        "hbm_view": {"bytes_per_launch": hbm_bytes, "achieved": hbm_bytes / (ms_plan / 1000.0) / 1e9, "peak": hbm_peak,
                     "frac": hbm_bytes / (ms_plan / 1000.0) / 1e9 / hbm_peak,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650"},
        "iterations_per_s_per_sm": P * N_ITER / (ms_plan / 1000.0) / sms,
        "blocks_per_sm": blocks_per_sm, "smem_bytes_per_block": smem_b,
    }
    line = {
        "metric": METRIC, "value": value, "unit": "plans/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "plans_per_gpu": P, "plans_total": plans_total, "threads_per_plan": args.threads or "default",
                   "l2": "inputs+outputs per step (%.0f MB) exceed the 126 MB L2; no explicit flush" % (hbm_bytes / 1e6),
                   "obstacle_fraction": float(db.og[: min(P, 256)].float().mean().item()),
                   "mean_vertices": float(all_stats[:, 0].mean()), "goal_found_frac": float(all_stats[:, 2].mean())},
        "clocks": clocks,
        "roofline": roofline,
        "collision_checks_per_s": checks * world / (ms_plan / 1000.0),
        "collision_cells_per_s": cells * world / (ms_plan / 1000.0),
        "kernel_ms": {"sample_streams": ms_sampler, "plan": ms_plan},
        "gpu_launches": 2 * args.steps,
        "e2e": e2e,
    }
    if overlapped is not None:
        line["overlapped_steps"] = overlapped
    if strong is not None:
        line["strong_scaling"] = strong
    if world == 1 and not args.no_cpu:
        m = args.cpu_plans
        gpu_trees = tuple(db.out[k][:m].cpu().numpy() for k in ("pts", "cost", "parent", "stats"))
        line["cpu_baseline"], line["matches_oracle"] = cpu_baseline_single(m, gpu_trees)
    if world == 1 and not args.no_collision:
        line["collision_microbench"] = collision_microbench(local, args.steps, args.warmup, not args.no_cpu, sm_mhz, measured)
    if world == 1 and not args.no_informed:
        line["informed_bench"] = informed_bench(local, args.steps, not args.no_cpu, measured)
    if world == 1 and not args.no_class_api:
        line["class_api_bench"] = class_api_bench(args.steps, not args.no_cpu)
    if world == 1 and not args.no_dubins:
        line["dubins_bench"] = dubins_bench(local, args.steps, not args.no_cpu)
    if dub_multi is not None:
        line["dubins_bench"] = dub_multi
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--plans", type=int, default=4096, help="plans per GPU per step")
    ap.add_argument("--threads", type=int, default=0, help="threads per plan block (0 = library default)")
    ap.add_argument("--e2e-plans", type=int, default=4096)
    ap.add_argument("--e2e-chunk", type=int, default=0, help="plans per pipeline chunk of the end-to-end call (0 = library default)")
    ap.add_argument("--cpu-plans", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (4096 plans in total, paths gathered to rank 0)")
    ap.add_argument("--no-collision", action="store_true", help="skip the cfg2 collision microbenchmark")
    ap.add_argument("--collision-only", action="store_true", help="run only the cfg2 collision microbenchmark (profiling aid)")
    ap.add_argument("--no-dubins", action="store_true", help="skip the cfg5 Dubins RRT* leg")
    ap.add_argument("--no-informed", action="store_true", help="skip the cfg4 RRTStarInformed leg")
    ap.add_argument("--no-class-api", action="store_true", help="skip the cfg1 class-API latency leg")
    ap.add_argument("--dubins-only", action="store_true", help="run only the cfg5 Dubins RRT* leg (profiling aid)")
    ap.add_argument("--informed-only", action="store_true", help="run only the cfg4 RRTStarInformed leg (profiling aid)")
    ap.add_argument("--dubins-plans", type=int, default=DUB_PLANS)
    ap.add_argument("--plan-only", action="store_true", help="device arm of the headline only (experiments): implies every --no-* flag")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the headline, write the trees of its last step (a fixed sample of plans) and the "
                         "result statistics of every plan as DIR/<name>.npy (rank 0's plans)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.collision_only or args.informed_only or args.dubins_only):
        ap.error("--dump-outputs writes the outputs of the native headline; it does not combine with --impl reference or --*-only")
    if args.plan_only:
        args.no_e2e = args.no_cpu = args.no_strong = args.no_collision = args.no_dubins = args.no_informed = args.no_class_api = True
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3
    if args.collision_only:
        import torch
        torch.cuda.set_device(0)
        from rrtplanner_b200 import peaks as onchip
        print(json.dumps(collision_microbench(0, args.steps, args.warmup, not args.no_cpu, 1965.0, onchip.measure(0))), flush=True)
    elif args.informed_only:
        import torch
        torch.cuda.set_device(0)
        from rrtplanner_b200 import peaks as onchip
        print(json.dumps(informed_bench(0, args.steps, not args.no_cpu, onchip.measure(0))), flush=True)
    elif args.dubins_only:
        import torch
        torch.cuda.set_device(0)
        print(json.dumps(dubins_bench(0, args.steps, not args.no_cpu, args.dubins_plans, args.threads)), flush=True)
    elif args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
