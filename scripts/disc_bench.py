"""What the configuration space of a disc robot costs on the device (csrc/disc.cu, rrtk_inflate_disc).

    python scripts/disc_bench.py [--steps K] [--plans P] [--out FILE]

One JSON line with
  (a) kernel: device time of rrtk_inflate_disc (CUDA events, median of K launches after a warm-up launch of every shape) for
      cfg3 (P x 512 x 512 value-noise worlds, seeds 1000 + w), cfg4 (1 x 1024 x 1024) and cfg2 (1 x 2048 x 2048), at radii
      1, 4, 16 and 64 cells; bytes per cell and the rate that makes against the pass-1 field written and read twice;
  (b) the cfg3 device step with radius 4 -- inflate, free rows, sampler, RRT* plan kernel (n = 5000, r_rewire = 50) --
      against the same step without a radius (sampler and plan kernel), each stage timed with events;
  (c) plan_batch end to end (host worlds in, trees out, seeds 0..P-1) with and without robot_radius = 4, alternated;
  (d) the CPU arm: scipy.ndimage.distance_transform_edt per 512 x 512 world on one host core of the same machine.
The card's name, power limit and clocks are read in the same run, before and after.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rrtplanner_b200 import _lib, batch, worlds  # noqa: E402

RADII = (1, 4, 16, 64)
R_REWIRE, N = 50.0, 5000


def gpu_card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else None


def kernel_times(db, steps):
    """rrtk_inflate_disc of every world of ``db`` at each radius: median ms over ``steps`` launches."""
    import torch
    nw, W, H = int(db.bits.shape[0]), db.W, db.H
    scratch = torch.empty(int(db.L.rrtk_inflate_disc_scratch_bytes(nw, W, H)), dtype=torch.uint8, device=db.dev)
    out = torch.empty_like(db.bits)
    src = torch.arange(nw, dtype=torch.int32, device=db.dev)
    stream = torch.cuda.current_stream(db.dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    res = {}
    for rho in RADII:
        r2 = torch.full((nw,), int(_lib.disc_r2(rho)), dtype=torch.int32, device=db.dev)

        def launch():
            _lib.check(db.L.rrtk_inflate_disc(db.bits.data_ptr(), nw, W, H, src.data_ptr(), r2.data_ptr(), nw, out.data_ptr(),
                                              scratch.data_ptr(), stream.cuda_stream), "inflate_disc")
        launch()
        ms = []
        for _ in range(steps):
            ev[0].record(stream)
            launch()
            ev[1].record(stream)
            torch.cuda.synchronize(db.dev)
            ms.append(ev[0].elapsed_time(ev[1]))
        t = float(np.median(ms))
        cells = nw * W * H
        # pass 1 reads the bit grid and writes the uint16 field; pass 2 reads the field twice and writes / reads / writes the words
        moved = cells / 8 + 2 * cells + 2 * 2 * cells + 3 * cells / 8
        res[str(rho)] = {"ms": t, "all_ms": ms, "ns_per_cell": t * 1e6 / cells, "bytes_per_cell": moved / cells,
                         "GB_per_s": moved / (t * 1e-3) / 1e9}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--plans", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    P, steps = args.plans, args.steps
    line = {"gpu": gpu_card()}

    # (a) kernel
    ids = np.arange(P)
    db = batch.DeviceBatch("star", 512, 512, N, R_REWIRE, device=0).gen_worlds([worlds.world_seed(int(p)) for p in ids])
    kern = {"cfg3_%dx512x512" % P: kernel_times(db, steps)}
    for S in (1024, 2048):
        one = batch.DeviceBatch("star", S, S, 8, device=0).gen_worlds([worlds.world_seed(0)])
        kern["1x%dx%d" % (S, S)] = kernel_times(one, steps)
        del one
    line["kernel"] = kern

    # (b) cfg3 device step with and without a radius: start / goal from the device sampler (seed 2000 + p) on each grid
    og_dev = db.og
    stream = torch.cuda.current_stream(dev)

    def step_times(radius):
        b = batch.DeviceBatch("star", 512, 512, N, R_REWIRE, device=0).set_worlds_u8(og_dev)
        if radius:
            b.inflate_disc(radius)
        pair = batch.DeviceBatch("star", 512, 512, 8, device=0)
        pair.bits, pair.rowcum = b.bits, b.rowcum
        pair.set_plans(batch.make_desc(ids, np.zeros((P, 2)), np.zeros((P, 2))))
        pair.seed_samples(2000 + ids)
        d = pair.samples.cpu().numpy().astype(np.int64)
        starts = d[:, 0]
        goals = d[np.arange(P), 1 + (d[:, 1:] != starts[:, None]).any(axis=2).argmax(axis=1)]
        b.set_plans(batch.make_desc(ids, starts, goals))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        rows = []
        for s in range(steps + 1):                                       # step 0: warm-up
            b.set_worlds_u8(og_dev)                                      # pack + free rows of the point-robot grid (untimed)
            ev[0].record(stream)
            if radius:
                b.inflate_disc(radius)                                   # inflate + free rows
            ev[1].record(stream)
            b.seed_samples(ids)
            ev[2].record(stream)
            b.run()
            ev[3].record(stream)
            torch.cuda.synchronize(dev)
            if s:
                rows.append([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])])
        found = int(b.out["stats"][:, 2].sum().item())
        r = np.median(np.array(rows), axis=0)
        return {"inflate_and_free_rows_ms": float(r[0]), "sampler_ms": float(r[1]), "plan_kernel_ms": float(r[2]),
                "step_ms": float(r.sum()), "inflate_share_of_step": float(r[0] / r.sum()), "goal_reached": found}

    line["cfg3_step"] = {"radius_4": step_times(4), "no_radius": step_times(None),
                         "workload": "%d RRT* plans, n=%d, r_rewire=%g, 512x512 worlds 1000+p, pairs from the device sampler "
                                     "(2000+p) on the grid planned on, seeds 0..%d" % (P, N, R_REWIRE, P - 1)}

    # (c) plan_batch end to end (host worlds, trees out), with and without robot_radius, alternated
    og_host = db.og.cpu().numpy()
    del db, og_dev
    torch.cuda.empty_cache()
    rng = np.random.default_rng(7)
    cs0 = None
    starts = np.empty((P, 2), np.int64)
    goals = np.empty((P, 2), np.int64)
    ctx = _lib.Context()
    cs_bits = ctx.inflate_disc(og_host, ids, np.full(P, int(_lib.disc_r2(4))))
    for p in range(P):                                                   # pairs free on the radius-4 grid (so on both)
        cs0 = _lib.unpack_grids_host(cs_bits[p:p + 1], 512, 512)[0]
        free = np.argwhere(cs0 == 0)
        starts[p], goals[p] = free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]
    seeds = ids

    def e2e(radius):
        t0 = time.perf_counter()
        batch.plan_batch("star", og_host, N, starts, goals, r_rewire=R_REWIRE, seeds=seeds, ctx=ctx, robot_radius=radius)
        return time.perf_counter() - t0

    e2e(None), e2e(4)                                                    # warm-up
    times = {"no_radius": [], "radius_4": []}
    for _ in range(max(2, steps // 2)):
        times["no_radius"].append(e2e(None))
        times["radius_4"].append(e2e(4))
    ctx.close()
    line["plan_batch_e2e"] = {k: {"s": float(np.median(v)), "all_s": v, "plans_per_s": P / float(np.median(v))} for k, v in times.items()}
    line["plan_batch_e2e"]["api"] = ("plan_batch('star', uint8 host worlds, seeds, trees out); no radius: rrtk_ctx_plan_worlds; "
                                     "radius 4: rrtk_ctx_inflate_disc (upload, inflate, packed download) then "
                                     "rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_TREES)")

    # (d) CPU arm: scipy's exact EDT per 512 x 512 world, one core
    from scipy import ndimage
    t = []
    for w in range(16):
        t0 = time.perf_counter()
        ndimage.distance_transform_edt(og_host[w] == 0)
        t.append(time.perf_counter() - t0)
    line["cpu_edt_ms_per_512x512_world"] = {"median_ms": 1e3 * float(np.median(t)), "worlds": 16, "cpus": os.cpu_count(),
                                            "host_core_s_for_cfg3": float(np.median(t)) * P}
    line["gpu_after"] = gpu_card()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
