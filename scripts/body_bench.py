"""What a car-shaped body costs and buys on the device (csrc/body.cu rrtk_inflate_body, K8 rrtk_plan2_batch_layers).

    python scripts/body_bench.py [--steps K] [--plans P] [--out FILE]

One JSON line with
  (a) kernel: device time of rrtk_inflate_body (CUDA events, median of K launches after a warm-up launch) for the cfg5 shape
      (P x 512 x 512 value-noise worlds, seeds world_seed(p)) and for one 2048 x 2048 world, with the car of DESIGN.md (8 cells
      ahead of the reference point, 2 behind, 2.5 to each side, 16 heading layers); the bytes of the layer grids written;
  (b) the cfg5 device step (Dubins RRT*, n = 5000, r_rewire = 50, rho = 6, ds = 1, 16 headings, rewire on) three ways:
      without a body, with the car (rrtk_inflate_body + rrtk_plan2_batch_layers) and with the disc that covers the car
      (robot_radius = its farthest corner, rrtk_inflate_disc + rrtk_plan2_batch), plan kernel timed with events; the same
      start / goal configurations for all three (device sampler, seed 2000 + p, on the world itself; headings as bench.py's
      cfg5 leg draws them), samples from each variant's own free cells;
  (c) the found rate of each of the three, which is what the body buys.
The card's name, power limit and clocks are read in the same run, before and after.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rrtplanner_b200 import _lib, batch, worlds  # noqa: E402
from rrtplanner_b200.body import body_runs, car_body  # noqa: E402

N, R_REWIRE, NH, RHO, DS = 5000, 50.0, 16, 6.0, 1.0
CAR = dict(front=8.0, rear=2.0, half_width=2.5, nlayers=16)


def gpu_card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else None


def median_ms(fn, steps):
    import torch
    stream = torch.cuda.current_stream()
    fn()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = []
    for _ in range(steps):
        ev[0].record(stream)
        fn()
        ev[1].record(stream)
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return float(np.median(ms)), ms


def kernel_time(db, stencils, steps):
    """rrtk_inflate_body on every world of ``db`` (the runs come back to the host once per call: the launch is sized by them)."""
    import torch
    nw, W, H = int(db.bits.shape[0]), db.W, db.H
    runs, lr = body_runs(stencils)
    L = lr.shape[0] - 1
    d_runs = torch.from_numpy(np.concatenate([runs.reshape(-1), np.zeros(1, np.int32)])).to(db.dev)
    d_lr = torch.from_numpy(lr).to(db.dev)
    layers = torch.empty((nw * L, db.words), dtype=torch.int32, device=db.dev)
    proj = torch.empty((nw, db.words), dtype=torch.int32, device=db.dev)
    stream = torch.cuda.current_stream(db.dev).cuda_stream

    def launch():
        _lib.check(db.L.rrtk_inflate_body(db.bits.data_ptr(), nw, W, H, d_runs.data_ptr(), d_lr.data_ptr(), L, layers.data_ptr(),
                                          proj.data_ptr(), stream), "inflate_body")
    med, all_ms = median_ms(launch, steps)
    return {"median_ms": med, "all_ms": all_ms, "layers": L, "runs": int(runs.shape[0]),
            "layer_bytes": int(layers.numel() * 4), "worlds": nw, "shape": [W, H]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--plans", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    P, steps = args.plans, args.steps
    car = car_body(CAR["front"], CAR["rear"], CAR["half_width"], CAR["nlayers"])
    cover = math.hypot(max(CAR["front"], CAR["rear"]), CAR["half_width"])
    line = {"gpu": gpu_card(), "car": dict(CAR, stencil=list(car.shape), mean_cells_per_layer=float(car.sum() / car.shape[0]),
                                           covering_disc_radius=cover)}
    ids = np.arange(P)
    seeds = [worlds.world_seed(int(p)) for p in ids]

    # (a) kernel
    probe = batch.DeviceBatch("star", 512, 512, 8, device=0).gen_worlds(seeds)
    kern = {"cfg5_%dx512x512" % P: kernel_time(probe, car, steps)}
    one = batch.DeviceBatch("star", 2048, 2048, 8, device=0).gen_worlds([worlds.world_seed(0)])
    kern["1x2048x2048"] = kernel_time(one, car, steps)
    del one, probe
    line["kernel"] = kern

    # (b, c) the cfg5 device step three ways, on the same start / goal configurations: the first two distinct draws of the device
    # sampler (seed 2000 + p) on the grid itself, headings as bench.py's cfg5 leg draws them
    hs = np.random.default_rng(6000).integers(0, NH, size=(P, 2))
    pair = batch.DeviceBatch("star", 512, 512, 8, device=0).gen_worlds(seeds)
    pair.set_plans(batch.make_desc(ids, np.zeros((P, 2)), np.zeros((P, 2)))).seed_samples(2000 + ids)
    draws = pair.samples.cpu().numpy().astype(np.int64)
    starts = draws[:, 0]
    differs = (draws[:, 1:] != starts[:, None]).any(axis=2)
    goals = draws[ids, 1 + differs.argmax(axis=1)]
    desc = batch.make_desc2(ids, np.concatenate([starts, hs[:, :1]], axis=1), np.concatenate([goals, hs[:, 1:]], axis=1))
    del pair
    steps_out = {}
    for variant in ("no_body", "car", "covering_disc"):
        db = batch.DeviceBatch2("dubins", 512, 512, N, r_rewire=R_REWIRE, nheadings=NH, rho=RHO, ds=DS, device=0)
        db.gen_worlds(seeds)
        stage = {}
        og = db.og
        if variant != "no_body":
            def grids():                                     # pack the worlds again, then inflate them (the timed unit)
                db.set_worlds_u8(og)
                if variant == "car":
                    db.inflate_body(car)
                else:
                    db.inflate_disc(cover)
            stage["pack_and_inflate_ms"] = median_ms(grids, 1)[0]
        nfree = db.nfree()
        keep = np.flatnonzero(nfree > 0)                    # the samplers need a free cell: plans only on worlds that have one
        db._require_free_cells = lambda: None               # (the check looks at every world, planned on or not)
        db.set_plans(desc[keep])
        db.seed_samples(ids[keep])
        db.seed_heads(7000 + ids[keep])
        med, all_ms = median_ms(db.run, steps)
        st = db.out["stats"].cpu().numpy()
        stage.update({"plan_kernel_ms": med, "all_ms": all_ms, "plans": int(keep.size), "worlds_without_a_free_cell": int(P - keep.size),
                      "found_rate": float(st[:, 2].sum()) / P, "mean_vertices": float(st[:, 0].mean()),
                      "mean_free_cells": float(nfree.mean()),
                      "kernel": "plan_rewire_kernel<DUBINS_LAYERS>" if variant == "car" else "plan_rewire_kernel<DUBINS>"})
        steps_out[variant] = stage
        del db
        torch.cuda.empty_cache()
    line["cfg5_step"] = steps_out
    line["cfg5_step"]["setup"] = ("%d plans, 512x512 worlds world_seed(p), n=%d, r_rewire=%g, rho=%g, ds=%g, %d headings, rewire on; "
                                  "the same start / goal configurations for all three (first two distinct draws of the device sampler, "
                                  "seed 2000 + p, on the world itself); a start or goal the body or disc blocks is not found, and "
                                  "found_rate counts a world without a free cell as not found"
                                  % (P, N, R_REWIRE, RHO, DS, NH))
    line["gpu_after"] = gpu_card()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
