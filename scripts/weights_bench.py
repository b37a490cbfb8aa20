"""What weighted sampling costs and what it changes on the cfg3 shape (csrc/rng.cu: rrtk_weight_index,
rrtk_sample_streams_weighted).

    python scripts/weights_bench.py [--steps K] [--plans P] [--out FILE]

Workload: P (default 4096) value-noise worlds of 512 x 512, one RRT* plan each (n = 5000, r_rewire = 50, seeds 0..P-1) between
two random free cells.  Each world gets a map of 255 within 24 cells of its start-goal segment and 4 elsewhere, a stand-in for
a learned heatmap.  One JSON line with
  (a) device times (CUDA events, median of K after a warm-up of every shape): the index build, the weighted sampler against the
      uniform sampler, and the device step (index + weighted sampler + plan kernel against sampler + plan kernel);
  (b) end to end: plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS | RRTK_SEED_WEIGHTS) against the same call without weights
      (alternated, host clock), and the one-time set_sample_weights upload;
  (c) the effect: found rate and mean path cost of the found plans, with and without the map;
  (d) numpy drawing the same weighted streams on one host core (what a caller does without this feature), per plan and for P.
The card's name, power limit and clocks are read in the same run.
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

W = H = 512
N, R_REWIRE = 5000, 50.0
WIDTH, HI, LO = 24.0, 255, 4


def gpu_card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else None


def corridor_maps(torch, starts, goals, dev):
    """(P, W, H) uint8 on the device: HI within WIDTH cells of the start-goal segment, LO elsewhere."""
    x = torch.arange(W, dtype=torch.float64, device=dev)[:, None]
    y = torch.arange(H, dtype=torch.float64, device=dev)[None, :]
    out = torch.empty((len(starts), W, H), dtype=torch.uint8, device=dev)
    a_all = torch.from_numpy(np.asarray(starts, np.float64)).to(dev)
    b_all = torch.from_numpy(np.asarray(goals, np.float64)).to(dev)
    for p in range(len(starts)):
        a, d = a_all[p], b_all[p] - a_all[p]
        L2 = torch.clamp(d @ d, min=1e-12)
        t = torch.clamp(((x - a[0]) * d[0] + (y - a[1]) * d[1]) / L2, 0.0, 1.0)
        dist2 = (x - a[0] - t * d[0]) ** 2 + (y - a[1] - t * d[1]) ** 2
        out[p] = torch.where(dist2 <= WIDTH * WIDTH, HI, LO).to(torch.uint8)
    return out


def timed(torch, fn, steps):
    stream = torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    fn()
    ms = []
    for _ in range(steps):
        ev[0].record(stream)
        fn()
        ev[1].record(stream)
        ev[1].synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--plans", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("weights_bench needs a CUDA device")
    P, K = args.plans, args.steps
    card0 = gpu_card()
    db = batch.DeviceBatch("star", W, H, N, R_REWIRE).gen_worlds([worlds.world_seed(p) for p in range(P)])
    ogs = db.og.cpu().numpy()
    rng = np.random.default_rng(0)
    starts, goals = np.zeros((P, 2), np.int64), np.zeros((P, 2), np.int64)
    for p in range(P):
        free = np.argwhere(ogs[p] == 0)
        starts[p], goals[p] = free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]
    wmap = corridor_maps(torch, starts, goals, db.dev)
    desc = batch.make_desc(np.arange(P), starts, goals)
    seeds = np.arange(P)
    db.set_plans(desc)
    L, st = db.L, torch.cuda.current_stream().cuda_stream
    index = torch.empty(int(L.rrtk_weight_index_bytes(P, W, H)), dtype=torch.uint8, device=db.dev)
    states = torch.from_numpy(batch.seed_states(seeds).view(np.int64)).to(db.dev)
    samples = torch.empty((P, N, 2), dtype=torch.int16, device=db.dev)

    def build_index():
        _lib.check(L.rrtk_weight_index(db.bits.data_ptr(), wmap.data_ptr(), P, W, H, index.data_ptr(), st), "weight_index")

    def weighted():
        _lib.check(L.rrtk_sample_streams_weighted(db.bits.data_ptr(), wmap.data_ptr(), index.data_ptr(), P, W, H, db.desc.data_ptr(), P,
                                                  states.data_ptr(), None, N, samples.data_ptr(), st), "sample_streams_weighted")

    def uniform():
        _lib.check(L.rrtk_sample_streams(db.bits.data_ptr(), db.rowcum.data_ptr(), W, H, db.desc.data_ptr(), P, states.data_ptr(), N,
                                         samples.data_ptr(), st), "sample_streams")

    def plan():
        db.samples = samples
        db.run()

    dev = {"index_ms": timed(torch, build_index, K), "weighted_sampler_ms": timed(torch, weighted, K),
           "uniform_sampler_ms": timed(torch, uniform, K)}
    dev["step_weighted_ms"] = timed(torch, lambda: (build_index(), weighted(), plan()), K)
    res_w = db.download()
    dev["step_uniform_ms"] = timed(torch, lambda: (uniform(), plan()), K)
    res_u = db.download()

    def effect(res):
        found = res.stat("found").astype(bool)
        cost = res.cost[np.arange(P), res.stat("vgoal")]
        return {"found_rate": float(found.mean()), "mean_path_cost": float(cost[found].mean())}

    # end to end from host arrays: packed worlds in, path records out
    bits = np.ascontiguousarray(db.bits.cpu().numpy().view(np.uint32))
    wh = wmap.cpu().numpy()
    ctx = _lib.Context()
    hstates = batch.seed_states(seeds)
    t0 = time.perf_counter()
    ctx.set_sample_weights(wh)
    upload_ms = (time.perf_counter() - t0) * 1e3
    e2e = {"weighted_ms": [], "uniform_ms": []}
    outs = {}
    for _ in range(K + 1):
        for key, sw in (("weighted_ms", True), ("uniform_ms", None)):
            t0 = time.perf_counter()
            outs[key] = ctx.plan_worlds2(_lib.KIND_STAR, bits, W, H, desc, N, R_REWIRE, states=hstates, bits=True, paths=True,
                                         sample_weights=sw)
            e2e[key].append((time.perf_counter() - t0) * 1e3)
    ctx.close()
    # the pipelined call plans what the device step planned: same j / vgoal / found per plan
    same_w = bool(np.array_equal(outs["weighted_ms"]["stats"][:, :3], res_w.stats[:, :3]))
    same_u = bool(np.array_equal(outs["uniform_ms"]["stats"][:, :3], res_u.stats[:, :3]))
    e2e = {k: float(np.median(v[1:])) for k, v in e2e.items()}
    # numpy on one host core: the same streams plan by plan
    from_np = min(P, 64)
    t0 = time.perf_counter()
    for p in range(from_np):
        e = np.where(ogs[p] == 0, wh[p].astype(np.int64), 0)
        cum = np.cumsum(e.ravel())
        k = np.searchsorted(cum, np.random.default_rng(p).integers(0, int(cum[-1]), size=N), side="right")
        np.stack(np.divmod(k, H), axis=1)
    np_ms = (time.perf_counter() - t0) * 1e3 / from_np
    line = {"bench": "weights", "card_before": card0, "card_after": gpu_card(), "plans": P, "W": W, "H": H, "n": N, "r_rewire": R_REWIRE,
            "map": {"width": WIDTH, "hi": HI, "lo": LO}, "steps": K, "device": dev,
            "end_to_end": {**e2e, "set_sample_weights_upload_ms": upload_ms, "weighted_stats_equal_device": same_w,
                           "uniform_stats_equal_device": same_u},
            "effect": {"weighted": effect(res_w), "uniform": effect(res_u)},
            "numpy_one_core": {"ms_per_plan": np_ms, "ms_for_all_plans": np_ms * P, "plans_timed": from_np}}
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
