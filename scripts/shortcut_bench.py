"""What the line-of-sight shortcut of path records costs and what it prunes (csrc/shortcut.cu).

    python scripts/shortcut_bench.py [--steps K] [--plans P] [--cfg4-plans P4] [--out FILE]

Two shapes, RRT* with r_rewire = 50, plan p on its own value-noise world (seed 1000 + p), start / goal from the device
sampler (seed 2000 + p) and free-space stream default_rng(p), as bench.py's cfg3 leg:
  cfg3  512 x 512, n = 5000, P plans (default 4096)
  cfg4  the cfg4 world size, 1024 x 1024 (longer segments), n = 20000, P4 plans (default 1024)
For each, one JSON object with
  (a) device arm (DeviceBatch, CUDA events): the plan kernel of the step against rrtk_shortcut_paths on the device-resident
      path records of that step (the records are restored from a copy before each timed pass);
  (b) end to end rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS) with and without RRTK_OUT_SHORTCUT, steps alternated;
  (c) mean path vertices before and after, and mean relative cost reduction over the plans that reached their goal;
and the check that the fused flag returns what (a) computed.
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

R_REWIRE, PATH_CAP = 50.0, 256


def gpu_card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else None


def shape_bench(S, P, n, steps):
    import torch

    dev = torch.device("cuda", 0)
    ids = np.arange(P)
    db = batch.DeviceBatch("star", S, S, n, R_REWIRE, device=0).gen_worlds([worlds.world_seed(int(p)) for p in ids])
    pair = batch.DeviceBatch("star", S, S, 8, device=0)
    pair.bits, pair.rowcum = db.bits, db.rowcum
    pair.set_plans(batch.make_desc(ids, np.zeros((P, 2)), np.zeros((P, 2))))
    pair.seed_samples(2000 + ids)
    d = pair.samples.cpu().numpy().astype(np.int64)
    starts = d[:, 0]
    goals = d[np.arange(P), 1 + (d[:, 1:] != starts[:, None]).any(axis=2).argmax(axis=1)]
    desc = batch.make_desc(ids, starts, goals)
    db.set_plans(desc)
    db.seed_samples(ids)
    stream = torch.cuda.current_stream(dev)

    # (a) device arm
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    plan_ms, sc_ms = [], []
    for step in range(steps + 1):                                        # step 0: warm-up
        ev[0].record(stream)
        db.run()
        ev[1].record(stream)
        rec = db.path_records(PATH_CAP)
        before = {k: v.clone() for k, v in rec.items()}
        ev[2].record(stream)
        db.shortcut_records(rec)
        ev[3].record(stream)
        torch.cuda.synchronize(dev)
        if step:
            plan_ms.append(ev[0].elapsed_time(ev[1]))
            sc_ms.append(ev[2].elapsed_time(ev[3]))
    # shortcut alone, repeated on the same records (restored from `before` outside the timed window)
    sc_rep = []
    for _ in range(max(steps, 5)):
        for k in rec:
            rec[k].copy_(before[k])
        ev[2].record(stream)
        db.shortcut_records(rec)
        ev[3].record(stream)
        torch.cuda.synchronize(dev)
        sc_rep.append(ev[2].elapsed_time(ev[3]))
    b = {k: v.cpu().numpy() for k, v in before.items()}
    a = {k: v.cpu().numpy() for k, v in rec.items()}
    fits = (b["len"] >= 1) & (b["len"] <= PATH_CAP)
    found = fits & (b["stats"][:, 2] == 1)
    rel = 1.0 - a["path_cost"][found] / b["path_cost"][found]

    # (b) end to end, with and without the flag, alternated
    og_host = db.og.cpu().numpy()
    bits_host = _lib.pack_grids_host(og_host)
    del og_host
    states = batch.seed_states(ids)
    pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()          # noqa: E731

    def outs():
        return {"stats": pin((P, _lib.STAT_COUNT), torch.int64), "path": pin((P, PATH_CAP), torch.int32),
                "xy": pin((P, PATH_CAP, 2), torch.int16), "len": pin((P,), torch.int32), "path_cost": pin((P,), torch.float64)}

    ctx = _lib.Context()
    bufs = {False: outs(), True: outs()}

    def e2e(shortcut):
        ctx.plan_worlds2(_lib.KIND_STAR, bits_host, S, S, desc, n, R_REWIRE, states=states, bits=True, trees=False, paths=True,
                         path_cap=PATH_CAP, out=bufs[shortcut], shortcut=shortcut)

    e2e(False), e2e(True)                                                # warm-up
    times = {False: [], True: []}
    for _ in range(steps):
        for flag in (False, True):
            t0 = time.perf_counter()
            e2e(flag)
            times[flag].append(time.perf_counter() - t0)
    ctx.close()
    f, g = bufs[True], bufs[False]
    fused_ok = bool(all(np.array_equal(f[k][fits], a[k][fits]) for k in ("path", "xy")) and np.array_equal(f["len"], a["len"]) and
                    np.array_equal(f["path_cost"].view(np.int64), a["path_cost"].view(np.int64)) and
                    all(np.array_equal(g[k][fits], b[k][fits]) for k in ("path", "xy")))
    assert fused_ok, "the fused flag and the device-resident shortcut disagree"
    plan, sc = float(np.mean(plan_ms)), float(np.median(sc_rep))
    return {
        "workload": "%dx%d, %d RRT* plans, n=%d, r_rewire=%g, worlds 1000+p, pairs 2000+p, seeds 0..%d, path_cap=%d"
                    % (S, S, P, n, R_REWIRE, P - 1, PATH_CAP),
        "device": {"plan_kernel_ms": plan, "shortcut_ms": sc, "shortcut_ms_in_step": float(np.mean(sc_ms)),
                   "shortcut_share_of_plan_kernel": sc / plan,
                   "note": "CUDA events; plan kernel mean of %d steps; shortcut median of %d passes on the step's records, "
                           "restored from a copy before each pass (grids %d MB of bit words)" % (steps, len(sc_rep), db.bits.numel() * 4 >> 20)},
        "e2e": {"paths_s": float(np.median(times[False])), "paths_shortcut_s": float(np.median(times[True])),
                "plans_per_s_paths": P / float(np.median(times[False])), "plans_per_s_paths_shortcut": P / float(np.median(times[True])),
                "all_s": {"paths": times[False], "paths_shortcut": times[True]},
                "api": "rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS [| RRTK_OUT_SHORTCUT]), pinned outputs, steps alternated"},
        "paths": {"plans": P, "records_that_fit": int(fits.sum()), "goal_reached": int(found.sum()),
                  "mean_vertices_before": float(b["len"][fits].mean()), "mean_vertices_after": float(a["len"][fits].mean()),
                  "mean_vertices_before_goal_reached": float(b["len"][found].mean()),
                  "mean_vertices_after_goal_reached": float(a["len"][found].mean()),
                  "mean_relative_cost_reduction": float(rel.mean()), "max_relative_cost_reduction": float(rel.max())},
        "fused_equals_device_form": fused_ok,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--plans", type=int, default=4096)
    ap.add_argument("--cfg4-plans", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    line = {"gpu": gpu_card(), "cfg3": shape_bench(512, args.plans, 5000, args.steps)}
    torch.cuda.empty_cache()
    line["cfg4_world_size"] = shape_bench(1024, args.cfg4_plans, 20000, max(2, args.steps // 2))
    line["gpu_after"] = gpu_card()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
