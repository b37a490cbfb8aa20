"""Seeded informed batches on the cfg4 shape: what the device-side unit-disc stream costs and saves.

    python scripts/informed_seed_bench.py [--steps K] [--plans P] [--out FILE]

One 1024x1024 value-noise world (seed 1000), P start/goal pairs (device sampler, seed 2000 + p, as bench.py's cfg4 leg),
n = 20000, r_rewire = 50, r_goal = 5, plan p seeded with p: every tree is what
RRTStarInformed(og, n, 50, 5, seed=p).plan(start_p, goal_p) builds.  One JSON line with
  (a) device arm (DeviceBatch, CUDA events per stage): sample streams, probe launch, rrtk_ball_streams, full launch;
  (b) end to end through rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS | RRTK_SEED_BALLS): plans/s, bytes per step;
  (c) the same trees built the way a batch caller had to before: a worlds2 probe, the generator advance and unitball()
      draws per plan in numpy, then worlds2 with the (P, n, 2) unit-disc array uploaded;
and the check that (b) and (c) return the same statistics and path records.
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

S, N, R_REWIRE, R_GOAL, PATH_CAP = 1024, 20000, 50.0, 5.0, 256


def gpu_card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        return None


def host_balls(states, nfree, first, n):
    """What RRTStarInformed.plan does to its generator, per plan in numpy: min(f + 1, n) bounded draws, then two uniforms
    per ellipse-phase iteration (uniform(size=...) hands them out in the order of the scalar unitball() calls)."""
    out = np.zeros((len(first), n, 2))
    m = (1 << 64) - 1
    for p, f in enumerate(first):
        g = np.random.Generator(np.random.PCG64())
        st = g.bit_generator.state
        w = [int(v) for v in states[p]]
        st["state"]["state"], st["state"]["inc"] = (w[0] << 64) | (w[1] & m), (w[2] << 64) | (w[3] & m)
        g.bit_generator.state = st
        g.integers(0, nfree, size=n if f < 0 else f + 1)
        if f >= 0:
            u = g.uniform(0, 1, size=(n - 1 - f, 2))
            r, a = np.sqrt(u[:, 0]), 2 * np.pi * u[:, 1]
            out[p, f + 1:, 0], out[p, f + 1:, 1] = r * np.cos(a), r * np.sin(a)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--plans", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    P, n = args.plans, N
    # the cfg4 workload of bench.py: world, pairs, rotations
    db = batch.DeviceBatch("informed", S, S, n, R_REWIRE, R_GOAL, device=0).gen_worlds([worlds.world_seed(0)])
    pair = batch.DeviceBatch("star", S, S, 8, device=0)
    pair.bits, pair.rowcum = db.bits, db.rowcum
    pair.set_plans(batch.make_desc(np.zeros(P, int), np.zeros((P, 2)), np.zeros((P, 2))))
    pair.seed_samples(2000 + np.arange(P))
    d = pair.samples.cpu().numpy().astype(np.int64)
    starts = d[:, 0]
    goals = d[np.arange(P), 1 + (d[:, 1:] != starts[:, None]).any(axis=2).argmax(axis=1)]
    og = db.og[0].cpu().numpy()
    nfree = int((og == 0).sum())
    desc = batch.make_desc(np.zeros(P, int), starts, goals, batch.informed_rotations(starts, goals))
    states = batch.seed_states(np.arange(P))
    db.set_plans(desc)
    stream = torch.cuda.current_stream(dev)
    L = _lib.lib()

    # (a) device arm: the four stages of DeviceBatch.seed_informed + run(), timed with events
    def device_step(ev):
        st = torch.from_numpy(states.view(np.int64)).to(dev)
        cr = torch.zeros((P, 2), dtype=torch.int32, device=dev)
        st_s, cr_s = st.clone(), cr.clone()
        db.samples = db._empty((P, n, 2), torch.int16)
        balls = db._empty((P, n, 2), torch.float64)
        ev[0].record(stream)
        _lib.check(L.rrtk_sample_streams_carry(db._p(db.bits), db._p(db.rowcum), S, S, db._p(db.desc), P, db._p(st_s), db._p(cr_s), n,
                                               db._p(db.samples), stream.cuda_stream), "sample_streams_carry")
        ev[1].record(stream)
        db.balls = None
        db.run()
        ev[2].record(stream)
        _lib.check(L.rrtk_ball_streams(db._p(db.rowcum), S, db._p(db.desc), P, n, db._p(st), db._p(cr),
                                       db.out["stats"][:, 5].data_ptr(), _lib.STAT_COUNT, db._p(balls), None, None, stream.cuda_stream),
                   "ball_streams")
        ev[3].record(stream)
        db.balls = balls
        db.run()
        ev[4].record(stream)

    names = ("sample_streams", "probe", "ball_streams", "plan")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    device_step(ev)                                                      # warm-up
    torch.cuda.synchronize(dev)
    per = {k: [] for k in names}
    for _ in range(args.steps):
        device_step(ev)
        torch.cuda.synchronize(dev)
        for i, k in enumerate(names):
            per[k].append(ev[i].elapsed_time(ev[i + 1]))
    dev_stats = db.out["stats"].cpu().numpy()
    # the same through DeviceBatch.seed_informed: equal statistics
    db.seed_informed(states).run()
    same_api = bool(np.array_equal(db.download().stats[:, 5:], dev_stats[:, 5:]))
    ms = {k: float(np.mean(v)) for k, v in per.items()}
    total = sum(ms.values())
    first = dev_stats[:, 5]
    device = {"ms_per_step": total, "plans_per_s": P / (total / 1e3), "stage_ms": ms,
              "stage_share": {k: v / total for k, v in ms.items()}, "matches_seed_informed": same_api,
              "note": "mean over %d steps; CUDA events on one stream around each stage" % args.steps}

    # (b) end to end with the flag, (c) the host way
    ctx = _lib.Context()
    bits_host = _lib.pack_grids_host(og[None])
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()          # noqa: E731
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]

    def flagged():
        return ctx.plan_worlds2(_lib.KIND_INFORMED, bits_host, S, S, desc, n, R_REWIRE, R_GOAL, states=states, bits=True, trees=False,
                                paths=True, path_cap=PATH_CAP, seed_balls=True)

    def host_way():
        t0 = time.perf_counter()
        probe = ctx.plan_worlds2(_lib.KIND_INFORMED, bits_host, S, S, desc, n, R_REWIRE, R_GOAL, states=states, bits=True, trees=False,
                                 paths=False)
        t1 = time.perf_counter()
        balls = pin(host_balls(states, nfree, probe["stats"][:, 5], n))
        t2 = time.perf_counter()
        got = ctx.plan_worlds2(_lib.KIND_INFORMED, bits_host, S, S, desc, n, R_REWIRE, R_GOAL, states=states, balls=balls, bits=True,
                               trees=False, paths=True, path_cap=PATH_CAP)
        t3 = time.perf_counter()
        return got, (t1 - t0, t2 - t1, t3 - t2)

    flagged()
    tb = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        b = flagged()
        tb.append(time.perf_counter() - t0)
    tc, parts = [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        c, pt = host_way()
        tc.append(time.perf_counter() - t0)
        parts.append(pt)
    ctx.close()
    rec = ("path", "xy", "len", "path_cost")
    same = bool(np.array_equal(b["stats"][:, keep], c["stats"][:, keep]) and
                all(np.array_equal(b[k].view(np.uint8), c[k].view(np.uint8)) for k in rec))
    assert same, "seeded-ball and host-ball paths disagree"
    assert np.array_equal(b["stats"][:, keep], dev_stats[:, keep]), "end-to-end and device arm disagree"
    h2d_common = int(bits_host.nbytes + P * (64 + 32))
    d2h = int(P * (PATH_CAP * 8 + 12 + _lib.STAT_COUNT * 8))
    line = {
        "workload": "cfg4 shape: one %dx%d world, %d pairs, n=%d, r_rewire=%g, r_goal=%g, seeds 0..%d" % (S, S, P, n, R_REWIRE, R_GOAL, P - 1),
        "gpu": gpu_card(),
        "solution_found_frac": float((first >= 0).mean()),
        "mean_first_solution_iter": float(first[first >= 0].mean()) if (first >= 0).any() else None,
        "device": device,
        "e2e_seed_balls": {"plans_per_s": P / min(tb), "best_s": min(tb), "mean_s": float(np.mean(tb)), "h2d_bytes_per_step": h2d_common,
                           "d2h_bytes_per_step": d2h,
                           "api": "rrtk_ctx_plan_worlds2(RRTK_IN_BITS | RRTK_OUT_PATHS | RRTK_SEED_BALLS)"},
        "e2e_host_balls": {"plans_per_s": P / min(tc), "best_s": min(tc), "mean_s": float(np.mean(tc)),
                           "h2d_bytes_per_step": h2d_common * 2 + P * n * 16, "d2h_bytes_per_step": d2h + P * _lib.STAT_COUNT * 8,
                           "split_s_of_best": dict(zip(("probe_call", "numpy_draws", "plan_call"), parts[int(np.argmin(tc))])),
                           "api": "worlds2 probe + numpy draws per plan + worlds2 with h_balls (pinned)"},
        "identical_stats_and_paths": same,
        "steps": args.steps,
    }
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
