"""Seeded informed batches on the GPU: rrtk_ball_streams against numpy's generator, and plan_batch(balls="seed"),
DeviceBatch.seed_informed / DeviceBatch2.seed_informed, plan_worlds2 / plan2_worlds(seed_balls=True) against the seeded
RRTStarInformed class and the reference's own trees (tests/golden/seeded_api.npz)."""
import os

import numpy as np
import pytest

from rrtplanner_b200 import _lib, batch, worlds
from rrtplanner_b200.rrt import RRTStarInformed
from tests.conftest import GOLDEN
from tests.test_gpu_api import graph_matches

pytestmark = pytest.mark.gpu

FIRST = _lib.STAT_NAMES.index("first_solution_iter")


def words_of(g: np.random.Generator):
    st = g.bit_generator.state
    m = (1 << 64) - 1
    s, inc = st["state"]["state"], st["state"]["inc"]
    return np.array([s >> 64, s & m, inc >> 64, inc & m], dtype=np.uint64), np.array([st["has_uint32"], st["uinteger"]], dtype=np.uint32)


def class_stream(g: np.random.Generator, nfree: int, f: int, n: int) -> np.ndarray:
    """What RRTStarInformed.plan does to its generator: f + 1 (n when f < 0) bounded draws, then unitball() per
    ellipse-phase iteration; rows <= f are zero."""
    g.integers(0, nfree, size=n if f < 0 else f + 1)
    balls = np.zeros((n, 2))
    if f >= 0:
        for i in range(f + 1, n):
            u = g.uniform(0, 1)
            a = 2 * np.pi * g.uniform(0, 1)
            balls[i] = [np.sqrt(u) * np.cos(a), np.sqrt(u) * np.sin(a)]
    return balls


def ulps(a, b):
    def ordered(x):
        i = np.ascontiguousarray(x, dtype=np.float64).view(np.int64)
        return np.where(i < 0, np.int64(-0x8000000000000000) - i, i)
    return np.abs(ordered(a) - ordered(b))


def test_ball_streams_match_numpy():
    import torch
    n, S = 600, 2048
    ogs = np.ones((3, S, S), dtype=np.uint8)
    ogs[0, 700, 900] = 0                                                  # nfree = 1
    rng = np.random.default_rng(5)
    ogs[1].reshape(-1)[rng.choice(S * S, 37, replace=False)] = 0          # nfree = 37
    ogs[2] = worlds.perlin_occupancygrid(S, S, seed=worlds.world_seed(3)).astype(np.uint8)
    nfree = (ogs == 0).reshape(3, -1).sum(axis=1)
    assert nfree[0] == 1 and nfree[1] == 37 and nfree[2] > 1_000_000
    P = 48
    wid = np.arange(P) % 3
    fs = np.array([[-1, 0, 1, n - 1][p % 4] if p < 24 else int(rng.integers(0, n - 1)) for p in range(P)])
    states, carry, gens = np.zeros((P, 4), np.uint64), np.zeros((P, 2), np.uint32), []
    for p in range(P):
        g = np.random.default_rng(300 + p)
        if p % 3 == 1:
            g.integers(0, 1000, size=3)                                   # odd number of 32-bit draws: has_uint32 = 1
        elif p % 3 == 2:
            g.integers(0, 1000, size=4)
            g.uniform(0, 1)
        states[p], carry[p] = words_of(g)
        gens.append(g)
    assert carry[1::3, 0].all() and not carry[2::3, 0].any()
    db = batch.DeviceBatch("informed", S, S, n, 30.0, 5.0, device=0).set_worlds_host(ogs)
    db.set_plans(batch.make_desc(wid, np.zeros((P, 2)), np.ones((P, 2))))
    dev = db.dev
    first = np.full((P, 3), 12345, dtype=np.int64)
    first[:, 1] = fs                                                       # read with a stride
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).to(dev)   # noqa: E731
    d_st, d_cr, d_first = t(states, np.int64), t(carry, np.int32), t(first, np.int64)
    balls = torch.full((P, n, 2), 7.0, dtype=torch.float64, device=dev)
    st_out, cr_out = torch.empty_like(d_st), torch.empty_like(d_cr)
    L = _lib.lib()
    _lib.check(L.rrtk_ball_streams(db.rowcum.data_ptr(), S, db.desc.data_ptr(), P, n, d_st.data_ptr(), d_cr.data_ptr(),
                                   d_first.data_ptr() + 8, 3, balls.data_ptr(), st_out.data_ptr(), cr_out.data_ptr(),
                                   torch.cuda.current_stream(dev).cuda_stream), "ball_streams")
    # the fresh-generator form (no carry in / out) and in-place state update
    fresh = np.array([p for p in range(P) if p % 3 == 0])
    d_st2 = t(states[fresh], np.int64)
    desc_f = db.desc[torch.from_numpy(fresh).to(dev)].contiguous()
    balls2 = torch.empty((fresh.size, n, 2), dtype=torch.float64, device=dev)
    d_first2 = t(fs[fresh].astype(np.int64), np.int64)
    _lib.check(L.rrtk_ball_streams(db.rowcum.data_ptr(), S, desc_f.data_ptr(), fresh.size, n, d_st2.data_ptr(), None, d_first2.data_ptr(), 1,
                                   balls2.data_ptr(), d_st2.data_ptr(), None, torch.cuda.current_stream(dev).cuda_stream), "ball_streams")
    torch.cuda.synchronize(dev)
    got, got_st, got_cr = balls.cpu().numpy(), st_out.cpu().numpy().view(np.uint64), cr_out.cpu().numpy().view(np.uint32)
    assert np.array_equal(balls2.cpu().numpy().view(np.int64), got[fresh].view(np.int64))
    assert np.array_equal(d_st2.cpu().numpy().view(np.uint64), got_st[fresh])
    worst, equal, total = 0, 0, 0
    for p in range(P):
        f = int(fs[p])
        want = class_stream(gens[p], int(nfree[wid[p]]), f, n)
        lo = f + 1 if f >= 0 else n
        assert np.array_equal(got[p, :lo].view(np.int64), np.zeros((lo, 2), dtype=np.int64)), p      # exactly +0.0
        if lo < n:
            u = ulps(got[p, lo:], want[lo:])
            worst, equal, total = max(worst, int(u.max())), equal + int((u == 0).sum()), total + u.size
            assert u.max() <= 4, (p, int(u.max()))
        w_st, w_cr = words_of(gens[p])
        assert np.array_equal(got_st[p], w_st), p
        assert np.array_equal(got_cr[p], w_cr), p
    print(f"ball streams vs numpy: max {worst} ulp, {equal}/{total} coordinates bit-equal ({equal / total:.6f})")


# ---- pinned to the reference: tests/golden/seeded_api.npz ----------------------------------------------------------------
@pytest.fixture(scope="module")
def seeded():
    z = np.load(os.path.join(GOLDEN, "seeded_api.npz"))
    d = {k: z[k] for k in z.files}
    w, h = (int(v) for v in d["og_shape"])
    d["og"] = np.unpackbits(d["og"], axis=1)[:, :h].astype(np.int64)
    return d


def batch_graph(helper, pts, cost, parent, stats):
    return helper._finish(pts, cost, parent, stats)


def test_reference_informed_trees_through_the_batch_paths(seeded):
    og = seeded["og"]
    n, r, rg, seed = 500, 30, 10, 44
    helper = RRTStarInformed(og, n, r, rg, pbar=False)
    xs, xg, xs2, xg2 = seeded["xs"], seeded["xg"], seeded["xs2"], seeded["xg2"]
    res = batch.plan_batch("informed", og, n, [xs], [xg], r_rewire=r, r_goal=rg, seeds=[seed], balls="seed")
    T, gv = batch_graph(helper, res.pts[0], res.cost[0], res.parent[0], res.stats[0])
    graph_matches(T, gv, seeded, "informed0")
    assert np.flatnonzero(~np.isnan(res.ell_c[0])).tolist() == [int(k) for k in seeded["informed0_ell_keys"]]
    W, H = og.shape
    db = batch.DeviceBatch("informed", W, H, n, r, rg, device=0).set_worlds_host(og[None])
    state_out = carry_out = None
    keys = set()
    for rep, (a, b) in enumerate(((xs, xg), (xs2, xg2))):
        db.set_plans(batch.make_desc([0], [a], [b], batch.informed_rotations([a], [b])))
        if rep == 0:
            db.seed_informed(batch.seed_states([seed]))
        else:
            db.seed_informed(state_out, carry_out)                       # the second plan() of the same object
        out = db.run().download()
        state_out, carry_out = db.state_out.clone(), db.carry_out.clone()
        T, gv = batch_graph(helper, out.pts[0], out.cost[0], out.parent[0], out.stats[0])
        graph_matches(T, gv, seeded, f"informed{rep}")
        # the object's ellipses dict keeps the keys of every plan() so far (rrt.py:701)
        keys |= set(np.flatnonzero(~np.isnan(out.ell_c[0])).tolist())
        assert sorted(keys) == [int(k) for k in seeded[f"informed{rep}_ell_keys"]]
    # the generator after both plans is where the seeded object's generator stands
    p = RRTStarInformed(og, n, r, rg, pbar=False, seed=seed)
    p.plan(xs.copy(), xg.copy())
    p.plan(xs2.copy(), xg2.copy())
    w_st, w_cr = words_of(p.rand_gen)
    assert np.array_equal(state_out.cpu().numpy().view(np.uint64)[0], w_st)
    assert np.array_equal(carry_out.cpu().numpy().view(np.uint32)[0], w_cr)


# ---- class equivalence -----------------------------------------------------------------------------------------------------
TREE_STATS = ("j", "vgoal", "found", "first_solution_iter", "ellipse_iters")


def assert_tree_equals_class(og, n, r, rg, seed, xs, xg, pts, cost, parent, stats, ell, names=_lib.STAT_NAMES, rewire="reference"):
    p = RRTStarInformed(og, n, r, rg, pbar=False, seed=int(seed), rewire=rewire)
    T, gv = p.plan(np.asarray(xs).copy(), np.asarray(xg).copy())
    helper = RRTStarInformed(og, n, r, rg, pbar=False)
    Tb, gvb = helper._finish(pts, cost, parent, stats)
    assert int(gv) == int(gvb)
    assert list(T.nodes) == list(Tb.nodes)
    assert np.array_equal(np.stack([T.nodes[v]["pt"] for v in T.nodes]), np.stack([Tb.nodes[v]["pt"] for v in Tb.nodes]))
    ea, eb = list(T.edges(data=True)), list(Tb.edges(data=True))
    assert [(a, b) for a, b, _ in ea] == [(a, b) for a, b, _ in eb]
    assert np.array_equal(np.array([float(d["cost"]) for *_, d in ea]).view(np.int64), np.array([float(d["cost"]) for *_, d in eb]).view(np.int64))
    st = dict(zip(names, (int(v) for v in stats)))
    keys = ("j", "vgoal", "found", "first_solution_iter", "ell_iters", "rewires") if rewire == "rrtstar" else TREE_STATS
    for k in keys:
        assert p.last_stats[k] == st[k], k
    if ell is not None:
        assert sorted(p.ellipses) == np.flatnonzero(~np.isnan(ell)).tolist()
    return st


@pytest.fixture(scope="module")
def three_worlds():
    W, H = 256, 192
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(w)) for w in (11, 12, 13)]).astype(np.uint8)
    P = 96
    wid = np.random.default_rng(9).permutation(np.arange(P) % 3)           # not sorted
    pairs = [worlds.start_goal(ogs[wid[p]], 500 + p) for p in range(P)]
    return ogs, wid, np.array([a for a, _ in pairs]), np.array([b for _, b in pairs]), 7000 + np.arange(P)


def test_batch_equals_the_seeded_class(three_worlds):
    ogs, wid, starts, goals, seeds = three_worlds
    n, r, rg = 3000, 20.0, 6.0
    res = batch.plan_batch("informed", ogs, n, starts, goals, world_ids=wid, r_rewire=r, r_goal=rg, seeds=seeds, balls="seed")
    firsts = res.stat("first_solution_iter")
    assert (firsts >= 0).any()
    for p in range(len(seeds)):
        assert_tree_equals_class(ogs[wid[p]], n, r, rg, seeds[p], starts[p], goals[p], res.pts[p], res.cost[p], res.parent[p],
                                 res.stats[p], res.ell_c[p])
    # the pipelined call with the flag: uint8 and bit grids, default chunks and chunks of 7, trees and path records
    order = np.argsort(wid, kind="stable")
    desc = batch.make_desc(wid[order], starts[order], goals[order], batch.informed_rotations(starts[order], goals[order]))
    states = batch.seed_states(seeds[order])
    ctx = _lib.Context()
    W, H = ogs.shape[1:]
    ref = None
    for grids, bits in ((ogs, False), (_lib.pack_grids_host(ogs), True)):
        for chunk in (0, 7):
            o = ctx.plan_worlds2(_lib.KIND_INFORMED, grids, W, H, desc, n, r, rg, states=states, bits=bits, trees=True, paths=True,
                                 chunk=chunk, seed_balls=True)
            for k, a in (("pts", res.pts), ("cost", res.cost), ("parent", res.parent), ("ell", res.ell_c)):
                assert np.array_equal(o[k].view(np.uint8), a[order].view(np.uint8)), (k, bits, chunk)
            keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
            assert np.array_equal(o["stats"][:, keep], res.stats[order][:, keep])
            rec = {k: o[k].copy() for k in ("path", "xy", "len", "path_cost")}
            if ref is None:
                ref = rec
            for k in rec:
                assert np.array_equal(rec[k].view(np.uint8), ref[k].view(np.uint8)), k
    ctx.close()


# ---- cfg4 at full size -----------------------------------------------------------------------------------------------------
def test_cfg4_full_size():
    S, n, P, r, rg = 1024, 20000, 1024, 50.0, 5.0
    db = batch.DeviceBatch("informed", S, S, n, r, rg, device=0).gen_worlds([worlds.world_seed(0)])
    og = db.og[0].cpu().numpy()
    starts, goals = [], []
    for p in range(P):
        a, b = worlds.start_goal(og, p)
        starts.append(a); goals.append(b)
    starts, goals = np.array(starts), np.array(goals)
    desc = batch.make_desc(np.zeros(P, int), starts, goals, batch.informed_rotations(starts, goals))
    states = batch.seed_states(np.arange(P))
    db.set_plans(desc).seed_informed(states)
    dev_stats = db.run().download().stats
    ctx = _lib.Context()
    o = ctx.plan_worlds2(_lib.KIND_INFORMED, _lib.pack_grids_host(og[None]), S, S, desc, n, r, rg, states=states, bits=True, trees=False,
                         paths=True, seed_balls=True)
    ctx.close()
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    assert np.array_equal(o["stats"][:, keep], dev_stats[:, keep])
    f = dev_stats[:, FIRST]
    assert (f < 0).any() and (f >= 0).any()
    picks = sorted({int(np.flatnonzero(f < 0)[0]), int(np.argmax(f)), int(np.flatnonzero(f >= 0)[0]), P // 2})
    res = db.download()
    for p in picks:
        assert_tree_equals_class(og, n, r, rg, p, starts[p], goals[p], res.pts[p], res.cost[p], res.parent[p], res.stats[p], res.ell_c[p])


# ---- K8: the rewire that fires ---------------------------------------------------------------------------------------------
def test_k8_seed_informed_equals_the_class():
    og = worlds.perlin_occupancygrid(120, 96, seed=33).astype(np.uint8)
    W, H = og.shape
    n, r, rg, P = 1200, 25.0, 8.0, 16
    pairs = [worlds.start_goal(og, 40 + p) for p in range(P)]
    starts, goals = np.array([a for a, _ in pairs]), np.array([b for _, b in pairs])
    seeds = 100 + np.arange(P)
    desc = batch.make_desc(np.zeros(P, int), starts, goals, batch.informed_rotations(starts, goals))
    db = batch.DeviceBatch2("euclid", W, H, n, r_rewire=r, star=True, rewire=True, informed=True, r_goal=rg, device=0)
    db.set_worlds_host(og[None]).set_plans(desc).seed_informed(batch.seed_states(seeds))
    out = db.run().download()
    ell = db.out["ell"].cpu().numpy()
    assert (out.stat("first_solution_iter") >= 0).any()
    for p in range(P):
        assert_tree_equals_class(og, n, r, rg, seeds[p], starts[p], goals[p], out.pts[p], out.cost[p], out.parent[p], out.stats[p], ell[p],
                                 names=_lib.STAT2_NAMES, rewire="rrtstar")
    ctx = _lib.Context()
    cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, r, informed=True, r_goal=rg)
    o = ctx.plan2_worlds(cfg, og[None], W, H, desc, n, states=batch.seed_states(seeds), trees=True, paths=False, seed_balls=True, chunk=5)
    ctx.close()
    for k, a in (("pts", out.pts), ("cost", out.cost), ("parent", out.parent), ("ell", ell)):
        assert np.array_equal(o[k].view(np.uint8), a.view(np.uint8)), k
    assert np.array_equal(o["stats"][:, [0, 1, 2, 5, 10, 11]], out.stats[:, [0, 1, 2, 5, 10, 11]])


# ---- edge cases ------------------------------------------------------------------------------------------------------------
def test_edge_cases():
    og = worlds.perlin_occupancygrid(96, 96, seed=3).astype(np.uint8)
    free = np.argwhere(og == 0)
    a, b = free[10], free[-10]
    n, r = 1500, 20.0
    # start == goal with a reachable goal region: the class and the batch both raise
    with pytest.raises(np.linalg.LinAlgError):
        RRTStarInformed(og, n, r, 6.0, pbar=False, seed=1).plan(a.copy(), a.copy())
    with pytest.raises(np.linalg.LinAlgError, match="plan 1"):
        batch.plan_batch("informed", og, n, [a, a], [b, a], r_rewire=r, r_goal=6.0, seeds=[0, 1], balls="seed")
    # r_goal = 0: no solution vertex, so the plan never needs the rotation and is planned like the class plans it
    res = batch.plan_batch("informed", og, n, [a, a], [b, a], r_rewire=r, r_goal=0.0, seeds=[0, 1], balls="seed")
    assert (res.stat("first_solution_iter") < 0).all()
    for p, (x, y) in enumerate(((a, b), (a, a))):
        assert_tree_equals_class(og, n, r, 0.0, p, x, y, res.pts[p], res.cost[p], res.parent[p], res.stats[p], res.ell_c[p])
    # a world without a free cell has nothing to draw: the seed-mode error
    two = np.stack([og, np.ones_like(og)])
    with pytest.raises(ValueError, match="no free cell"):
        batch.plan_batch("informed", two, n, [a, a], [b, b], world_ids=[0, 1], r_rewire=r, r_goal=6.0, seeds=[0, 1], balls="seed")
