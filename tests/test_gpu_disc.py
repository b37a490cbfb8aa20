"""Configuration space of a disc robot on the GPU (csrc/disc.cu, rrtk_inflate_disc / rrtk_ctx_inflate_disc) against the scipy
oracles of tests/test_disc_host.py, bit for bit including padding bits; the robot_radius option of every planner class and of
plan_batch against the same planner on the scipy-inflated grid; DeviceBatch.inflate_disc; the cfg3 shape at full size."""
import math

import numpy as np
import pytest

from rrtplanner_b200 import RRTDubins, RRTStandard, RRTStar, RRTStarDubins, RRTStarInformed, _lib, batch, worlds
from tests.test_disc_host import blobs, cspace_edt, sq_dist_to_obstacle

pytestmark = pytest.mark.gpu

RADII = [0, 0.5, 1, math.sqrt(2), 1.5, 2, 3.9999, 7, 33, 100]


@pytest.fixture(scope="module")
def ctx():
    c = _lib.Context()
    yield c
    c.close()


def disc_worlds(W, H, seed):
    rng = np.random.default_rng(seed)
    single = np.zeros((W, H), dtype=np.uint8)
    single[rng.integers(0, W), rng.integers(0, H)] = 1
    border = np.zeros((W, H), dtype=np.uint8)
    border[0, rng.integers(0, H)] = border[W - 1, rng.integers(0, H)] = border[rng.integers(0, W), 0] = border[rng.integers(0, W), H - 1] = 1
    border[0, 0] = border[W - 1, H - 1] = 1
    return np.stack([blobs(W, H, seed, density=2000), np.zeros((W, H), np.uint8), np.ones((W, H), np.uint8), single, border,
                     (rng.random((W, H)) < 0.002).astype(np.uint8)])


@pytest.mark.parametrize("shape", [(64, 64), (43, 100), (100, 43), (33, 31), (130, 70), (512, 512), (1024, 1024), (3001, 45),
                                   (45, 3001)])
def test_kernel_against_the_oracle(ctx, shape):
    W, H = shape
    ogs = disc_worlds(W, H, W * 7 + H)
    nw = ogs.shape[0]
    radii = RADII + [math.sqrt((W - 1) ** 2 + (H - 1) ** 2), 1e9]
    # every world at every radius in one call, in a shuffled order: nout > nworlds, sources and radii mixed
    src = np.repeat(np.arange(nw), len(radii))
    rad = np.tile(radii, nw)
    perm = np.random.default_rng(W + H).permutation(src.size)
    src, rad = src[perm], rad[perm]
    r2 = _lib.disc_r2(rad)
    got = ctx.inflate_disc(ogs, src, r2)
    d2 = [sq_dist_to_obstacle(og) for og in ogs]
    want = _lib.pack_grids_host(np.stack([cspace_edt(ogs[s], int(q), d2[s]) for s, q in zip(src, r2)]))
    for o in range(src.size):
        assert np.array_equal(got[o], want[o]), (shape, int(src[o]), rad[o])
    # r2 = 0 is the grid itself; an empty world stays empty, a full one full
    assert np.array_equal(ctx.inflate_disc(ogs, np.arange(nw), np.zeros(nw)), _lib.pack_grids_host(ogs))
    # nothing to write
    assert ctx.inflate_disc(ogs, [], []).shape == (0, int(_lib.lib().rrtk_grid_words(W, H)))


def test_exact_disc_and_argument_checks(ctx):
    W, H = 200, 150
    og = np.zeros((1, W, H), np.uint8)
    og[0, 77, 61] = 1
    X, Y = np.indices((W, H))
    for rho in (1, math.sqrt(2), 3.9999, 7, 33, 100):
        r2 = int(_lib.disc_r2(rho))
        got = _lib.unpack_grids_host(ctx.inflate_disc(og, [0], [r2]), W, H)[0]
        assert np.array_equal(got, ((X - 77) ** 2 + (Y - 61) ** 2 <= r2).astype(np.uint8)), rho
    with pytest.raises(ValueError, match="source world"):
        ctx.inflate_disc(og, [1], [4])
    with pytest.raises(ValueError, match="r2"):
        ctx.inflate_disc(og, [0], [-1])


def test_device_entry_leaves_bad_outputs_unwritten():
    import torch
    W, H = 70, 50
    ogs = disc_worlds(W, H, 3)[:2]
    words = int(_lib.lib().rrtk_grid_words(W, H))
    bits = torch.from_numpy(_lib.pack_grids_host(ogs).view(np.int32)).cuda()
    src = torch.tensor([1, 5, 0, -1], dtype=torch.int32, device="cuda")
    r2 = torch.tensor([9, 9, -3, 4], dtype=torch.int32, device="cuda")
    out = torch.full((4, words), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    scratch = torch.empty(int(_lib.lib().rrtk_inflate_disc_scratch_bytes(2, W, H)), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(_lib.lib().rrtk_inflate_disc(bits.data_ptr(), 2, W, H, src.data_ptr(), r2.data_ptr(), 4, out.data_ptr(), scratch.data_ptr(), st))
    o = out.cpu().numpy()
    assert np.array_equal(o[0].view(np.uint32), _lib.pack_grids_host(cspace_edt(ogs[1], 9))[0])
    assert (o[1:] == 0x5A5A5A5A).all()
    _lib.check(_lib.lib().rrtk_inflate_disc(bits.data_ptr(), 2, W, H, None, None, 0, None, None, st))


# ---- planner classes ----------------------------------------------------------------------------------------------------------
def graph_rows(T):
    nodes = list(T.nodes)
    pts = np.stack([np.asarray(T.nodes[v]["pt"]) for v in nodes])
    edges = [(int(a), int(b)) for a, b in T.edges]
    dist = np.array([float(d["dist"]) for *_, d in T.edges(data=True)])
    cost = np.array([float(d["cost"]) for *_, d in T.edges(data=True)])
    heads = [T.nodes[v].get("heading") for v in nodes]
    return nodes, pts, edges, dist, cost, heads


def assert_same_graph(a, b):
    (Ta, gva), (Tb, gvb) = a, b
    assert int(gva) == int(gvb)
    na, pa, ea, da, ca, ha = graph_rows(Ta)
    nb, pb, eb, db, cb, hb = graph_rows(Tb)
    assert na == nb and ea == eb and ha == hb
    assert np.array_equal(pa, pb)
    assert np.array_equal(da.view(np.int64), db.view(np.int64)) and np.array_equal(ca.view(np.int64), cb.view(np.int64))


def free_pair(cs, seed):
    free = np.argwhere(cs == 0)
    rng = np.random.default_rng(seed)
    return free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]


CLASSES = {
    "standard": (lambda og, **k: RRTStandard(og, 600, pbar=False, **k), 2),
    "star": (lambda og, **k: RRTStar(og, 600, 12.0, pbar=False, **k), 2),
    "star_rrtstar": (lambda og, **k: RRTStar(og, 600, 12.0, pbar=False, rewire="rrtstar", **k), 2),
    "informed": (lambda og, **k: RRTStarInformed(og, 600, 12.0, 6.0, pbar=False, **k), 2),
    "dubins": (lambda og, **k: RRTDubins(og, 400, 3.0, 8, pbar=False, **k), 3),
    "star_dubins": (lambda og, **k: RRTStarDubins(og, 400, 10.0, 3.0, 8, pbar=False, **k), 3),
}


@pytest.mark.parametrize("name", list(CLASSES))
def test_class_plans_on_the_configuration_space(name):
    make, dims = CLASSES[name]
    W, H = 96, 80
    og = blobs(W, H, 5, density=700).astype(np.int64)
    og[3, 3] = 7                                                      # any non-zero value is an obstacle
    rho = 2.5
    cs = cspace_edt(og, int(_lib.disc_r2(rho)))
    for seed in (0, 3):
        a, b = free_pair(cs, 100 + seed)
        if dims == 3:
            a, b = np.array([*a, 1]), np.array([*b, 5])
        p = make(og, seed=seed, robot_radius=rho)
        assert p.og is og
        assert np.array_equal(p.free, np.argwhere(cs == 0))
        want = make(cs, seed=seed).plan(a.copy(), b.copy())
        assert_same_graph(p.plan(a.copy(), b.copy()), want)
        # shortcut_path works on the configuration space
        if dims == 2 and int(want[1]) > 0:
            q = make(cs, seed=seed)
            path = q.route2gv(want[0], want[1])
            assert p.shortcut_path(want[0], path) == q.shortcut_path(want[0], path)
        # set_og inflates the new grid (same radius)
        og2 = np.flipud(og).copy()
        p.set_og(og2)
        assert p.og is og2
        cs2 = cspace_edt(og2, int(_lib.disc_r2(rho)))
        assert np.array_equal(p.free, np.argwhere(cs2 == 0))
        a2, b2 = free_pair(cs2, 200 + seed)
        if dims == 3:
            a2, b2 = np.array([*a2, 2]), np.array([*b2, 6])
        q = make(cs, seed=seed)
        q.plan(a.copy(), b.copy())                                     # same generator position as p
        q.set_og(cs2)
        assert_same_graph(p.plan(a2.copy(), b2.copy()), q.plan(a2.copy(), b2.copy()))


@pytest.mark.parametrize("name", list(CLASSES))
def test_no_radius_and_zero_radius_are_todays_planner(name):
    make, dims = CLASSES[name]
    og = blobs(64, 72, 8, density=600)
    a, b = free_pair(og, 1)
    if dims == 3:
        a, b = np.array([*a, 0]), np.array([*b, 4])
    want = make(og, seed=4).plan(a.copy(), b.copy())
    for r in (None, 0, 0.5):
        p = make(og, seed=4, robot_radius=r)
        assert p.og is og and np.array_equal(p.free, np.argwhere(og == 0))
        assert_same_graph(p.plan(a.copy(), b.copy()), want)


def test_start_inside_the_inflated_obstacles_behaves_as_an_occupied_start():
    og = np.zeros((64, 64), np.uint8)
    og[30:34, 30:34] = 1
    start, goal = np.array([29, 31]), np.array([5, 60])               # free in og, blocked at radius 3
    p = RRTStar(og, 300, 10.0, pbar=False, seed=1, robot_radius=3)
    q = RRTStar(cspace_edt(og, 9), 300, 10.0, pbar=False, seed=1)
    assert_same_graph(p.plan(start, goal), q.plan(start, goal))
    assert int(p.last_stats["found"]) == 0


# ---- batches ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def three_worlds():
    W, H = 160, 128
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(w)) for w in (21, 22, 23)]).astype(np.uint8)
    P = 48
    wid = np.random.default_rng(4).permutation(np.arange(P) % 3)               # not sorted
    radii = np.random.default_rng(5).choice([0.0, 1.0, 2.5, 4.0], size=P)
    return ogs, wid, radii


def plans_for(ogs, wid, r2, seed):
    starts, goals = [], []
    for p in range(len(wid)):
        a, b = free_pair(cspace_edt(ogs[wid[p]], int(r2[p])), seed + p)
        starts.append(a)
        goals.append(b)
    return np.array(starts), np.array(goals)


KEEP = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]


@pytest.mark.parametrize("kind", ["standard", "star", "informed"])
@pytest.mark.parametrize("per_plan", [False, True])
def test_plan_batch_with_radius(three_worlds, kind, per_plan):
    ogs, wid, radii = three_worlds
    radius = radii if per_plan else 2.5
    r2 = _lib.disc_r2(np.broadcast_to(radius, wid.shape))
    starts, goals = plans_for(ogs, wid, r2, 40)
    seeds = 900 + np.arange(len(wid))
    n = 1500
    kw = dict(r_rewire=15.0, r_goal=6.0, balls="seed") if kind == "informed" else dict(r_rewire=15.0)
    res = batch.plan_batch(kind, ogs, n, starts, goals, world_ids=wid, seeds=seeds, robot_radius=radius, **kw)
    # the same plans, each on its own scipy-inflated world
    cs = np.stack([cspace_edt(ogs[wid[p]], int(r2[p])) for p in range(len(wid))])
    want = batch.plan_batch(kind, cs, n, starts, goals, world_ids=np.arange(len(wid)), seeds=seeds, **kw)
    for k in ("pts", "cost", "parent", "ell_c"):
        a, b = getattr(res, k), getattr(want, k)
        assert (a is None) == (b is None), k
        if a is not None:
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
    assert np.array_equal(res.stats[:, KEEP], want.stats[:, KEEP])
    assert res.stat("found").any()
    # and a few of them as single seeded planner objects on the inflated grid
    for p in (0, 7):
        if kind == "informed":
            q = RRTStarInformed(ogs[wid[p]], n, 15.0, 6.0, pbar=False, seed=int(seeds[p]), robot_radius=float(np.broadcast_to(radius, wid.shape)[p]))
        elif kind == "star":
            q = RRTStar(ogs[wid[p]], n, 15.0, pbar=False, seed=int(seeds[p]), robot_radius=float(np.broadcast_to(radius, wid.shape)[p]))
        else:
            q = RRTStandard(ogs[wid[p]], n, pbar=False, seed=int(seeds[p]), robot_radius=float(np.broadcast_to(radius, wid.shape)[p]))
        assert_same_graph(q._finish(res.pts[p], res.cost[p], res.parent[p], res.stats[p]), q.plan(starts[p].copy(), goals[p].copy()))


def test_plan_batch_with_host_samples(three_worlds):
    ogs, wid, radii = three_worlds
    r2 = _lib.disc_r2(radii)
    starts, goals = plans_for(ogs, wid, r2, 70)
    n = 800
    rng = np.random.default_rng(2)
    samples = np.stack([np.argwhere(cspace_edt(ogs[wid[p]], int(r2[p])) == 0)[rng.integers(0, 1000, n) % 1000] for p in range(len(wid))])
    res = batch.plan_batch("star", ogs, n, starts, goals, world_ids=wid, r_rewire=12.0, samples=samples, robot_radius=radii)
    cs = np.stack([cspace_edt(ogs[wid[p]], int(r2[p])) for p in range(len(wid))])
    want = batch.plan_batch("star", cs, n, starts, goals, world_ids=np.arange(len(wid)), r_rewire=12.0, samples=samples)
    assert np.array_equal(res.parent, want.parent) and np.array_equal(res.cost.view(np.int64), want.cost.view(np.int64))


@pytest.mark.parametrize("two", [False, True])
def test_device_batch_inflate_disc(three_worlds, two):
    ogs, _, _ = three_worlds
    W, H = ogs.shape[1:]
    radius = [1.0, 3.5, 0.0]
    r2 = _lib.disc_r2(radius)
    cs = np.stack([cspace_edt(ogs[w], int(r2[w])) for w in range(3)])
    mk = (lambda: batch.DeviceBatch2("euclid", W, H, 700, r_rewire=12.0)) if two else (lambda: batch.DeviceBatch("star", W, H, 700, 12.0))
    a = mk().set_worlds_host(ogs).inflate_disc(radius)
    b = mk().set_worlds_host(cs)
    assert np.array_equal(a.bits.cpu().numpy(), b.bits.cpu().numpy())
    assert np.array_equal(a.rowcum.cpu().numpy(), b.rowcum.cpu().numpy())
    assert np.array_equal(a.og.cpu().numpy(), ogs)                     # og keeps the worlds as given
    starts, goals = plans_for(ogs, [0, 1, 2, 1], r2[[0, 1, 2, 1]], 11)
    desc = batch.make_desc([0, 1, 2, 1], starts, goals)
    outs = []
    for db in (a, b):
        db.set_plans(desc).seed_samples([1, 2, 3, 4]).run()
        rec = db.shortcut_records(db.path_records(64))
        outs.append((db.download(), {k: v.cpu().numpy() for k, v in rec.items()}))
    (ra, pa), (rb, pb) = outs
    assert np.array_equal(ra.parent, rb.parent) and np.array_equal(ra.cost.view(np.int64), rb.cost.view(np.int64))
    for k in ("xy", "len", "path_cost"):
        assert np.array_equal(pa[k], pb[k]), k
    # a scalar radius
    c = mk().set_worlds_host(ogs).inflate_disc(2)
    assert np.array_equal(c.bits.cpu().numpy().view(np.uint32), _lib.pack_grids_host(np.stack([cspace_edt(og, 4) for og in ogs])))
    with pytest.raises(ValueError):
        mk().set_worlds_host(ogs).inflate_disc([1.0, 2.0])


# ---- cfg3 shape at full size --------------------------------------------------------------------------------------------------
def test_cfg3_full_size_radius_4():
    import torch
    W = H = 512
    n, P, rho = 5000, 4096, 4
    r2 = int(_lib.disc_r2(rho))
    db = batch.DeviceBatch("star", W, H, n, 50.0).gen_worlds(1000 + np.arange(P))
    og = db.og.cpu().numpy()
    db.inflate_disc(rho)
    bits = db.bits.cpu().numpy().view(np.uint32)
    sample = np.random.default_rng(0).choice(P, 64, replace=False)
    for w in sample:
        assert np.array_equal(bits[w], _lib.pack_grids_host(cspace_edt(og[w], r2))[0]), int(w)
    cs = _lib.unpack_grids_host(bits, W, H)
    pairs = []
    for p in range(P):
        free = np.argwhere(cs[p] == 0)
        rng = np.random.default_rng(p)
        pairs.append((free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]))
    db.set_plans(batch.make_desc(np.arange(P), [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(P)).run()
    out = db.out
    parent = out["parent"]
    child = parent >= 0
    pw, cidx = torch.nonzero(child, as_tuple=True)
    par = parent[pw, cidx].long()
    segs = torch.cat([out["pts"][pw, par], out["pts"][pw, cidx]], dim=1).int().contiguous()
    world = pw.int().contiguous()
    free = torch.empty(segs.shape[0], dtype=torch.uint8, device=segs.device)
    _lib.check(db.L.rrtk_collision_segments(db.bits.data_ptr(), W, H, segs.data_ptr(), world.data_ptr(), segs.shape[0], free.data_ptr(),
                                            None, db._stream()))
    assert segs.shape[0] > P and bool((free == 1).all())
    res = db.download()
    assert res.stat("found").any()
    # every vertex keeps d^2 > r2 from every obstacle cell of its original world
    filled = res.pts[:, :, 0] != -32768
    pw, vi = np.nonzero(filled)
    x, y = res.pts[pw, vi, 0].astype(np.int64), res.pts[pw, vi, 1].astype(np.int64)
    R = math.isqrt(r2)
    for i in range(-R, R + 1):
        for j in range(-R, R + 1):
            if i * i + j * j > r2:
                continue
            u, v = x + i, y + j
            inside = (u >= 0) & (u < W) & (v >= 0) & (v < H)
            hit = og[pw[inside], u[inside], v[inside]] != 0
            assert not hit.any(), (i, j)
