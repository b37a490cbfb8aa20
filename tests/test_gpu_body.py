"""Bodies with a heading on the GPU: rrtk_inflate_body against the scipy reference bit for bit, K8 on heading layers
(rrtk_plan2_batch_layers) against the layered specification of oracle/body_oracle.c, every Python entry point, and the
safety and corridor properties a car-shaped body is for."""
import math

import numpy as np
import pytest

from oracle import body_oracle as B
from oracle.rrt_oracle import ellipse_rotation
from rrtplanner_b200 import DeviceBatch2, RRTDubins, RRTStarDubins, _lib, dubins_collisionfree, dubins_points
from rrtplanner_b200.batch import make_desc, make_desc2
from rrtplanner_b200.body import DM_TWO_PI, body_layer, body_runs, car_body

pytestmark = pytest.mark.gpu

CAR = car_body(8, 2, 2.5, 16)


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _inflate(torch, og, stencils, proj=True):
    """Raw words of rrtk_inflate_body: (layers (nw, L, words), proj (nw, words) or None)."""
    og = np.ascontiguousarray(np.asarray(og) != 0, dtype=np.uint8)
    nw, W, H = og.shape
    runs, lr = body_runs(stencils)
    L = lr.shape[0] - 1
    lib = _lib.lib()
    words = int(lib.rrtk_grid_words(W, H))
    bits = torch.from_numpy(_lib.pack_grids_host(og).view(np.int32)).cuda()
    d_runs = torch.from_numpy(np.concatenate([runs.reshape(-1), np.zeros(1, np.int32)])).cuda()
    d_lr = torch.from_numpy(lr).cuda()
    layers = torch.full((nw * L, words), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    pj = torch.full((nw, words), 0x5A5A5A5A, dtype=torch.int32, device="cuda") if proj else None
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.rrtk_inflate_body(bits.data_ptr(), nw, W, H, d_runs.data_ptr(), d_lr.data_ptr(), L, layers.data_ptr(),
                                     None if pj is None else pj.data_ptr(), st), "inflate_body")
    torch.cuda.synchronize()
    lw = layers.cpu().numpy().view(np.uint32).reshape(nw, L, words)
    return lw, None if pj is None else pj.cpu().numpy().view(np.uint32)


def _want(og, stencils):
    lay = np.stack([B.layers_scipy(g, stencils) for g in og])           # (nw, L, W, H)
    nw, L, W, H = lay.shape
    lw = _lib.pack_grids_host(lay.reshape(nw * L, W, H)).reshape(nw, L, -1)
    return lw, _lib.pack_grids_host(np.stack([B.projection(x) for x in lay]))


def _worlds(rng, W, H):
    empty = np.zeros((W, H), np.uint8)
    full = np.ones((W, H), np.uint8)
    single = empty.copy()
    single[W // 2, H // 2] = 1
    border = empty.copy()
    border[0, :] = border[-1, :] = border[:, 0] = border[:, -1] = 1
    rand = (rng.random((W, H)) < 0.05).astype(np.uint8)
    return np.stack([empty, full, single, border, rand])


def _asym(rng, L, S, p=0.3):
    s = rng.random((L, S, S)) < p
    s[:, (S - 1) // 2, (S - 1) // 2] = True
    return s


@pytest.mark.parametrize("W, H", [(37, 45), (3001, 40), (1, 100), (100, 1), (64, 64), (70, 33)])
@pytest.mark.parametrize("stencil", ["point1", "point16", "asym16", "car64", "wide255"])
def test_inflate_body_bit_exact(torch, W, H, stencil):
    rng = np.random.default_rng(W * 7 + H)
    s = {"point1": lambda: np.ones((1, 1, 1), bool),
         "point16": lambda: np.ones((16, 1, 1), bool),
         "asym16": lambda: _asym(rng, 16, 9),                      # asymmetric, rows with several runs
         "car64": lambda: car_body(5, 2, 1.5, 64, 0.7),
         "wide255": lambda: _asym(rng, 1, 255, 0.002)}[stencil]()
    og = _worlds(rng, W, H)
    lw, pw = _inflate(torch, og, s)
    wl, wp = _want(og, s)
    assert np.array_equal(lw, wl)
    assert np.array_equal(pw, wp)
    lw2, none = _inflate(torch, og[3:], s, proj=False)
    assert none is None and np.array_equal(lw2, wl[3:])


def test_inflate_body_rejects_bad_runs(torch):
    lib = _lib.lib()
    bits = torch.zeros(1024, dtype=torch.int32, device="cuda")
    out = torch.zeros(4096, dtype=torch.int32, device="cuda")
    for runs, lr, L in [([0, 1, 2], [0, 1], 1),              # no centre
                        ([0, -1, 1], [0, 1], 0),              # no layer
                        ([0, 2, 1], [0, 1], 1),               # lo > hi
                        ([128, 0, 0, 0, 0, 0], [0, 2], 1)]:   # outside 255 x 255
        d_runs = torch.tensor(runs, dtype=torch.int32, device="cuda")
        d_lr = torch.tensor(lr, dtype=torch.int32, device="cuda")
        rc = lib.rrtk_inflate_body(bits.data_ptr(), 1, 32, 32, d_runs.data_ptr(), d_lr.data_ptr(), L, out.data_ptr(), None,
                                   torch.cuda.current_stream().cuda_stream)
        assert rc == -1


# ---- K8 on heading layers against the layered specification ------------------------------------------------
def _case(seed, W=72, H=64, p=0.004):
    rng = np.random.default_rng(seed)
    og = (rng.random((W, H)) < p).astype(np.uint8)
    start, goal = (6, 8, 0), (W - 9, H - 10, 5)
    og[max(0, start[0] - 4): start[0] + 10, max(0, start[1] - 4): start[1] + 5] = 0
    og[goal[0] - 10: goal[0] + 4, goal[1] - 4: goal[1] + 5] = 0
    return rng, og, start, goal


def _batch(og, start, goal, smp, star, rewire, r, nh, rho, stencils, use_table=True, threads=0, informed=None):
    W, H = og.shape
    n = smp.shape[0]
    b = DeviceBatch2("dubins", W, H, n, r_rewire=r, star=star, rewire=rewire, nheadings=nh, rho=rho, ds=1.0, threads=threads,
                     use_table=use_table, informed=informed is not None, r_goal=0.0 if informed is None else informed["r_goal"])
    b.set_worlds_host(og[None])
    if stencils is not None:
        b.inflate_body(stencils)
    d = make_desc2([0], [start], [goal])
    if informed is not None:
        d["rot"][0] = np.asarray(informed["rot"]).reshape(4)
    b.set_plans(d).set_samples_host(smp[None, :, :2]).set_heads_host(smp[None, :, 2])
    if informed is not None and informed.get("balls") is not None:
        b.set_balls_host(informed["balls"][None])
    b.run()
    res = b.download()
    ell = b.out["ell"].cpu().numpy()[0] if informed is not None else None
    return res, ell


def _same_bits(a, b):
    """Equal float64 arrays bit for bit, any NaN equal to any NaN (the device's and numpy's NaN differ in sign)."""
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64))


# the number of edge tests ("checks") is the one statistic the kernel does not fix: warps stop testing candidates once a cheaper
# free one is known, and when that becomes known depends on timing
DETERMINISTIC = [i for i, k in enumerate(_lib.STAT2_NAMES) if k != "checks"]


def _same(res, want, p=0):
    st = dict(zip(_lib.STAT2_NAMES, (int(v) for v in res.stats[p])))
    ws = want["stats"]
    for k in ("j", "vgoal", "found", "accepted", "rewires", "propagated", "ring_members"):
        assert st[k] == ws[k], (k, st[k], ws[k])
    top = ws["j"] + (1 if ws["found"] else 0)
    assert np.array_equal(res.pts[p, :top].astype(np.int32), want["pts"][:top])
    assert np.array_equal(res.head[p, :top].astype(np.int32), want["head"][:top])
    assert np.array_equal(res.parent[p, :top], want["parent"][:top])
    assert np.array_equal(res.cost[p, :top].view(np.int64), want["cost"][:top].view(np.int64))
    assert np.array_equal(res.elen[p, :top].view(np.int64), want["elen"][:top].view(np.int64))


@pytest.mark.parametrize("star, rewire", [(False, False), (True, False), (True, True)])
@pytest.mark.parametrize("L, use_table, threads", [(16, True, 0), (16, False, 128), (8, True, 128), (5, False, 256)])
def test_layered_plans_bit_exact_against_the_specification(star, rewire, L, use_table, threads):
    rng, og, start, goal = _case(L * 3 + star + 2 * rewire)
    n, nh, rho, r = 400, 16, 4.0, 14.0
    stencils = car_body(4, 1, 1.5, L)
    layers = B.layers_scipy(og, stencils).astype(np.uint8)
    free = np.argwhere(B.projection(layers) == 0)
    cells = free[rng.integers(0, free.shape[0], n)]
    smp = np.concatenate([cells, rng.integers(0, nh, (n, 1))], axis=1)
    want = B.plan_layers(layers, n, start, goal, smp, star=star, rewire=rewire, r_rewire=r, nh=nh, rho=rho, ds=1.0)
    res, _ = _batch(og, start, goal, smp, star, rewire, r, nh, rho, stencils, use_table, threads)
    _same(res, want)
    assert want["stats"]["accepted"] > 20
    if rewire:
        assert want["stats"]["rewires"] > 0


@pytest.mark.parametrize("rewire, threads", [(False, 0), (True, 128)])
def test_layered_informed_plans_bit_exact(rewire, threads):
    rng, og, start, goal = _case(21 + rewire)
    n, nh, rho, r = 400, 16, 4.0, 14.0
    layers = B.layers_scipy(og, CAR).astype(np.uint8)
    free = np.argwhere(B.projection(layers) == 0)
    smp = np.concatenate([free[rng.integers(0, free.shape[0], n)], rng.integers(0, nh, (n, 1))], axis=1)
    u, a = rng.random(n), rng.random(n) * 2 * math.pi
    balls = np.stack([np.sqrt(u) * np.cos(a), np.sqrt(u) * np.sin(a)], axis=1)
    inf = dict(r_goal=12.0, rot=ellipse_rotation(np.array(start[:2]), np.array(goal[:2])), balls=balls)
    want = B.plan_layers(layers, n, start, goal, smp, star=True, rewire=rewire, r_rewire=r, nh=nh, rho=rho, ds=1.0, informed=inf)
    res, ell = _batch(og, start, goal, smp, True, rewire, r, nh, rho, CAR, threads=threads, informed=inf)
    _same(res, want)
    assert _same_bits(ell, want["ell"])
    assert res.stat("ell_iters")[0] > 0


# ---- one point layer is no body at all ------------------------------------------------------------------------
def test_one_point_layer_equals_no_body_through_every_entry():
    point = np.ones((1, 1, 1), bool)
    rng, og, start, goal = _case(5)
    n, nh = 300, 16
    free = np.argwhere(og == 0)
    smp = np.concatenate([free[rng.integers(0, free.shape[0], n)], rng.integers(0, nh, (n, 1))], axis=1)
    a, _ = _batch(og, start, goal, smp, True, True, 12.0, nh, 3.0, None)
    b, _ = _batch(og, start, goal, smp, True, True, 12.0, nh, 3.0, point)
    for k in ("pts", "head", "parent"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert np.array_equal(a.stats[:, DETERMINISTIC], b.stats[:, DETERMINISTIC])
    assert np.array_equal(a.cost.view(np.int64), b.cost.view(np.int64))
    # host-buffer context: plan2 and the collision test
    ctx = _lib.Context()
    cfg = _lib.plan2_cfg(_lib.MODEL_DUBINS, True, True, 12.0, nh, 3.0, 1.0)
    desc = make_desc2([0], [start], [goal])
    args = dict(samples=smp[None, :, :2].astype(np.int16), heads=smp[None, :, 2].astype(np.uint8))
    nf0 = ctx.set_grids(og[None])
    p0 = ctx.plan2(cfg, desc, n, **args)
    q = np.stack([rng.integers(0, 72, 3000), rng.integers(0, 64, 3000), rng.integers(0, nh, 3000),
                  rng.integers(0, 72, 3000), rng.integers(0, 64, 3000), rng.integers(0, nh, 3000)], axis=1)
    f0 = ctx.dubins_collision(q, nh, 3.0, 0.8)
    runs, lr = body_runs(point)
    nf1 = ctx.set_body_grids(og[None], runs, lr)
    p1 = ctx.plan2(cfg, desc, n, **args)
    f1 = ctx.dubins_collision(q, nh, 3.0, 0.8)
    assert np.array_equal(nf0, nf1) and np.array_equal(f0, f1)
    for x, y in zip(p0[:5], p1[:5]):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert np.array_equal(p0[5][:, DETERMINISTIC], p1[5][:, DETERMINISTIC])
    assert np.array_equal(p0[0][0], b.pts[0]) and np.array_equal(p0[5][0, DETERMINISTIC], b.stats[0, DETERMINISTIC])
    ctx.close()


def test_set_grids_after_a_body_restores_the_point_vehicle():
    rng, og, start, goal = _case(9)
    n, nh = 300, 16
    free = np.argwhere(og == 0)
    smp = np.concatenate([free[rng.integers(0, free.shape[0], n)], rng.integers(0, nh, (n, 1))], axis=1)
    cfg = _lib.plan2_cfg(_lib.MODEL_DUBINS, True, True, 12.0, nh, 3.0, 1.0)
    desc = make_desc2([0], [start], [goal])
    args = dict(samples=smp[None, :, :2].astype(np.int16), heads=smp[None, :, 2].astype(np.uint8))
    fresh = _lib.Context()
    fresh.set_grids(og[None])
    want = fresh.plan2(cfg, desc, n, **args)
    ctx = _lib.Context()
    ctx.set_body_grids(og[None], *body_runs(CAR))
    body = ctx.plan2(cfg, desc, n, **args)
    ctx.set_grids(og[None])
    got = ctx.plan2(cfg, desc, n, **args)
    for x, y in zip(got[:5], want[:5]):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert np.array_equal(got[5][:, DETERMINISTIC], want[5][:, DETERMINISTIC])
    assert not np.array_equal(body[2].view(np.uint8), want[2].view(np.uint8))      # the body did change the plan
    # a Euclidean plan has no heading: refused on a context that holds body layers
    ctx.set_body_grids(og[None], *body_runs(CAR))
    with pytest.raises(ValueError, match="only DUBINS"):
        ctx.plan2(_lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 12.0), make_desc([0], [start[:2]], [goal[:2]]), n, **args)
    fresh.close()
    ctx.close()


def test_dubins_collisionfree_with_a_body_against_a_host_walk():
    rng = np.random.default_rng(17)
    W, H, nh, rho, ds = 80, 70, 16, 5.0, 0.9
    og = (rng.random((W, H)) < 0.01).astype(np.uint8)
    layers = B.layers_scipy(og, CAR)
    L = CAR.shape[0]
    q0 = np.stack([rng.integers(0, W, 300), rng.integers(0, H, 300), rng.integers(0, nh, 300)], axis=1)
    q1 = np.stack([rng.integers(0, W, 300), rng.integers(0, H, 300), rng.integers(0, nh, 300)], axis=1)
    got = dubins_collisionfree(og, q0, q1, rho, nh, ds, body=CAR)
    for i in range(q0.shape[0]):
        P = dubins_points(q0[i], q1[i], rho, nh, ds)
        cx, cy = np.floor(P[:, 0] + 0.5), np.floor(P[:, 1] + 0.5)
        ok = bool(((cx >= 0) & (cx < W) & (cy >= 0) & (cy < H)).all())
        if ok:
            ok = not layers[body_layer(P[:, 2], L), cx.astype(int), cy.astype(int)].any()
            ok = ok and not layers[body_layer(q1[i, 2] * (DM_TWO_PI / nh), L), q1[i, 0], q1[i, 1]]
        assert got[i] == ok, i
    assert 0 < got.sum() < got.size
    # the body never frees what the point vehicle finds blocked
    assert not (got & ~dubins_collisionfree(og, q0, q1, rho, nh, ds)).any()


@pytest.mark.parametrize("cls", ["rrt", "star", "star_norewire"])
def test_device_batch_equals_the_class(cls):
    rng, og, start, goal = _case(33, 96, 80, 0.002)
    n, nh, rho, r = 500, 16, 5.0, 16.0
    for seed in (1, 2, 3):
        if cls == "rrt":
            p = RRTDubins(og, n, rho, nh, pbar=False, seed=seed, body=CAR)
        else:
            p = RRTStarDubins(og, n, r, rho, nh, pbar=False, seed=seed, body=CAR, rewire=cls == "star")
        assert np.array_equal(p.free, np.argwhere(B.projection(B.layers_scipy(og, CAR)) == 0))
        g = np.random.default_rng(seed)
        cells = p.free[g.integers(0, p.free.shape[0], size=n)]
        heads = g.integers(0, nh, size=n)
        T, gv = p.plan(np.array(start), np.array(goal))
        smp = np.concatenate([cells, heads[:, None]], axis=1)
        res, _ = _batch(og, start, goal, smp, cls != "rrt", cls == "star", r if cls != "rrt" else 0.0, nh, rho, CAR)
        st = res.stats[0]
        assert p.last_stats["j"] == st[0] and p.last_stats["found"] == st[2] and p.last_stats["accepted"] == st[4]
        assert st[4] > 20
        j = int(st[0])
        for v in range(1, j):
            (u,) = T.predecessors(v)
            assert u == res.parent[0, v]
            assert T.nodes[v]["heading"] == res.head[0, v]
            assert T.edges[u, v]["dist"] == res.elen[0, v]


def test_set_og_rebuilds_the_layers():
    rng, og, start, goal = _case(41, 96, 80, 0.002)
    p = RRTStarDubins(np.zeros_like(og), 200, 12.0, 4.0, 16, pbar=False, seed=3, body=CAR)
    p.set_og(og)
    assert np.array_equal(p.free, np.argwhere(B.projection(B.layers_scipy(og, CAR)) == 0))
    q = RRTStarDubins(og, 200, 12.0, 4.0, 16, pbar=False, seed=3, body=CAR)
    T1, g1 = p.plan(np.array(start), np.array(goal))
    T2, g2 = q.plan(np.array(start), np.array(goal))
    assert g1 == g2 and p.last_stats == q.last_stats
    assert [T1.nodes[v]["heading"] for v in T1.nodes] == [T2.nodes[v]["heading"] for v in T2.nodes]


# ---- what the body is for ---------------------------------------------------------------------------------------
def test_corridor_is_open_to_the_car_and_closed_to_its_covering_disc():
    W, H, c = 200, 64, 32
    og = np.ones((W, H), np.uint8)
    og[10:190, c - 5: c + 6] = 0                                   # a straight corridor 11 cells wide
    R_cover = math.hypot(8, 2.5)
    ctx = _lib.Context()
    disc = _lib.unpack_grids_host(ctx.inflate_disc(og[None], [0], [_lib.disc_r2(R_cover)]), W, H)[0]
    ctx.close()
    assert disc[10:190, c - 5: c + 6].all()                        # the covering disc fits nowhere
    start, goal = np.array([30, c, 0]), np.array([170, c, 0])
    for cls in (RRTDubins(og, 60, 6.0, 16, pbar=False, seed=4, body=CAR),
                RRTStarDubins(og, 60, 20.0, 6.0, 16, pbar=False, seed=4, body=CAR)):
        T, gv = cls.plan(start, goal)
        assert cls.last_stats["found"] == 1
        assert cls.collisionfree(og, [30, c, 0], [170, c, 0])


def test_full_size_car_never_touches_an_obstacle(torch):
    """The cfg5 shape (1024 worlds of 512 x 512, n = 5000, r = 50, rho = 6, ds = 1, 16 headings) with the car: every pose of every
    tree edge of 64 sampled plans keeps the rectangle turned by its own angle, placed at its rounded cell, off every obstacle
    cell centre."""
    from rrtplanner_b200.batch import seed_states  # noqa: F401  (the batch's own sampler is used below)

    nw, W, H, n, nh = 1024, 512, 512, 5000, 16
    b = DeviceBatch2("dubins", W, H, n, r_rewire=50.0, star=True, rewire=True, nheadings=nh, rho=6.0, ds=1.0)
    b.gen_worlds(np.arange(nw))
    og = b.og
    b.inflate_body(CAR)
    rng = np.random.default_rng(0)
    nfree = b.nfree()
    pick = np.sort(rng.choice(nw, 64, replace=False))
    proj = torch.zeros((nw, W, H), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib().rrtk_unpack_grid(b.bits.data_ptr(), nw, W, H, proj.data_ptr(), torch.cuda.current_stream().cuda_stream))
    starts, goals = [], []
    for w in pick:
        free = torch.nonzero(proj[w] == 0).cpu().numpy()
        assert nfree[w] == free.shape[0] and free.shape[0] > 2
        a, z = free[rng.choice(free.shape[0], 2, replace=False)]
        starts.append([*a, rng.integers(0, nh)])
        goals.append([*z, rng.integers(0, nh)])
    b.set_plans(make_desc2(pick, np.array(starts), np.array(goals))).seed_samples(pick + 1000).seed_heads(pick + 2000).run()
    res = b.download()
    assert res.stat("overflow").max() == 0 and res.stat("found").sum() > 0
    ctx = _lib.Context()
    R_car = math.hypot(8, 2.5)
    k = int(math.ceil(R_car))
    d = torch.arange(-k, k + 1, device="cuda", dtype=torch.float64)
    ox, oy = torch.meshgrid(d, d, indexing="ij")
    ox, oy = ox.reshape(-1), oy.reshape(-1)
    checked = 0
    for p, w in enumerate(pick):
        j = int(res.stat("j")[p]) + int(res.stat("found")[p])
        v = np.arange(1, j)
        if v.size == 0:                                            # the root never grew
            continue
        u = res.parent[p, v]
        q = np.concatenate([res.pts[p, u], res.head[p, u, None], res.pts[p, v], res.head[p, v, None]], axis=1).astype(np.int32)
        _, _, ln = ctx.dubins_paths(q, nh, 6.0)
        cap = int(np.floor(ln.max())) + 1
        xyth, cnt = ctx.dubins_sample(q, nh, 6.0, 1.0, cap)
        mask = np.arange(cap)[None, :] < cnt[:, None]
        P = torch.from_numpy(xyth[mask]).cuda()
        checked += P.shape[0]
        g = og[w].bool()
        for lo in range(0, P.shape[0], 65536):
            Q = P[lo: lo + 65536]
            cx, cy = torch.floor(Q[:, 0] + 0.5), torch.floor(Q[:, 1] + 0.5)
            c, s = torch.cos(Q[:, 2:3]), torch.sin(Q[:, 2:3])
            along, across = c * ox + s * oy, -s * ox + c * oy
            inside = (along > -2 + 1e-6) & (along < 8 - 1e-6) & (across.abs() < 2.5 - 1e-6)
            X, Y = cx[:, None] + ox, cy[:, None] + oy
            ing = (X >= 0) & (X < W) & (Y >= 0) & (Y < H)
            hit = inside & ing & g[X.clamp(0, W - 1).long(), Y.clamp(0, H - 1).long()]
            assert not bool(hit.any()), (p, int(w))
    ctx.close()
    assert checked > 64 * 1000
