"""Weighted sampling on the GPU: rrtk_weight_index + rrtk_sample_streams_weighted against oracle/sampler_oracle.py bit for bit
(samples, generator state and carry) in every regime of integers(0, T), and every entry point that takes weights -- the
planner classes, plan_batch, DeviceBatch / DeviceBatch2 and the pipelined calls -- against each other and against the same
planner fed the oracle's stream."""
import numpy as np
import pytest

from oracle import c_oracle, sampler_oracle as S
from rrtplanner_b200 import RRTDubins, RRTStandard, RRTStar, RRTStarDubins, RRTStarInformed, _lib, batch, worlds
from rrtplanner_b200.body import car_body
from tests.test_gpu_disc import assert_same_graph
from tests.test_weights_host import weights_with_total

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _worlds(seed, nw, W, H, p=0.25):
    rng = np.random.default_rng(seed)
    return (rng.random((nw, W, H)) < p).astype(np.uint8)


def device_streams(torch, ogs, w, n, states, carry=None, worlds_of=None):
    """(samples, state words, carry) of rrtk_sample_streams_weighted; plan p on world worlds_of[p] (default p)."""
    nw, W, H = ogs.shape
    P = states.shape[0]
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    bits = torch.from_numpy(_lib.pack_grids_host(ogs).view(np.int32)).cuda()
    d_w = torch.from_numpy(np.ascontiguousarray(w)).cuda()
    index = torch.empty(int(L.rrtk_weight_index_bytes(nw, W, H)), dtype=torch.uint8, device="cuda")
    _lib.check(L.rrtk_weight_index(bits.data_ptr(), d_w.data_ptr(), nw, W, H, index.data_ptr(), st), "weight_index")
    desc = batch.make_desc(np.arange(P) if worlds_of is None else worlds_of, np.zeros((P, 2)), np.zeros((P, 2)))
    d_desc = torch.from_numpy(desc.view(np.uint8)).cuda()
    d_st = torch.from_numpy(np.ascontiguousarray(states).view(np.int64)).cuda()
    d_cr = None if carry is None else torch.from_numpy(np.ascontiguousarray(carry, dtype=np.uint32).view(np.int32)).cuda()
    out = torch.empty((P, n, 2), dtype=torch.int16, device="cuda")
    _lib.check(L.rrtk_sample_streams_weighted(bits.data_ptr(), d_w.data_ptr(), index.data_ptr(), nw, W, H, d_desc.data_ptr(), P,
                                              d_st.data_ptr(), None if d_cr is None else d_cr.data_ptr(), n, out.data_ptr(), st),
               "sample_streams_weighted")
    tot = index[: 8 * nw].view(torch.int64).cpu().numpy()
    return (out.cpu().numpy().astype(np.int64), d_st.cpu().numpy().view(np.uint64),
            None if d_cr is None else d_cr.cpu().numpy().view(np.uint32), tot)


def maps(kind, og, rng):
    W, H = og.shape
    if kind == "ones":
        return np.ones((W, H), np.uint8)
    if kind == "random":
        return rng.integers(0, 256, size=(W, H)).astype(np.uint8)
    if kind == "single":                              # T = 1
        w = np.zeros((W, H), np.uint8)
        free = np.argwhere(og == 0)
        w[tuple(free[len(free) // 2])] = 1
        return w
    w = rng.integers(0, 256, size=(W, H)).astype(np.uint8)       # heavy weight on occupied cells, masked away
    w[og != 0] = 255
    w[(og == 0) & (rng.random((W, H)) < 0.7)] = 0
    return w


SHAPES = [(64, 64), (37, 45), (1, 70), (3001, 45), (45, 3001)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
@pytest.mark.parametrize("kind", ["ones", "random", "single", "occupied"])
@pytest.mark.parametrize("n", [1000, 20000])              # parallel kernel / sequential kernel (raw window exceeds shared memory)
def test_kernel_against_the_oracle(torch, shape, kind, n):
    W, H = shape
    rng = np.random.default_rng(W * 7 + H + n)
    ogs = _worlds(W + H, 3, W, H)
    w = np.stack([maps(kind, og, rng) for og in ogs])
    seeds = np.array([3, 17, 40001])
    states = batch.seed_states(seeds)
    # a carried generator: plan p's generator after a few draws that leave a buffered 32-bit half
    gens = [np.random.default_rng(int(s) + 1) for s in seeds]
    for g in gens:
        g.integers(0, 1000, size=3)
    cw = [S.generator_words(g) for g in gens]
    cstates, carry = np.stack([c[0] for c in cw]), np.stack([c[1] for c in cw])
    got, _, _, tot = device_streams(torch, ogs, w, n, states)
    got_c, st_c, cr_c, _ = device_streams(torch, ogs, w, n, cstates.copy(), carry.copy())
    for p in range(3):
        e = S.effective_weights(w[p], ogs[p] == 0)
        assert tot[p] == e.sum()
        want, _, _ = S.weighted_stream(w[p], ogs[p] == 0, n, seed=int(seeds[p]))
        assert np.array_equal(got[p], want), p
        want_c, ws, wc = S.weighted_stream(w[p], ogs[p] == 0, n, state=cstates[p], carry=carry[p])
        assert np.array_equal(got_c[p], want_c) and np.array_equal(st_c[p], ws) and np.array_equal(cr_c[p], wc), p
    if kind == "ones":                                   # byte for byte the uniform sampler's stream
        db = batch.DeviceBatch("standard", W, H, n).set_worlds_host(ogs)
        db.set_plans(batch.make_desc(np.arange(3), np.zeros((3, 2)), np.zeros((3, 2)))).seed_samples(seeds)
        assert np.array_equal(db.samples.cpu().numpy().astype(np.int64), got)


@pytest.mark.parametrize("total", [2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1])
def test_totals_around_two_to_the_32(torch, total):
    W, H = 4160, 4096
    w = weights_with_total((W, H), total)[None]
    og = np.zeros((1, W, H), np.uint8)
    gen = np.random.default_rng(99)
    gen.integers(0, 5, size=1)
    words, carry = S.generator_words(gen)
    for n in (3000, 20000):
        got, st, cr, tot = device_streams(torch, og, w, n, words[None].copy(), carry[None].copy())
        assert tot[0] == total
        want, ws, wc = S.weighted_stream(w[0], og[0] == 0, n, state=words, carry=carry)
        assert np.array_equal(got[0], want) and np.array_equal(st[0], ws) and np.array_equal(cr[0], wc)


def test_16384_squared_all_255(torch):
    S2 = 16384
    og = np.zeros((1, S2, S2), np.uint8)
    w = np.full((1, S2, S2), 255, np.uint8)
    n = 5000
    got, st, _, tot = device_streams(torch, og, w, n, batch.seed_states([7]))
    T = 255 * S2 * S2
    assert tot[0] == T
    rng = np.random.default_rng(7)
    k = rng.integers(0, T, size=n) // 255                 # searchsorted on cum = 255 (i + 1)
    assert np.array_equal(got[0], np.stack(np.divmod(k, S2), axis=1))


# ---- planner classes against the same class fed the oracle's stream --------------------------------------------------------
class _Oracle:
    """sample_all_free overridden by the specification: one weighted draw per call from the planner's generator."""

    def sample_all_free(self):
        e = S.effective_weights(self._w, self._mask)
        cum = np.cumsum(e.ravel())
        k = int(np.searchsorted(cum, self.rand_gen.integers(0, int(cum[-1])), side="right"))
        return np.array(divmod(k, e.shape[1]))


def _oracle_class(base, w, mask):
    return type("Oracle" + base.__name__, (_Oracle, base), {"_w": w, "_mask": mask})


def _case(seed, W=64, H=56):
    og = _worlds(seed, 1, W, H, 0.12)[0]
    w = maps("random", og, np.random.default_rng(seed))
    free = np.argwhere(og == 0)
    rng = np.random.default_rng(seed + 1)
    return og, w, free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]


def _cspace(og, radius):
    return _lib.unpack_grids_host(_lib.shared_context().inflate_disc(og[None], [0], [_lib.disc_r2(radius)]), *og.shape)[0]


EUCLID = {
    "standard": lambda cls, og, **k: cls(og, 500, pbar=False, seed=4, **k),
    "star": lambda cls, og, **k: cls(og, 500, 12.0, pbar=False, seed=4, **k),
    "star_rrtstar": lambda cls, og, **k: cls(og, 500, 12.0, pbar=False, seed=4, rewire="rrtstar", **k),
    "informed": lambda cls, og, **k: cls(og, 500, 12.0, 6.0, pbar=False, seed=4, **k),
    "informed_rrtstar": lambda cls, og, **k: cls(og, 500, 12.0, 6.0, pbar=False, seed=4, rewire="rrtstar", **k),
}
BASES = {"standard": RRTStandard, "star": RRTStar, "star_rrtstar": RRTStar, "informed": RRTStarInformed, "informed_rrtstar": RRTStarInformed}


@pytest.mark.parametrize("radius", [None, 2.5])
@pytest.mark.parametrize("name", list(EUCLID))
def test_classes_equal_the_oracle_sampler(name, radius):
    og, w, a, b = _case(5)
    mask = (og if radius is None else _cspace(og, radius)) == 0
    free = np.argwhere(mask)
    a, b = free[3], free[-5]
    make, base = EUCLID[name], BASES[name]
    got = make(base, og, robot_radius=radius, sample_weights=w)
    want = make(_oracle_class(base, w, mask), og, robot_radius=radius)
    assert_same_graph(got.plan(a, b), want.plan(a, b))
    assert_same_graph(got.plan(b, a), want.plan(b, a))                   # the generators carry on identically


class _DubinsOracle:
    """the stock Dubins stream (n cells, then n headings) with the cells from the specification"""

    def _draw_configs(self, count):
        e = S.effective_weights(self._w, self._mask)
        cum = np.cumsum(e.ravel())
        k = np.searchsorted(cum, self.rand_gen.integers(0, int(cum[-1]), size=count), side="right")
        cells = np.stack(np.divmod(k, e.shape[1]), axis=1)
        return cells, self.rand_gen.integers(0, self.nheadings, size=count)


@pytest.mark.parametrize("body", [False, True])
@pytest.mark.parametrize("star", [False, True])
def test_dubins_classes_equal_the_oracle_sampler(star, body):
    og, w, _, _ = _case(8, 72, 64)
    og[:] = 0
    og[30:34, 10:50] = 1
    stencils = car_body(4, 1, 1.5, 8) if body else None
    probe = RRTDubins(og, 10, 3.0, 8, pbar=False, body=stencils)
    mask = np.zeros(og.shape, bool)
    mask[tuple(probe.free.T)] = True
    a, b = probe.free[0], probe.free[-1]
    base = RRTStarDubins if star else RRTDubins
    args = (og, 300, 10.0, 3.0, 8) if star else (og, 300, 3.0, 8)
    cls = type("OracleDubins", (_DubinsOracle, base), {"_w": w, "_mask": mask})
    got = base(*args, pbar=False, seed=2, body=stencils, sample_weights=w)
    want = cls(*args, pbar=False, seed=2, body=stencils)
    qa, qb = [a[0], a[1], 0], [b[0], b[1], 4]
    assert_same_graph(got.plan(qa, qb), want.plan(qa, qb))


# ---- batch entry points -------------------------------------------------------------------------------------------------
def _batch_case(seed=11, nw=3, W=48, H=40, P=10):
    ogs = _worlds(seed, nw, W, H, 0.15)
    rng = np.random.default_rng(seed)
    w = np.stack([maps("random", og, rng) for og in ogs])
    wid = np.sort(rng.integers(0, nw, P))
    starts, goals = np.zeros((P, 2), int), np.zeros((P, 2), int)
    for p in range(P):
        free = np.argwhere(_cspace(ogs[wid[p]], 2.0) == 0)
        starts[p], goals[p] = free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]
    return ogs, w, wid, starts, goals, 100 + np.arange(P)


# j, vgoal, found: the statistics that describe the tree (the check / cell counters of the parallel kernel form are diagnostics)
TREE_STATS = slice(0, 3)


def _same_batch(a, b):
    assert np.array_equal(a.stats[:, TREE_STATS], b.stats[:, TREE_STATS]) and np.array_equal(a.pts, b.pts) and np.array_equal(a.parent, b.parent)
    assert np.array_equal(np.asarray(a.cost).view(np.int64), np.asarray(b.cost).view(np.int64))


@pytest.mark.parametrize("kind", ["standard", "star"])
@pytest.mark.parametrize("radius", [None, 0.0, 2.0, "mixed"])
def test_plan_batch_equals_the_classes(kind, radius):
    ogs, w, wid, starts, goals, seeds = _batch_case()
    n = 300
    rr = np.where(np.arange(len(wid)) % 2, 2.0, 1.0) if radius == "mixed" else radius
    res = batch.plan_batch(kind, ogs, n, starts, goals, world_ids=wid, r_rewire=10.0, seeds=seeds, robot_radius=rr, sample_weights=w)
    for p in range(len(wid)):
        rp = None if rr is None else float(np.broadcast_to(rr, len(wid))[p])
        cls = RRTStandard(ogs[wid[p]], n, pbar=False, seed=int(seeds[p]), robot_radius=rp, sample_weights=w[wid[p]]) if kind == "standard" \
            else RRTStar(ogs[wid[p]], n, 10.0, pbar=False, seed=int(seeds[p]), robot_radius=rp, sample_weights=w[wid[p]])
        T, gv = cls.plan(starts[p], goals[p])
        assert int(res.stat("vgoal")[p]) == int(gv) or not res.stat("found")[p]
        j = int(res.stat("j")[p]) + int(res.stat("found")[p])
        pts = np.stack([np.asarray(T.nodes[v]["pt"]) for v in range(j)])
        assert np.array_equal(res.pts[p, :j].astype(np.int64), pts), p
    if radius is None:                                  # all-ones weights: the uniform batch, tree for tree
        ones = batch.plan_batch(kind, ogs, n, starts, goals, world_ids=wid, r_rewire=10.0, seeds=seeds, sample_weights=np.ones_like(w[0]))
        _same_batch(ones, batch.plan_batch(kind, ogs, n, starts, goals, world_ids=wid, r_rewire=10.0, seeds=seeds))


@pytest.mark.parametrize("inflate", [False, True])
def test_device_batches_and_pipelined_calls_equal_plan_batch(torch, inflate):
    ogs, w, wid, starts, goals, seeds = _batch_case(P=24)
    n, W, H = 300, ogs.shape[1], ogs.shape[2]
    radius = 2.0 if inflate else None
    want = batch.plan_batch("star", ogs, n, starts, goals, world_ids=wid, r_rewire=10.0, seeds=seeds, robot_radius=radius, sample_weights=w)
    desc = batch.make_desc(wid, starts, goals)
    db = batch.DeviceBatch("star", W, H, n, 10.0).set_worlds_host(ogs)
    if inflate:
        db.inflate_disc(radius)
    db.set_sample_weights(torch.from_numpy(w).cuda()).set_plans(desc).seed_samples(seeds)
    _same_batch(db.run().download(), want)
    # DeviceBatch2 (Euclid, no rewire) draws the same cell stream and computes the same RRT* trees
    db2 = batch.DeviceBatch2("euclid", W, H, n, 10.0, star=True, rewire=False).set_worlds_host(ogs)
    if inflate:
        db2.inflate_disc(radius)
    db2.set_sample_weights(w).set_plans(desc).seed_samples(seeds)
    assert np.array_equal(db2.samples.cpu().numpy(), db.samples.cpu().numpy())
    r2 = db2.run().download()
    assert np.array_equal(r2.pts, want.pts) and np.array_equal(r2.parent, want.parent)
    # the pipelined calls on the same grids, several chunk sizes
    grids = _lib.unpack_grids_host(db.bits.cpu().numpy().view(np.uint32), W, H)
    ctx = _lib.Context()
    states = batch.seed_states(seeds)
    for chunk in (0, 1, 5, 24):
        o = ctx.plan_worlds2(_lib.KIND_STAR, grids, W, H, desc, n, 10.0, states=states, trees=True, paths=True, chunk=chunk, sample_weights=w)
        assert np.array_equal(o["pts"], want.pts) and np.array_equal(o["stats"][:, TREE_STATS], want.stats[:, TREE_STATS]), chunk
        cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, False, 10.0)
        o2 = ctx.plan2_worlds(cfg, grids, W, H, desc, n, states=states, trees=True, chunk=chunk, sample_weights=True)
        assert np.array_equal(o2["pts"], want.pts) and np.array_equal(o2["parent"], want.parent), chunk
    # all-ones weights through the pipelined call and DeviceBatch: the uniform results, bit for bit
    ones = np.ones_like(w)
    u = ctx.plan_worlds2(_lib.KIND_STAR, grids, W, H, desc, n, 10.0, states=states, trees=True, paths=True)
    o = ctx.plan_worlds2(_lib.KIND_STAR, grids, W, H, desc, n, 10.0, states=states, trees=True, paths=True, sample_weights=ones)
    u["stats"], o["stats"] = u["stats"][:, TREE_STATS], o["stats"][:, TREE_STATS]
    for k in u:
        assert np.array_equal(np.asarray(u[k]).view(np.uint8), np.asarray(o[k]).view(np.uint8)), k
    # weights in a view that starts at an odd byte offset (H % 4 == 0): the index reads them cell by cell, same streams
    buf = torch.zeros(1 + w.size, dtype=torch.uint8, device="cuda")
    buf[1:] = torch.from_numpy(w.reshape(-1)).cuda()
    db.set_sample_weights(w).seed_samples(seeds)
    s0 = db.samples.clone()
    db.set_sample_weights(buf[1:].view(w.shape)).seed_samples(seeds)
    assert db.weights.data_ptr() % 2 == 1 and bool((db.samples == s0).all())
    db.set_sample_weights(ones).seed_samples(seeds)
    s1 = db.samples.clone()
    db.set_sample_weights(None).seed_samples(seeds)
    assert bool((db.samples == s1).all())
    ctx.close()


def test_errors(torch):
    ogs, w, wid, starts, goals, seeds = _batch_case()
    n, W, H = 50, ogs.shape[1], ogs.shape[2]
    zw = int(wid[len(wid) // 2])
    zero = w.copy()
    zero[zw][ogs[zw] == 0] = 0                            # weight on occupied cells only: nothing to draw
    with pytest.raises(ValueError, match="world %d" % zw):
        batch.plan_batch("standard", ogs, n, starts, goals, world_ids=wid, seeds=seeds, sample_weights=zero)
    # the error names the caller's plan and world, also with unsorted worlds and per-plan radii (grids of (world, r2) pairs)
    perm = np.random.default_rng(3).permutation(len(wid))
    radii = np.where(np.arange(len(wid)) % 2, 2.0, 1.0)
    with pytest.raises(ValueError, match=r"world %d at robot_radius" % zw) as err:
        batch.plan_batch("standard", ogs, n, starts[perm], goals[perm], world_ids=wid[perm], seeds=seeds, robot_radius=radii,
                         sample_weights=zero)
    assert wid[perm][int(str(err.value).split(":")[0].split()[1])] == zw
    desc = batch.make_desc(wid, starts, goals)
    db = batch.DeviceBatch("standard", W, H, n).set_worlds_host(ogs).set_sample_weights(zero).set_plans(desc)
    with pytest.raises(ValueError, match="world %d" % zw):
        db.seed_samples(seeds)
    with pytest.raises(ValueError):
        db.set_sample_weights(w[:, :-1])
    with pytest.raises(TypeError):
        db.set_sample_weights(torch.ones((3, W, H), dtype=torch.float32))
    ctx = _lib.Context()
    states = batch.seed_states(seeds)
    with pytest.raises(ValueError, match="without weights"):
        ctx.plan_worlds2(_lib.KIND_STANDARD, ogs, W, H, desc, n, states=states, sample_weights=True)
    ctx.set_sample_weights(w[:2])
    with pytest.raises(ValueError, match="maps of"):
        ctx.plan_worlds2(_lib.KIND_STANDARD, ogs, W, H, desc, n, states=states, sample_weights=True)
    with pytest.raises(ValueError, match="seed mode"):
        ctx.plan_worlds2(_lib.KIND_STANDARD, ogs[:2], W, H, desc[:2], n, samples=np.zeros((2, n, 2)), sample_weights=True)
    with pytest.raises(ValueError):
        batch.plan_batch("informed", ogs, n, starts, goals, world_ids=wid, r_rewire=5.0, r_goal=3.0, seeds=seeds, balls="seed",
                         sample_weights=w)
    inf = batch.DeviceBatch("informed", W, H, n, 5.0, 3.0).set_worlds_host(ogs).set_sample_weights(w)
    inf.set_plans(batch.make_desc(wid, starts, goals, batch.informed_rotations(starts, goals)))
    with pytest.raises(ValueError, match="weighted informed"):
        inf.seed_informed(states)
    ctx.close()


def test_cfg3_size_run():
    """4096 plans of n = 5000 on 512 x 512 worlds with a corridor heatmap: 64 streams against the oracle, every sample on a cell of
    non-zero effective weight, 16 trees against the C oracle on the same streams."""
    W = H = 512
    n, P = 5000, 4096
    db = batch.DeviceBatch("star", W, H, n, 50.0).gen_worlds([worlds.world_seed(p) for p in range(P)])
    ogs = db.og.cpu().numpy()
    rng = np.random.default_rng(0)
    starts, goals = np.zeros((P, 2), int), np.zeros((P, 2), int)
    for p in range(P):
        free = np.argwhere(ogs[p] == 0)
        starts[p], goals[p] = free[rng.integers(0, len(free))], free[rng.integers(0, len(free))]
    w = corridor_maps(starts, goals, W, H)
    db.set_sample_weights(w).set_plans(batch.make_desc(np.arange(P), starts, goals)).seed_samples(np.arange(P))
    res = db.run().download()
    smp = db.samples.cpu().numpy().astype(np.int64)
    for p in range(P):
        assert (w[p][smp[p, :, 0], smp[p, :, 1]] > 0).all() and (ogs[p][smp[p, :, 0], smp[p, :, 1]] == 0).all()
    for p in range(0, P, 64):
        assert np.array_equal(smp[p], S.weighted_stream(w[p], ogs[p] == 0, n, seed=p)[0]), p
    for p in range(0, P, 256):
        wp, _, wpar, st, _ = c_oracle.plan_raw("star", ogs[p], n, starts[p], goals[p], smp[p], 50.0)
        t = st["j"] + (1 if st["found"] else 0)
        assert int(res.stat("j")[p]) == st["j"] and np.array_equal(res.pts[p, :t], wp[:t]) and np.array_equal(res.parent[p, :t], wpar[:t])


def corridor_maps(starts, goals, W, H, width=24.0, hi=255, lo=4):
    """A stand-in for a learned heatmap: ``hi`` within ``width`` cells of each plan's start-goal segment, ``lo`` elsewhere."""
    x, y = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64), indexing="ij")
    out = np.empty((len(starts), W, H), np.uint8)
    for p, (a, b) in enumerate(zip(np.asarray(starts, float), np.asarray(goals, float))):
        d = b - a
        L2 = max(float(d @ d), 1e-12)
        t = np.clip(((x - a[0]) * d[0] + (y - a[1]) * d[1]) / L2, 0.0, 1.0)
        dist2 = (x - a[0] - t * d[0]) ** 2 + (y - a[1] - t * d[1]) ** 2
        out[p] = np.where(dist2 <= width * width, hi, lo)
    return out
