"""GPU parity tests: the CUDA path, called through the C ABI (ctypes -> librrtk.so), against the
pinned oracle and the golden vectors produced by the real reference.  Bit-exact everywhere (integer
/ index work and FP64 costs alike); the only tolerance in this file is the 1e-5 relative bound on
path cost that BASELINE.json's north star states, checked in addition to bit equality."""
import glob
import os

import numpy as np
import pytest

from oracle import c_oracle, rrt_oracle as O
from rrtplanner_b200 import _lib, batch, worlds
from tests.conftest import GOLDEN, load_plan

pytestmark = pytest.mark.gpu

KIND = {"standard": 0, "star": 1, "informed": 2}


@pytest.fixture(scope="module")
def ctx():
    c = _lib.Context()
    yield c
    c.close()


def tiled_bits(og):
    """numpy statement of the tiled bit layout documented in include/rrtk.h"""
    W, H = og.shape
    TX, TY = (W + 31) // 32, (H + 31) // 32
    pad = np.ones((TX * 32, TY * 32), dtype=np.uint64)
    pad[:W, :H] = og != 0
    t = pad.reshape(TX, 32, TY, 32).transpose(0, 2, 1, 3)            # tx, ty, x&31, y&31
    words = (t << np.arange(32, dtype=np.uint64)).sum(axis=3)
    return words.reshape(-1).astype(np.uint32)


# ---- K0 / free-space index / world generator ---------------------------------------------------
@pytest.mark.parametrize("shape", [(64, 64), (43, 100), (100, 43), (33, 31), (1, 1), (256, 512)])
def test_pack_and_free_rows(shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    ogs = (rng.random((3,) + shape) < 0.3).astype(np.uint8)
    db = batch.DeviceBatch("star", shape[0], shape[1], 16).set_worlds_host(ogs)
    bits = db.bits.cpu().numpy().view(np.uint32)
    rowcum = db.rowcum.cpu().numpy()
    for w in range(3):
        assert np.array_equal(bits[w], tiled_bits(ogs[w]))
        want = np.concatenate([[0], np.cumsum((ogs[w] == 0).sum(axis=1))])
        assert np.array_equal(rowcum[w], want)


@pytest.mark.parametrize("dtype", [int, float, np.uint32, np.uint64, np.int32, np.int64, np.float32, np.float64])
def test_any_dtype_grid_means_nonzero_is_obstacle(ctx, dtype):
    # the reference's fixture grid: tests/test_rrt.py:8-17,31-36
    og = np.zeros((43, 100), dtype=dtype)
    og[43 // 4: 3 * 43 // 4, 100 // 4: 3 * 100 // 4] = 1
    og[5, 5] = 3 if np.issubdtype(np.dtype(dtype), np.integer) else 0.25
    ctx.set_grids((og != 0).astype(np.uint8)[None])
    rng = np.random.default_rng(1)
    segs = np.stack([rng.integers(0, 43, 500), rng.integers(0, 100, 500), rng.integers(0, 43, 500), rng.integers(0, 100, 500)], 1)
    got = ctx.collision(segs)
    want = np.array([O.collisionfree(og, s[:2], s[2:]) for s in segs])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("shape,seed", [((64, 48), 3), ((256, 256), 1000), ((512, 512), 1001), ((130, 70), 77)])
def test_world_generator_bit_identical_to_numpy(shape, seed):
    db = batch.DeviceBatch("star", shape[0], shape[1], 16).gen_worlds([seed, seed + 1])
    og = db.og.cpu().numpy()
    for k in range(2):
        assert np.array_equal(og[k], worlds.perlin_occupancygrid(shape[0], shape[1], seed=seed + k).astype(np.uint8))


# ---- K1 -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "collision_*.npz"))), ids=lambda p: os.path.basename(p)[10:-4])
def test_collision_golden(ctx, path):
    z = np.load(path)
    og, segs, want = z["og"], z["segs"].astype(np.int32), z["free"]
    ctx.set_grids((og != 0).astype(np.uint8)[None])
    free, cells = ctx.collision(segs, cells=True)
    assert np.array_equal(free, want)                       # verdicts of the unmodified reference
    _, want_cells = c_oracle.collision_batch(og, segs)
    assert np.array_equal(cells, want_cells)                # and the same first-hit position


@pytest.mark.parametrize("size,nseg", [(2048, 200_000), (1024, 100_000), (512, 100_000), (97, 20_000)])
def test_collision_random_vs_oracle(ctx, size, nseg):
    og = worlds.perlin_occupancygrid(size, size, seed=9).astype(np.uint8)
    ctx.set_grids(og[None])
    rng = np.random.default_rng(0)
    segs = rng.integers(0, size, size=(nseg, 4)).astype(np.int32)      # cfg2's segment distribution
    segs[:64, 2:] = segs[:64, :2]                                       # degenerate a == b
    segs[64:128, 2] = segs[64:128, 0]                                   # vertical / horizontal
    segs[128:192, 3] = segs[128:192, 1]
    free, cells = ctx.collision(segs, cells=True)
    want_free, want_cells = c_oracle.collision_batch(og, segs)
    assert np.array_equal(free, want_free)
    assert np.array_equal(cells, want_cells)
    # direction matters in the reference (SURVEY 3.4): reversed segments are their own cases
    rev = segs[:20000, [2, 3, 0, 1]].copy()
    assert np.array_equal(ctx.collision(rev), c_oracle.collision_batch(og, rev)[0])


def test_collision_rejects_points_outside_grid(ctx):
    ctx.set_grids(np.zeros((1, 20, 20), dtype=np.uint8))
    with pytest.raises(ValueError):
        ctx.collision(np.array([[0, 0, 20, 3]]))


def test_collision_multi_world_device_api():
    import torch
    ogs = np.stack([worlds.perlin_occupancygrid(128, 96, seed=s) for s in range(5)]).astype(np.uint8)
    db = batch.DeviceBatch("star", 128, 96, 16).set_worlds_host(ogs)
    rng = np.random.default_rng(4)
    nseg = 30000
    segs = np.stack([rng.integers(0, 128, nseg), rng.integers(0, 96, nseg), rng.integers(0, 128, nseg), rng.integers(0, 96, nseg)], 1).astype(np.int32)
    wid = rng.integers(0, 5, nseg).astype(np.int32)
    d_segs, d_w = torch.from_numpy(segs).cuda(), torch.from_numpy(wid).cuda()
    d_free = torch.empty(nseg, dtype=torch.uint8, device="cuda")
    d_cells = torch.empty(nseg, dtype=torch.int32, device="cuda")
    _lib.check(db.L.rrtk_collision_segments(db.bits.data_ptr(), 128, 96, d_segs.data_ptr(), d_w.data_ptr(), nseg,
                                            d_free.data_ptr(), d_cells.data_ptr(), torch.cuda.current_stream().cuda_stream))
    free, cells = d_free.cpu().numpy().astype(bool), d_cells.cpu().numpy()
    for w in range(5):
        m = wid == w
        wf, wc = c_oracle.collision_batch(ogs[w], segs[m])
        assert np.array_equal(free[m], wf) and np.array_equal(cells[m], wc)


# ---- K2 / K3 ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["lattice", "sparse"])
def test_queries_golden(ctx, tag):
    z = np.load(os.path.join(GOLDEN, "queries.npz"))
    pts, qs, radii = z[f"{tag}_pts"], z[f"{tag}_qs"], z[f"{tag}_radii"]
    flat, lens, d2 = z[f"{tag}_within_flat"], z[f"{tag}_within_len"], z[f"{tag}_near0_d2"]
    idx, key = ctx.nearest(pts, qs)
    assert np.array_equal(key, d2)                                        # same minimum as the unmodified reference
    for q, v, k in zip(qs, idx, key):
        assert v == int(np.flatnonzero(((pts - q) ** 2).sum(1) == k)[0])   # pinned: lowest index
    off = 0
    for q, r, m in zip(qs, radii, lens):
        out, ln = ctx.within(pts, q[None], r)
        assert ln[0] == m and np.array_equal(out[0, :m], flat[off:off + m])
        off += m


def test_within_reference_kat_float_query(ctx):
    # tests/test_rrt.py:116-119 -- the reference's only known-answer vector
    pts = np.array([[0, 0], [1, 0], [1, 1], [0, 1]])
    out, ln = ctx.within(pts, np.array([[0.5, 0.5]]), 1.0)
    assert ln[0] == 4 and out[0, :4].tolist() == [0, 1, 2, 3]
    import rrtplanner_b200 as R
    assert R.RRT.within(pts, np.array([0.5, 0.5]), 1.0).shape[0] == 4


def test_near_full_order_is_stable_argsort(ctx):
    rng = np.random.default_rng(5)
    for m in (1, 7, 1000, 5000):
        pts = rng.integers(0, 60, size=(m, 2)).astype(np.int64)
        x = rng.integers(0, 60, size=2)
        assert np.array_equal(ctx.near_order(pts, x), O.near_sorted(pts, x, stable=True))
    ptsf = rng.random((777, 2)) * 50
    xf = rng.random(2) * 50
    assert np.array_equal(ctx.near_order(ptsf, xf), O.near_sorted(ptsf, xf, stable=True))


def test_nearest_prefix_counts_device_api():
    import torch
    rng = np.random.default_rng(6)
    pts = rng.integers(0, 512, size=(5000, 2)).astype(np.int32)
    qs = rng.integers(0, 512, size=(300, 2)).astype(np.int32)
    cnt = rng.integers(1, 5001, size=300).astype(np.int32)
    L = _lib.lib()
    d = [torch.from_numpy(a).cuda() for a in (pts, qs, cnt)]
    idx = torch.empty(300, dtype=torch.int32, device="cuda")
    d2 = torch.empty(300, dtype=torch.int64, device="cuda")
    _lib.check(L.rrtk_nearest_batch(d[0].data_ptr(), 5000, d[1].data_ptr(), d[2].data_ptr(), 300, idx.data_ptr(), d2.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream))
    out = torch.empty((300, 64), dtype=torch.int32, device="cuda")
    ln = torch.empty(300, dtype=torch.int32, device="cuda")
    _lib.check(L.rrtk_within_batch(d[0].data_ptr(), 5000, d[1].data_ptr(), d[2].data_ptr(), 300, 50.0, 64, out.data_ptr(), ln.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    idx, d2, out, ln = idx.cpu().numpy(), d2.cpu().numpy(), out.cpu().numpy(), ln.cpu().numpy()
    for q in range(300):
        v, dd = c_oracle.nearest(pts, int(cnt[q]), qs[q])
        assert (idx[q], d2[q]) == (v, dd)
        w = c_oracle.within(pts, int(cnt[q]), qs[q], 50.0)
        assert ln[q] == len(w) and np.array_equal(out[q, :min(64, len(w))], w[:64])


# ---- sampler -----------------------------------------------------------------------------------------
def test_sample_stream_matches_numpy_pcg64(ctx):
    og = worlds.perlin_occupancygrid(200, 150, seed=21).astype(np.uint8)
    ctx.set_grids(np.stack([og, 1 - og]))
    seeds = [0, 1, 12345, 2 ** 31 - 1, 987654321]
    desc = batch.make_desc([0, 1, 0, 1, 0], np.zeros((5, 2)), np.zeros((5, 2)))
    got = ctx.samples(desc, 4000, batch.seed_states(seeds))
    for p, s in enumerate(seeds):
        g = og if p % 2 == 0 else 1 - og
        assert np.array_equal(got[p].astype(np.int64), O.sample_stream(g, 4000, s))


def test_sample_stream_matches_reference_sampler(ctx):
    z = np.load(os.path.join(GOLDEN, "sampler_seed12345.npz"))      # drawn by the reference's RRT.sample_all_free
    ctx.set_grids((z["og"] != 0).astype(np.uint8)[None])
    got = ctx.samples(batch.make_desc([0], [[0, 0]], [[0, 0]]), 300, batch.seed_states([12345]))
    assert np.array_equal(got[0], z["drawn"])


def test_sampler_rejection_path(ctx):
    """A free-cell count just above 2^31 / k makes Lemire's rejection loop fire often enough to
    be exercised; tiny worlds (nfree = 3) stress the threshold arithmetic."""
    og = np.ones((40, 40), dtype=np.uint8)
    og[3, 7] = og[20, 0] = og[39, 39] = 0
    ctx.set_grids(og[None])
    got = ctx.samples(batch.make_desc([0], [[3, 7]], [[3, 7]]), 6000, batch.seed_states([5]))
    assert np.array_equal(got[0].astype(np.int64), O.sample_stream(og, 6000, 5))


def test_sample_stream_large_n_takes_the_sequential_kernel(ctx):
    """Above ~29 000 draws the raw window of the parallel generator no longer fits shared memory and the launcher falls back to
    the one-thread generator; both must give numpy's stream."""
    og = worlds.perlin_occupancygrid(96, 80, seed=3).astype(np.uint8)
    ctx.set_grids(og[None])
    for n in (28000, 40000):
        got = ctx.samples(batch.make_desc([0], [[0, 0]], [[0, 0]]), n, batch.seed_states([77]))
        assert np.array_equal(got[0].astype(np.int64), O.sample_stream(og, n, 77))


def test_sampler_with_many_rejections(ctx):
    """nfree = 3700^2: 2^32 mod nfree is large, so one draw in ~430 is rejected -- ~19 rejections at n = 8000 (handled by
    the parallel compaction) and ~65 at n = 28000 (around the slack of the raw window, so some seeds take the sequential
    fallback).  Both must reproduce numpy's stream, including the generator state that is carried on."""
    import torch
    S = 3700
    og = np.zeros((S, S), dtype=np.uint8)
    ctx.set_grids(og[None])
    seeds = np.arange(70, 78)
    thr = (1 << 32) % (S * S)
    for n in (8000, 28000):
        got = ctx.samples(batch.make_desc(np.zeros(len(seeds), int), np.zeros((len(seeds), 2)), np.zeros((len(seeds), 2))), n,
                          batch.seed_states(seeds))
        nrej = []
        for p, sd in enumerate(seeds):
            idx = np.random.default_rng(int(sd)).integers(0, S * S, size=n)
            assert np.array_equal(got[p].astype(np.int64), np.stack([idx // S, idx % S], axis=1)), (n, sd)
            raw = np.random.default_rng(int(sd)).integers(0, 1 << 32, size=n + 200, dtype=np.uint64)   # raw 32-bit stream
            nrej.append(int((((raw * np.uint64(S * S)) & np.uint64(0xffffffff)) < thr)[:n].sum()))
        assert max(nrej) > 5
        if n == 28000:
            assert min(nrej) <= 62 < max(nrej)                          # both the compaction and the fallback are exercised
    # carried generator state across two calls of odd length
    db = batch.DeviceBatch("standard", S, S, 4001).set_worlds_host(og[None])
    A = len(seeds)
    db.set_plans(batch.make_desc(np.zeros(A, int), np.zeros((A, 2)), np.zeros((A, 2))))
    state = torch.from_numpy(batch.seed_states(seeds).view(np.int64)).cuda()
    carry = torch.zeros((A, 2), dtype=torch.int32, device="cuda")
    smp = torch.empty((A, 4001, 2), dtype=torch.int16, device="cuda")
    gens = [np.random.default_rng(int(sd)) for sd in seeds]
    for call in range(3):
        _lib.check(db.L.rrtk_sample_streams_carry(db.bits.data_ptr(), db.rowcum.data_ptr(), S, S, db.desc.data_ptr(), A, state.data_ptr(),
                                                  carry.data_ptr(), 4001, smp.data_ptr(), torch.cuda.current_stream().cuda_stream), "carry")
        got = smp.cpu().numpy().astype(np.int64)
        for a in range(A):
            idx = gens[a].integers(0, S * S, size=4001)
            assert np.array_equal(got[a], np.stack([idx // S, idx % S], axis=1)), (call, a)
        for a in range(A):                                                # generator state equals numpy's
            stt = gens[a].bit_generator.state
            want = [stt["state"]["state"] >> 64, stt["state"]["state"] & ((1 << 64) - 1)]
            have = [int(v) & ((1 << 64) - 1) for v in state[a, :2].cpu().numpy()]
            assert have == want and int(carry[a, 0]) == stt["has_uint32"]
            if stt["has_uint32"]:
                assert (int(carry[a, 1]) & 0xffffffff) == stt["uinteger"]


# ---- K7: whole plans ----------------------------------------------------------------------------------
def run_golden(ctx, g):
    ctx.set_grids(g["og"][None])
    rot = O.ellipse_rotation(g["xstart"], g["xgoal"]) if g["kind"] == "informed" else None
    desc = batch.make_desc([0], g["xstart"][None], g["xgoal"][None], None if rot is None else rot[None])
    balls = g["balls"][None] if g["kind"] == "informed" else None
    return ctx.plan(KIND[g["kind"]], desc, g["n"], float(g["r_rewire"]), float(g["r_goal"]),
                    samples=g["samples"][None].astype(np.int16), balls=balls)


def test_plan_golden(ctx, golden_plan):
    g = golden_plan
    pts, cost, parent, stats, ell = run_golden(ctx, g)
    st = dict(zip(_lib.STAT_NAMES, (int(v) for v in stats[0])))
    P, Cc, Pa = c_oracle.rows_like_reference(pts[0], cost[0], parent[0], st["j"], st["vgoal"], bool(st["found"]), g["n"])
    assert P.shape[0] == int(g["rows"])
    assert np.array_equal(P, g["points"])
    assert np.array_equal(Pa, g["parents"])
    assert np.array_equal(Cc.view(np.int64), g["vcosts"].view(np.int64))          # FP64 bit-exact
    assert st["vgoal"] == int(g["vgoal"])
    if g["kind"] == "informed":
        keys = np.flatnonzero(~np.isnan(ell[0]))
        assert np.array_equal(keys, g["ell_keys"])
    # rows the reference leaves unfilled carry the documented sentinels
    top = st["j"] + (1 if st["found"] else 0)
    assert (pts[0][top:] == -32768).all() and np.isinf(cost[0][top:]).all() and (parent[0][top:] == -1).all()


def test_plan_golden_wide_kernel(ctx, golden_plan, monkeypatch):
    """The 32-bit-distance kernel (csrc/plan_wide.cu: grids beyond the packed-key kernel's 2896 / 2048 / 1448 cells a side,
    or tree shapes it does not take) on every golden fixture; RRTK_PLAN_IMPL is read at each launch."""
    monkeypatch.setenv("RRTK_PLAN_IMPL", "wide")
    test_plan_golden(ctx, golden_plan)


@pytest.mark.parametrize("kind", ["standard", "star", "informed"])
def test_wide_grid_takes_the_wide_kernel_by_default(kind):
    """A 3008 x 3008 world is beyond the packed keys: the default dispatch must hand it to plan_wide.cu and still equal the
    C oracle bit for bit (also with the environment override absent)."""
    assert "RRTK_PLAN_IMPL" not in os.environ
    W = H = 3008
    n = 700
    og = worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(5))
    xs, xg = worlds.start_goal(og, 5)
    if kind == "informed":                       # a goal the tree reaches early, so the ellipse phase runs
        free = np.argwhere(og == 0)
        near = free[np.argsort(((free - xs) ** 2).sum(1), kind="stable")]
        xg = near[min(len(near) - 1, 4000)]
    smp = O.sample_stream(og, n, 9)
    rot = O.ellipse_rotation(xs, xg) if kind == "informed" else None
    u = np.random.default_rng(3).uniform(0, 1, size=(n, 2))
    balls = np.stack([np.sqrt(u[:, 0]) * np.cos(2 * np.pi * u[:, 1]), np.sqrt(u[:, 0]) * np.sin(2 * np.pi * u[:, 1])], axis=-1) if kind == "informed" else None
    r, rg = (0.0, 0.0) if kind == "standard" else (400.0, 300.0 if kind == "informed" else 0.0)
    db = batch.DeviceBatch(kind, W, H, n, r, rg)
    db.set_worlds_host(og[None].astype(np.uint8))
    db.set_plans(batch.make_desc([0], xs[None], xg[None], None if rot is None else rot[None]))
    db.set_samples_host(smp[None])
    if kind == "informed":
        db.set_balls_host(balls[None])
    res = db.run().download()
    assert_same_as_oracle(res, 0, oracle_tree(kind, og.astype(np.uint8), n, xs, xg, smp, r, rg, balls, rot))


@pytest.mark.parametrize("threads", [64, 128, 256])
def test_plan_result_independent_of_block_size(golden_plan, threads):
    g = golden_plan
    db = batch.DeviceBatch(g["kind"], g["og"].shape[0], g["og"].shape[1], g["n"], float(g["r_rewire"]), float(g["r_goal"]), threads=threads)
    db.set_worlds_host(g["og"][None])
    rot = O.ellipse_rotation(g["xstart"], g["xgoal"]) if g["kind"] == "informed" else None
    db.set_plans(batch.make_desc([0], g["xstart"][None], g["xgoal"][None], None if rot is None else rot[None]))
    db.set_samples_host(g["samples"][None])
    if g["kind"] == "informed":
        db.set_balls_host(g["balls"][None])
    r = db.run().download()
    P, Cc, Pa = c_oracle.rows_like_reference(r.pts[0], r.cost[0], r.parent[0], int(r.stats[0, 0]), int(r.stats[0, 1]), bool(r.stats[0, 2]), g["n"])
    assert np.array_equal(P, g["points"]) and np.array_equal(Pa, g["parents"])
    assert np.array_equal(Cc.view(np.int64), g["vcosts"].view(np.int64))


def oracle_tree(kind, og, n, xs, xg, samples, r=0.0, rg=0.0, balls=None, rot=None):
    return c_oracle.plan_raw(kind, og, n, xs, xg, samples, r, rg, balls, rot)


def assert_same_as_oracle(res, p, want):
    wp, wc, wpar, wst, well = want
    j, found = wst["j"], bool(wst["found"])
    top = j + (1 if found else 0)
    assert int(res.stats[p, 0]) == j and int(res.stats[p, 1]) == wst["vgoal"] and bool(res.stats[p, 2]) == found
    assert np.array_equal(res.pts[p, :top], wp[:top])
    assert np.array_equal(res.parent[p, :top], wpar[:top])
    assert np.array_equal(res.cost[p, :top].view(np.int64), wc[:top].view(np.int64))
    assert int(res.stats[p, _lib.STAT_NAMES.index("nn_pairs")]) <= wst["nn_pairs"]
    assert int(res.stats[p, _lib.STAT_NAMES.index("accepted")]) == wst["accepted"]
    if "ring_members" in wst:   # sum over accepted iterations of |within(points, xnew, r_rewire)| (filled rows)
        assert int(res.stats[p, _lib.STAT_NAMES.index("ring_members")]) == wst["ring_members"]
    if found:   # north star: path cost within 1e-5 relative (it is bit-equal, checked above)
        assert abs(res.path_cost(p) - wc[j]) <= 1e-5 * wc[j]


@pytest.mark.parametrize("kind", ["standard", "star"])
def test_cfg3_batch_vs_oracle(kind):
    """BASELINE cfg3 shape (512^2, n=5000, r=50) on a 24-plan batch: every tree bit-exact."""
    W = H = 512
    n, nplans = 5000, 24
    db = batch.DeviceBatch(kind, W, H, n, 50.0).gen_worlds([worlds.world_seed(w) for w in range(nplans)])
    ogs = db.og.cpu().numpy()
    pairs = [worlds.start_goal(ogs[p], p) for p in range(nplans)]
    db.set_plans(batch.make_desc(np.arange(nplans), [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(nplans))
    res = db.run().download()
    samples = db.samples.cpu().numpy()
    for p in range(nplans):
        assert np.array_equal(samples[p].astype(np.int64), O.sample_stream(ogs[p], n, p))
        want = oracle_tree(kind, ogs[p], n, pairs[p][0], pairs[p][1], samples[p], 50.0)
        assert_same_as_oracle(res, p, want)
    # device-side path extraction == parent walk
    path, ln = db.paths(512)
    path, ln = path.cpu().numpy(), ln.cpu().numpy()
    for p in range(nplans):
        assert path[p, :ln[p]].tolist() == res.path(p)


@pytest.mark.parametrize("kind,W,H,n,r", [("star", 300, 200, 2500, 30.0), ("star", 1000, 700, 3000, 80.0), ("standard", 2048, 64, 4000, 0.0),
                                           ("star", 512, 512, 2100, 12.5), ("star", 130, 130, 5100, 300.0)])
def test_bucket_kernel_shapes_vs_oracle(kind, W, H, n, r):
    """The bucket form of K7 (plan_grid.cuh) on shapes other than cfg3 -- non-square and non-power-of-two grids, keys that do not
    fit one word (1000 x 700), a radius below one bucket and one that covers the grid (every vertex is a member: the list
    overflows into the all-slot path) -- must be the kernel the dispatch picks, and every tree equal to the C oracle's."""
    nplans = 3
    db = batch.DeviceBatch(kind, W, H, n, r)
    assert db.L.rrtk_plan_kernel(db.kind, W, H, n, 0).decode() == "grid"
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=50 + w) for w in range(nplans)]).astype(np.uint8)
    db.set_worlds_host(ogs)
    pairs = [worlds.start_goal(ogs[p], p) for p in range(nplans)]
    db.set_plans(batch.make_desc(np.arange(nplans), [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(10 + np.arange(nplans))
    res = db.run().download()
    samples = db.samples.cpu().numpy()
    for p in range(nplans):
        want = oracle_tree(kind, ogs[p], n, pairs[p][0], pairs[p][1], samples[p], r)
        assert_same_as_oracle(res, p, want)


def test_cfg4_informed_vs_oracle():
    """BASELINE cfg4 shape: one 1024^2 world, several pairs, n=20000, r=50, r_goal=5."""
    W = H = 1024
    n, nplans = 20000, 4
    og = worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(0)).astype(np.uint8)
    pairs = [worlds.start_goal(og, p) for p in range(nplans)]
    rots = np.stack([O.ellipse_rotation(a, b) for a, b in pairs])
    rng = np.random.default_rng(3)
    balls = np.stack([np.stack([O.unitball_from_uniform(*rng.uniform(0, 1, 2)) for _ in range(n)]) for _ in range(nplans)])
    samples = np.stack([O.sample_stream(og, n, 100 + p) for p in range(nplans)])
    res = batch.plan_batch("informed", og, n, [a for a, _ in pairs], [b for _, b in pairs], np.zeros(nplans, int), 50.0, 5.0,
                           samples=samples, balls=balls, rots=rots)
    for p in range(nplans):
        want = oracle_tree("informed", og, n, pairs[p][0], pairs[p][1], samples[p], 50.0, 5.0, balls[p], rots[p])
        assert_same_as_oracle(res, p, want)
        assert int(res.stats[p, 5]) == want[3]["first_solution_iter"] and int(res.stats[p, 6]) == want[3]["ellipse_iters"]
        well = want[4]
        got = res.ell_c[p]
        assert np.array_equal(np.isnan(got), np.isnan(well)) and np.array_equal(got[~np.isnan(got)], well[~np.isnan(well)])


def test_batch_properties_full_size():
    """Size-independent properties on a 296-plan cfg3 batch (more plans than one wave of blocks)."""
    W = H = 512
    n, nplans, nworlds = 5000, 296, 37
    db = batch.DeviceBatch("star", W, H, n, 50.0).gen_worlds([worlds.world_seed(w) for w in range(nworlds)])
    ogs = db.og.cpu().numpy()
    wid = np.arange(nplans) % nworlds
    pairs = [worlds.start_goal(ogs[wid[p]], p) for p in range(nplans)]
    db.set_plans(batch.make_desc(wid, [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(nplans) % 50)          # plans p and p+50k on the same world share a stream only if wid matches
    a = db.run().download()
    b = db.run().download()                           # idempotent: same inputs, same bits
    for f in ("pts", "cost", "parent"):
        assert np.array_equal(getattr(a, f), getattr(b, f))
    # statistics too, except the two work counters: how many goal-connection candidates get pruned
    # depends on which warp publishes its result first (results never do)
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    assert np.array_equal(a.stats[:, keep], b.stats[:, keep])
    j = a.stat("j")
    assert (j >= 2).all() and (j <= n).all()
    for p in range(0, nplans, 7):
        jp = int(j[p])
        par, pts, cost = a.parent[p], a.pts[p].astype(np.int64), a.cost[p]
        assert (par[1:jp] >= 0).all() and (par[1:jp] < np.arange(1, jp)).all()      # parents precede children
        seg = np.sqrt(((pts[1:jp] - pts[par[1:jp]]) ** 2).sum(1).astype(np.float64))
        assert np.array_equal(cost[1:jp], cost[par[1:jp]] + seg)                      # cost = parent cost + length, exactly
        # every tree edge is collision free in the oracle's grid walk
        segs = np.concatenate([pts[par[1:jp]], pts[1:jp]], axis=1)
        assert c_oracle.collision_batch(ogs[wid[p]], segs)[0].all()
        assert len(np.unique(pts[1:jp], axis=0)) == jp - 1                            # `sampled` set: no duplicate vertices >= 1
    # a plan's result does not depend on its position in the batch: rerun a slice alone
    sub = [5, 100, 295]
    db2 = batch.DeviceBatch("star", W, H, n, 50.0).set_worlds_host(ogs)
    db2.set_plans(batch.make_desc(wid[sub], [pairs[p][0] for p in sub], [pairs[p][1] for p in sub]))
    db2.set_samples_host(db.samples.cpu().numpy()[sub])
    c = db2.run().download()
    for k, p in enumerate(sub):
        assert np.array_equal(c.pts[k], a.pts[p]) and np.array_equal(c.cost[k].view(np.int64), a.cost[p].view(np.int64))
        assert np.array_equal(c.parent[k], a.parent[p]) and np.array_equal(c.stats[k][keep], a.stats[p][keep])


def test_pipelined_host_call_equals_device_batch():
    """rrtk_ctx_plan_worlds (chunked upload/plan/download on rotating streams) == one-shot DeviceBatch,
    including plans given in arbitrary world order and several plans per world."""
    W, H, n, nworlds, nplans = 160, 128, 600, 9, 41
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=30 + w) for w in range(nworlds)]).astype(np.uint8)
    rng = np.random.default_rng(2)
    wid = rng.integers(0, nworlds, nplans)
    pairs = [worlds.start_goal(ogs[wid[p]], p) for p in range(nplans)]
    starts, goals = [a for a, _ in pairs], [b for _, b in pairs]
    seeds = np.arange(100, 100 + nplans)
    db = batch.DeviceBatch("star", W, H, n, 30.0).set_worlds_host(ogs)
    db.set_plans(batch.make_desc(wid, starts, goals))
    db.seed_samples(seeds)
    want = db.run().download()
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    for chunk in (0, 7, 64):
        c = _lib.Context()
        got = batch.plan_batch("star", ogs, n, starts, goals, wid, 30.0, seeds=seeds, ctx=c) if chunk == 0 else None
        if got is None:
            order = np.argsort(wid, kind="stable")
            res = c.plan_worlds(1, ogs, batch.make_desc(wid, starts, goals)[order], n, 30.0, states=batch.seed_states(seeds)[order], chunk=chunk)
            inv = np.empty_like(order)
            inv[order] = np.arange(nplans)
            got = batch.BatchResult(*[a[inv] if a is not None else None for a in res])
        c.close()
        assert np.array_equal(got.pts, want.pts) and np.array_equal(got.parent, want.parent)
        assert np.array_equal(got.cost.view(np.int64), want.cost.view(np.int64))
        assert np.array_equal(got.stats[:, keep], want.stats[:, keep])
    with pytest.raises(ValueError):      # unordered plans are rejected by the C entry point itself
        c = _lib.Context()
        c.plan_worlds(1, ogs, batch.make_desc([1, 0], starts[:2], goals[:2]), n, 30.0, states=batch.seed_states(seeds[:2]))


def test_packed_grids_in_path_records_out():
    """rrtk_ctx_plan_worlds2: tiled bit grids from the host packer in (RRTK_IN_BITS), path records out (RRTK_OUT_PATHS) ==
    the trees the tree mode returns, walked on the host the way RRT.route2gv / vertices_as_ndarray do (rrt.py:87-129)."""
    W, H, n, nworlds = 100, 70, 500, 6                       # H not a multiple of 32: padded tiles
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=60 + w) for w in range(nworlds)]).astype(np.uint8)
    wid = np.repeat(np.arange(nworlds), 3)
    nplans = wid.size
    pairs = [worlds.start_goal(ogs[wid[p]], 7 * p) for p in range(nplans)]
    desc = batch.make_desc(wid, [a for a, _ in pairs], [b for _, b in pairs])
    st = batch.seed_states(np.arange(500, 500 + nplans))
    c = _lib.Context()
    cap = 64
    trees = c.plan_worlds2(1, ogs, W, H, desc, n, 25.0, states=st, bits=False, trees=True, paths=False, chunk=5)
    bits = _lib.pack_grids_host(ogs)
    assert np.array_equal(bits, np.stack([tiled_bits(g) for g in ogs]))
    both = c.plan_worlds2(1, bits, W, H, desc, n, 25.0, states=st, bits=True, trees=True, paths=True, path_cap=cap, chunk=4)
    only = c.plan_worlds2(1, bits, W, H, desc, n, 25.0, states=st, bits=True, trees=False, paths=True, path_cap=cap)
    c.close()
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    for k in ("pts", "parent"):
        assert np.array_equal(trees[k], both[k])
    assert np.array_equal(trees["cost"].view(np.int64), both["cost"].view(np.int64))
    assert np.array_equal(trees["stats"][:, keep], both["stats"][:, keep]) and np.array_equal(only["stats"][:, keep], both["stats"][:, keep])
    assert "pts" not in only
    res = batch.BatchResult(trees["pts"], trees["cost"], trees["parent"], trees["stats"])
    some_found = False
    for p in range(nplans):
        want = res.path(p)                                   # parent walk on the host
        some_found |= bool(trees["stats"][p, 2])
        for got in (both, only):
            assert int(got["len"][p]) == len(want)
            assert got["path_cost"][p].view(np.int64) == np.float64(res.path_cost(p)).view(np.int64)
            if len(want) <= cap:
                assert got["path"][p, : len(want)].tolist() == want and (got["path"][p, len(want):] == -1).all()
                assert np.array_equal(got["xy"][p, : len(want)], trees["pts"][p][want])
                assert (got["xy"][p, len(want):] == -32768).all()
    assert some_found
    with pytest.raises(ValueError):                          # a requested mode without its buffers is refused by the C entry point
        L = _lib.lib()
        _lib.check(L.rrtk_ctx_plan_worlds2(_lib.Context()._h, 1, _lib.ptr(bits), nworlds, W, H, _lib.ptr(desc), nplans, n, 25.0, 0.0, None,
                                           _lib.ptr(st), None, 1 | 4, cap, None, None, None, _lib.ptr(only["stats"]), None, None, None, None, None, 0))


def test_device_path_records_and_gather_single_rank():
    """DeviceBatch.path_records (rrtk_extract_paths_xy) on real trees; multigpu.gather_tensors with one rank over NCCL."""
    import torch
    import torch.distributed as dist
    from rrtplanner_b200 import multigpu
    W, H, n, P = 128, 128, 800, 24
    db = batch.DeviceBatch("star", W, H, n, 30.0).gen_worlds([worlds.world_seed(w) for w in range(P)])
    ogs = db.og.cpu().numpy()
    pairs = [worlds.start_goal(ogs[p], p) for p in range(P)]
    db.set_plans(batch.make_desc(np.arange(P), [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(P))
    res = db.run().download()
    rec = db.path_records(96)
    torch.cuda.synchronize()
    for p in range(P):
        want = res.path(p)
        assert int(rec["len"][p]) == len(want) and rec["path"][p, : len(want)].tolist() == want
        assert np.array_equal(rec["xy"][p, : len(want)].cpu().numpy(), res.pts[p][want])
        assert rec["path_cost"][p].item() == res.path_cost(p)
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29531")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    got = multigpu.gather_tensors(rec, P, dst=0)
    assert all(torch.equal(got[k], rec[k]) for k in rec)
    dist.destroy_process_group()


# ---- edge cases ----------------------------------------------------------------------------------------
def small_case(ctx, kind, og, n, xs, xg, samples, r=0.0, rg=0.0, balls=None):
    ctx.set_grids((og != 0).astype(np.uint8)[None])
    rot = O.ellipse_rotation(xs, xg) if kind == "informed" and not np.array_equal(xs, xg) else np.eye(2)
    desc = batch.make_desc([0], np.asarray(xs)[None], np.asarray(xg)[None], rot[None])
    pts, cost, parent, stats, ell = ctx.plan(KIND[kind], desc, n, r, rg, samples=np.asarray(samples, dtype=np.int16)[None],
                                             balls=None if balls is None else balls[None])
    res = batch.BatchResult(pts, cost, parent, stats, ell)
    want = oracle_tree(kind, og, n, xs, xg, np.asarray(samples), r, rg, balls, rot)
    assert_same_as_oracle(res, 0, want)
    return res


def edge_cases():
    """(name, og, n, xs, xg, samples, r, rg, balls) of the small worlds the edge-case tests run, in a fixed draw order."""
    rng = np.random.default_rng(8)
    balls = lambda n: np.stack([O.unitball_from_uniform(*rng.uniform(0, 1, 2)) for _ in range(n)])  # noqa: E731
    empty = np.zeros((30, 20), dtype=np.uint8)
    cases = []
    # n = 1: a single iteration, tree can never grow (j != n gate), goal connects to the root
    cases.append(("n1", empty, 1, [2, 2], [25, 15], [[5, 5]], 10, 5, balls(1)))
    # n = 2
    cases.append(("n2", empty, 2, [2, 2], [25, 15], [[5, 5], [6, 6]], 10, 5, balls(2)))
    # every sample identical; sample equal to the start; sample equal to the goal
    cases.append(("same_sample", empty, 20, [2, 2], [25, 15], [[7, 7]] * 20, 10, 5, balls(20)))
    cases.append(("start_goal_samples", empty, 20, [2, 2], [25, 15], [[2, 2]] * 10 + [[25, 15]] * 10, 10, 5, balls(20)))
    # start == goal (probe of the informed phase uses the identity rotation here)
    cases.append(("start_is_goal", empty, 30, [9, 9], [9, 9], rng.integers(0, 20, (30, 2)), 8, 3, balls(30)))
    # wall: goal unreachable, vgoal = 0
    wall = np.zeros((40, 30), dtype=np.uint8)
    wall[20] = 1
    left = np.argwhere(wall[:20] == 0)
    cases.append(("wall", wall, 50, [3, 3], [35, 20], left[rng.integers(0, len(left), 50)], 10, 4, balls(50)))
    # start inside an obstacle: nothing is ever visible from it
    blocked = np.zeros((16, 16), dtype=np.uint8)
    blocked[4, 4] = 1
    cases.append(("blocked_start", blocked, 25, [4, 4], [12, 12], rng.integers(0, 16, (25, 2)), 6, 3, balls(25)))
    # huge radius on a tiny grid: the radius set is the whole tree every time
    cases.append(("huge_radius", empty, 120, [0, 0], [29, 19], rng.integers(0, 20, (120, 2)), 1e6, 4, balls(120)))
    # radius 0 and non-integer radius
    cases.append(("radius0", empty, 60, [0, 0], [29, 19], rng.integers(0, 20, (60, 2)), 0.0, 0.0, balls(60)))
    cases.append(("radius7.5", empty, 60, [0, 0], [29, 19], rng.integers(0, 20, (60, 2)), 7.5, 2.5, balls(60)))
    # 1-wide grids
    line = np.zeros((1, 64), dtype=np.uint8)
    line[0, 40] = 1
    cases.append(("one_wide", line, 40, [0, 1], [0, 60], np.stack([np.zeros(40, int), rng.integers(0, 64, 40)], 1), 9, 3, balls(40)))
    return cases


def run_edge_case(ctx, kind, case):
    name, og, n, xs, xg, samples, r, rg, balls = case
    res = small_case(ctx, kind, og, n, xs, xg, samples, r, rg, balls)
    if name == "wall":
        assert int(res.stats[0, 1]) == 0 and int(res.stats[0, 2]) == 0
    return res


@pytest.mark.parametrize("kind", ["standard", "star", "informed"])
def test_edge_cases(ctx, kind):
    for case in edge_cases():
        run_edge_case(ctx, kind, case)


def test_plan_rejects_bad_inputs(ctx):
    ctx.set_grids(np.zeros((1, 20, 20), dtype=np.uint8))
    good = batch.make_desc([0], [[1, 1]], [[5, 5]])
    smp = np.zeros((1, 10, 2), dtype=np.int16)
    with pytest.raises(ValueError):
        ctx.plan(1, batch.make_desc([0], [[1, 1]], [[20, 5]]), 10, 5.0, samples=smp)
    with pytest.raises(ValueError):
        ctx.plan(1, batch.make_desc([1], [[1, 1]], [[5, 5]]), 10, 5.0, samples=smp)
    bad = smp.copy()
    bad[0, 3] = (25, 0)
    with pytest.raises(ValueError):
        ctx.plan(1, good, 10, 5.0, samples=bad)
    with pytest.raises(ValueError):
        ctx.plan(1, good, 10, 5.0)                      # neither samples nor seeds
    with pytest.raises(MemoryError):
        ctx.plan(1, good, 65000, 5.0, samples=np.zeros((1, 65000, 2), dtype=np.int16))   # tree does not fit shared memory


def test_world_without_free_cells_cannot_be_sampled(ctx):
    """Seed mode draws free[choice(nfree)] (rrt.py:240); numpy raises for nfree = 0, and so do the host-buffer entry points and
    the DeviceBatch wrapper instead of handing the planner an occupied cell (explicit sample streams stay legal)."""
    full = np.ones((2, 40, 40), dtype=np.uint8)
    full[1, 3, 4] = 0                                             # world 1 has exactly one free cell
    assert ctx.set_grids(full).tolist() == [0, 1]
    st = batch.seed_states([5])
    with pytest.raises(ValueError, match="no free cell"):
        ctx.plan(1, batch.make_desc([0], [[1, 1]], [[2, 2]]), 10, 5.0, states=st)
    with pytest.raises(ValueError, match="no free cell"):
        ctx.samples(batch.make_desc([0], [[1, 1]], [[2, 2]]), 10, st)
    smp = ctx.samples(batch.make_desc([1], [[1, 1]], [[2, 2]]), 10, st)        # one free cell: every draw is that cell
    assert (smp[0] == [3, 4]).all()
    ctx.plan(1, batch.make_desc([0], [[1, 1]], [[2, 2]]), 4, 5.0, samples=np.zeros((1, 4, 2), dtype=np.int16))
    db = batch.DeviceBatch("star", 40, 40, 10, 5.0).set_worlds_host(full)
    db.set_plans(batch.make_desc([0], [[1, 1]], [[2, 2]]))
    with pytest.raises(ValueError, match="no free cell"):
        db.seed_samples([5])
    # the pipelined calls find out on the device (the free-cell index is built there) and report after the call
    desc2 = batch.make_desc([0, 1], [[1, 1], [3, 4]], [[2, 2], [3, 4]])
    with pytest.raises(ValueError, match="no free cell"):
        ctx.plan_worlds2(1, full, 40, 40, desc2, 10, 5.0, states=batch.seed_states([5, 6]))
    ctx.plan_worlds2(1, full, 40, 40, desc2[1:], 10, 5.0, states=batch.seed_states([6]))          # world 1 alone is fine
    ctx.plan_worlds2(1, full, 40, 40, desc2, 4, 5.0, samples=np.zeros((2, 4, 2), dtype=np.int16))  # explicit streams stay legal
    with pytest.raises(ValueError, match="no free cell"):
        ctx.plan2_worlds(_lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 5.0), full, 40, 40, desc2, 10, states=batch.seed_states([5, 6]))
