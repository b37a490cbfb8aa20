"""Path shortcutting on the device (csrc/shortcut.cu, rrtk_shortcut_paths / rrtk_ctx_shortcut / RRTK_OUT_SHORTCUT) against
its specification oracle/shortcut_oracle.py, bit for bit: random polylines, real path records, the fused pipeline flag and
the Python entry points."""
import os

import numpy as np
import pytest

from oracle import shortcut_oracle as S
from rrtplanner_b200 import RRTStar, _lib, batch, worlds
from tests.conftest import golden_plans, load_plan
from tests.test_shortcut_host import hand_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = _lib.Context()
    yield c
    c.close()


def assert_same(got, want):
    for k in ("xy", "len", "keep"):
        assert np.array_equal(got[k], want[k]), k
    assert (got["path"] is None) == (want["path"] is None)
    if want["path"] is not None:
        assert np.array_equal(got["path"], want["path"])
    assert np.array_equal(got["cost"].view(np.int64), want["cost"].view(np.int64))


def blobs(W, H, seed):
    """Random discs of obstacle on an empty (W, H) grid."""
    rng = np.random.default_rng(seed)
    og = np.zeros((W, H), dtype=np.uint8)
    xs, ys = np.meshgrid(np.arange(W), np.arange(H), indexing="ij")
    for _ in range(max(2, W * H // 900)):
        cx, cy, r = rng.integers(0, W), rng.integers(0, H), rng.integers(1, max(2, min(W, H) // 6) + 1)
        og[(xs - cx) ** 2 + (ys - cy) ** 2 <= r * r] = 1
    return og


def random_rows(ogs, P, cap, rng, max_len=None):
    """P rows of cap entries: random-walk polylines (steps up to a tenth of the grid) of random length, some lengths
    outside [1, cap] (not processed), world ids mixed; entries past the length hold junk."""
    nw, W, H = ogs.shape
    xy = rng.integers(-32768, 32767, size=(P, cap, 2)).astype(np.int16)
    top = cap if max_len is None else min(cap, max_len)
    ln = rng.integers(1, top + 1, size=P).astype(np.int32)
    ln[rng.random(P) < 0.1] = 0
    ln[rng.random(P) < 0.05] = cap + 1
    ln[rng.random(P) < 0.02] = -2
    sx, sy = max(1, W // 10), max(1, H // 10)
    for p in range(P):
        m = min(max(int(ln[p]), 0), cap)
        start = rng.integers(0, [W, H])
        steps = np.stack([rng.integers(-sx, sx + 1, m), rng.integers(-sy, sy + 1, m)], axis=1)
        pts = start + np.cumsum(steps, axis=0)
        xy[p, :m] = np.stack([np.clip(pts[:, 0], 0, W - 1), np.clip(pts[:, 1], 0, H - 1)], axis=1)
    world = rng.integers(0, nw, size=P).astype(np.int32)
    ids = rng.integers(0, 60000, size=(P, cap)).astype(np.int32)
    return xy, ln, world, ids


@pytest.mark.parametrize("case", hand_cases(), ids=lambda c: c[0])
def test_hand_made_cases(ctx, case):
    _, og, pts, want = case
    pts = np.asarray(pts)
    cap = len(pts) + 2
    xy = np.full((1, cap, 2), -32768, dtype=np.int16)
    xy[0, : len(pts)] = pts
    ctx.set_grids(og[None])
    got = ctx.shortcut(xy, [len(pts)], path=np.arange(cap, dtype=np.int32)[None])
    assert got["keep"][0, : len(want)].tolist() == want
    assert_same(got, S.shortcut_records(og, xy, [len(pts)], path=np.arange(cap)[None]))


@pytest.mark.parametrize("shape,cap,P", [((100, 77), 32, 300), ((61, 47), 1, 64), ((130, 200), 1024, 6), ((16384, 4), 32, 120),
                                         ((4, 16384), 32, 120), ((16384, 4), 1024, 3)])
def test_random_polylines_vs_oracle(ctx, shape, cap, P):
    W, H = shape
    rng = np.random.default_rng(W * 7 + H + cap)
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=11).astype(np.uint8), blobs(W, H, 12), (rng.random((W, H)) < 0.02).astype(np.uint8)])
    xy, ln, world, ids = random_rows(ogs, P, cap, rng)
    ctx.set_grids(ogs)
    got = ctx.shortcut(xy, ln, world=world, path=ids)
    assert_same(got, S.shortcut_records(ogs, xy, ln, world=world, path=ids))
    assert (got["len"][(ln >= 1) & (ln <= cap)] >= 1).all()
    no_path = ctx.shortcut(xy, ln, world=world)                  # optional outputs left out: the same rows
    assert no_path["path"] is None and np.array_equal(no_path["xy"], got["xy"]) and np.array_equal(no_path["len"], got["len"])


def test_host_entry_rejects_bad_worlds_and_points(ctx):
    ogs = np.zeros((2, 40, 30), dtype=np.uint8)
    ctx.set_grids(ogs)
    xy = np.full((2, 4, 2), 5, dtype=np.int16)
    xy[1, 3] = (40, 0)                                           # past the length of row 1: not checked, not touched
    with pytest.raises(ValueError, match="world"):
        ctx.shortcut(xy, [4, 3], world=[0, 2])
    xy[0, 2] = (3, 30)
    with pytest.raises(ValueError, match="outside"):
        ctx.shortcut(xy, [4, 3])
    got = ctx.shortcut(xy, [2, 3])                               # row 0 processed up to its length only
    assert got["len"].tolist() == [2, 2] and np.array_equal(got["xy"][1, 1], xy[1, 2])


def check_records(ctx, ogs, world, rec, cap):
    """The properties of shortcut records built from tree paths; returns the shortcut dict."""
    got = ctx.shortcut(rec["xy"], rec["len"], world=world, path=rec["path"])
    want = S.shortcut_records(ogs, rec["xy"], rec["len"], world=world, path=rec["path"])
    assert_same(got, want)
    for p in range(len(rec["len"])):
        m, t = int(rec["len"][p]), int(got["len"][p])
        if m < 1 or m > cap:
            continue
        keep = got["keep"][p, :t]
        assert keep[0] == 0 and keep[-1] == m - 1 and (np.diff(keep) > 0).all()
        assert np.array_equal(got["path"][p, :t], rec["path"][p, keep])
        assert got["cost"][p] <= rec["path_cost"][p] * (1 + 1e-12)
        if t == m:
            assert got["cost"][p].view(np.int64) == np.float64(rec["path_cost"][p]).view(np.int64)
        if t > 1:
            segs = np.concatenate([got["xy"][p, : t - 1], got["xy"][p, 1:t]], axis=1).astype(np.int32)
            assert ctx.collision(segs, world=int(world[p])).all()
    again = ctx.shortcut(got["xy"], got["len"], world=world, path=got["path"])        # the greedy pass is idempotent
    for k in ("xy", "len", "path"):
        assert np.array_equal(again[k], got[k]), k
    return got


def test_golden_plan_paths(ctx):
    """The reference's own trees (tests/golden/plan_*.npz): each vgoal's root path as a record on its world."""
    recs = []
    for path in golden_plans():
        g = load_plan(path)
        v, ids = int(g["vgoal"]), []
        while v >= 0:
            ids.append(v)
            v = int(g["parents"][v]) if v > 0 else -1
        ids = ids[::-1]
        recs.append((g, ids))
    for g, ids in recs:
        cap = len(ids) + 1
        rec = dict(xy=np.full((1, cap, 2), -32768, dtype=np.int16), len=np.array([len(ids)], dtype=np.int32),
                   path=np.full((1, cap), -1, dtype=np.int32), path_cost=np.array([g["vcosts"][ids[-1]]]))
        rec["xy"][0, : len(ids)] = g["points"][ids]
        rec["path"][0, : len(ids)] = ids
        ctx.set_grids(g["og"][None])
        check_records(ctx, g["og"][None], np.zeros(1, dtype=np.int32), rec, cap)


def cfg3_batch(P, kind="star"):
    W = H = 512
    n = 5000
    db = batch.DeviceBatch(kind, W, H, n, 50.0).gen_worlds([worlds.world_seed(w) for w in range(P)])
    ogs = db.og.cpu().numpy()
    pairs = [worlds.start_goal(ogs[p], p) for p in range(P)]
    db.set_plans(batch.make_desc(np.arange(P), [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(P))
    db.run()
    return db, ogs, pairs


def test_cfg3_shape_batch_records():
    """Seeded cfg3-shape batch (512^2, n = 5000, RRT*, r = 50): path records of the device trees, shortcut on the host
    entry and by DeviceBatch.shortcut_records, both against the oracle; then a one-rank NCCL gather of the shortcut records."""
    import torch
    import torch.distributed as dist
    from rrtplanner_b200 import multigpu
    P, cap = 96, 1024
    db, ogs, _ = cfg3_batch(P)
    rec = db.path_records(cap)
    host = {k: v.cpu().numpy() for k, v in rec.items()}
    assert (host["len"] > 2).any()
    c = _lib.Context()
    c.set_grids(ogs)
    world = np.arange(P, dtype=np.int32)
    got = check_records(c, ogs, world, host, cap)
    c.close()
    assert (got["len"] < host["len"]).any()
    out = db.shortcut_records(rec)
    assert out is rec
    torch.cuda.synchronize()
    for k in ("xy", "len", "path"):
        assert np.array_equal(rec[k].cpu().numpy(), got[k]), k
    assert np.array_equal(rec["path_cost"].cpu().numpy().view(np.int64), got["cost"].view(np.int64))
    assert np.array_equal(rec["stats"].cpu().numpy(), host["stats"])
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    gathered = multigpu.gather_tensors(rec, P, dst=0)
    assert all(torch.equal(gathered[k], rec[k]) for k in rec)
    dist.destroy_process_group()


def test_device_records_with_unwritten_rows_and_unsorted_worlds():
    """DeviceBatch.shortcut_records equals the host form with plans on worlds out of order and a cap some paths exceed."""
    import torch
    W, H, n, P = 160, 120, 1500, 40
    db = batch.DeviceBatch("star", W, H, n, 25.0).gen_worlds([worlds.world_seed(w) for w in range(5)])
    ogs = db.og.cpu().numpy()
    world = np.random.default_rng(4).integers(0, 5, P).astype(np.int32)
    pairs = [worlds.start_goal(ogs[world[p]], p) for p in range(P)]
    db.set_plans(batch.make_desc(world, [a for a, _ in pairs], [b for _, b in pairs]))
    db.seed_samples(np.arange(P))
    db.run()
    lens = np.sort(db.path_records(1024)["len"].cpu().numpy())
    cap = int(lens[P // 2])                                      # about half of the paths do not fit the records
    rec = db.path_records(cap)
    host = {k: v.cpu().numpy() for k, v in rec.items()}
    assert (host["len"] > cap).any() and (host["len"] <= cap).any()
    want = batch.shortcut_paths(ogs, host["xy"], host["len"], world_ids=world, path=host["path"])
    db.shortcut_records(rec)
    torch.cuda.synchronize()
    live = host["len"] <= cap
    for k in ("xy", "len", "path"):
        assert np.array_equal(rec[k].cpu().numpy(), want[k]), k
    cost = rec["path_cost"].cpu().numpy()
    assert np.array_equal(cost[live].view(np.int64), want["cost"][live].view(np.int64))
    assert np.array_equal(cost[~live].view(np.int64), host["path_cost"][~live].view(np.int64))   # unwritten rows untouched


@pytest.mark.parametrize("bits", [False, True], ids=["uint8", "bits"])
@pytest.mark.parametrize("chunk", [0, 37])
def test_fused_flag_equals_shortcut_after_download(bits, chunk):
    W, H, n, P, nw, cap = 200, 150, 2000, 150, 6, 64
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=worlds.world_seed(w)).astype(np.uint8) for w in range(nw)])
    world = np.sort(np.random.default_rng(5).integers(0, nw, P)).astype(np.int32)
    pairs = [worlds.start_goal(ogs[world[p]], p) for p in range(P)]
    desc = batch.make_desc(world, [a for a, _ in pairs], [b for _, b in pairs])
    st = batch.seed_states(np.arange(P))
    grids = _lib.pack_grids_host(ogs) if bits else ogs
    c = _lib.Context()
    kw = dict(states=st, bits=bits, trees=True, paths=True, path_cap=cap, chunk=chunk)
    plain = c.plan_worlds2(_lib.KIND_STAR, grids, W, H, desc, n, 30.0, **kw)
    fused = c.plan_worlds2(_lib.KIND_STAR, grids, W, H, desc, n, 30.0, shortcut=True, **kw)
    c.set_grids(ogs)
    after = c.shortcut(plain["xy"], plain["len"], world=world, path=plain["path"])
    c.close()
    for k in ("pts", "parent"):
        assert np.array_equal(plain[k], fused[k]), k
    same = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]      # as test_packed_grids_in_path_records_out
    assert np.array_equal(plain["stats"][:, same], fused["stats"][:, same])
    assert np.array_equal(plain["cost"].view(np.int64), fused["cost"].view(np.int64))
    live = (plain["len"] >= 1) & (plain["len"] <= cap)
    assert live.sum() > P // 2 and (after["len"][live] < plain["len"][live]).any()
    assert np.array_equal(fused["len"], after["len"])
    for k in ("xy", "path"):
        assert np.array_equal(fused[k][live], after[k][live]), k
    remapped = np.where(after["keep"][live] >= 0, np.take_along_axis(plain["path"][live], np.maximum(after["keep"][live], 0), axis=1), -1)
    assert np.array_equal(fused["path"][live], remapped)
    assert np.array_equal(fused["path_cost"][live].view(np.int64), after["cost"][live].view(np.int64))
    assert np.array_equal(fused["path_cost"][~live].view(np.int64), plain["path_cost"][~live].view(np.int64))


def test_planner_shortcut_path_follows_set_og():
    og = worlds.perlin_occupancygrid(140, 110, seed=21).astype(np.uint8)
    planner = RRTStar(og, 1500, 25.0, pbar=False, seed=3)
    for pair in range(20):                                       # the first pair whose goal is reached over several edges
        T, gv = planner.plan(*worlds.start_goal(og, pair))
        route = planner.route2gv(T, gv)
        if len(route) > 2:
            break
    assert len(route) > 2
    pts = np.array([T.nodes[v]["pt"] for v in route])
    for grid in (og, np.zeros_like(og), og | blobs(140, 110, 22)):
        if grid is not og:
            planner.set_og(grid)
        got = planner.shortcut_path(T, route)
        assert got == [route[k] for k in S.shortcut_indices(grid, pts)]
    planner.set_og(np.zeros_like(og))
    assert planner.shortcut_path(T, route) == [route[0], route[-1]]
    assert len(planner.vertices_as_ndarray(T, planner.shortcut_path(T, route))) == 1
    assert planner.shortcut_path(T, []) == [] and planner.shortcut_path(T, route[:1]) == route[:1]
