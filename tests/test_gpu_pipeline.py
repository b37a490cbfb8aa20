"""The chunked upload / plan / download pipeline of the pipelined host calls (rrtk_ctx_plan_worlds2, rrtk_ctx_plan2_worlds).

Small cases with many more chunks than the pipeline has slots, so that every slot is reused and each chunk waits for the
slot's previous chunk to be downloaded, against the resident calls (rrtk_ctx_set_grids + rrtk_ctx_plan / rrtk_ctx_plan2) on
the same inputs; and contexts that ran a pipelined call give all their device memory back on close()."""
import numpy as np
import pytest

from rrtplanner_b200 import _lib, batch, worlds

pytestmark = pytest.mark.gpu

W = H = 96
NWORLDS, NPLANS, N, CAP, CHUNK = 6, 25, 300, 64, 2       # 13 chunks over the 5 slots


def case(seed):
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=seed + w) for w in range(NWORLDS)]).astype(np.uint8)
    wid = np.sort(np.random.default_rng(seed).integers(0, NWORLDS, NPLANS))
    pairs = [worlds.start_goal(ogs[wid[p]], seed + p) for p in range(NPLANS)]
    starts, goals = np.array([a for a, _ in pairs]), np.array([b for _, b in pairs])
    rng = np.random.default_rng(seed + 1)
    free = [np.argwhere(og == 0) for og in ogs]
    smp = np.stack([free[w][rng.integers(0, len(free[w]), N)] for w in wid]).astype(np.int16)
    states = batch.seed_states(np.arange(NPLANS) + seed)
    balls = rng.uniform(-0.7, 0.7, (NPLANS, N, 2))          # inside the unit disc
    return ogs, wid, starts, goals, smp, states, balls, rng


def parent_chain(parent, v):
    chain = [v]
    while chain[-1] > 0:
        chain.append(int(parent[chain[-1]]))
    return chain[::-1]


def assert_records(got, pts, cost, parent, stats, head=None):
    """Path records of the pipelined call == the parent walk of the resident trees."""
    for p in range(NPLANS):
        v = int(stats[p, 1])                                                    # vgoal, in both families' statistics
        chain = parent_chain(parent[p], v)
        assert got["len"][p] == len(chain)
        assert got["path_cost"][p].view(np.int64) == cost[p, v].view(np.int64)
        if len(chain) <= CAP:
            assert list(got["path"][p, :len(chain)]) == chain and (got["path"][p, len(chain):] == -1).all()
            assert np.array_equal(got["xy"][p, :len(chain)], pts[p, chain])
            if head is not None:
                assert np.array_equal(got["path_head"][p, :len(chain)], head[p, chain])


@pytest.mark.parametrize("kind,bits,source", [("star", False, "samples"), ("star", True, "samples"), ("star", False, "states"),
                                              ("star", True, "states"), ("informed", True, "states")])
def test_plan_worlds2_reuses_every_slot(kind, bits, source):
    ogs, wid, starts, goals, smp, states, balls, _ = case(70)
    k = {"star": _lib.KIND_STAR, "informed": _lib.KIND_INFORMED}[kind]
    rots = batch.informed_rotations(starts, goals) if kind == "informed" else None
    desc = batch.make_desc(wid, starts, goals, rots)
    inp = dict(samples=smp) if source == "samples" else dict(states=states)
    b = balls if kind == "informed" else None
    c = _lib.Context()
    c.set_grids(ogs)
    pts, cost, parent, stats, ell = c.plan(k, desc, N, 20.0, 6.0, balls=b, **inp)
    grids = _lib.pack_grids_host(ogs) if bits else ogs
    kw = dict(bits=bits, trees=True, paths=True, path_cap=CAP, chunk=CHUNK, balls=b, **inp)
    got = c.plan_worlds2(k, grids, W, H, desc, N, 20.0, 6.0, **kw)
    cut = c.plan_worlds2(k, grids, W, H, desc, N, 20.0, 6.0, shortcut=True, **kw)
    after = c.shortcut(got["xy"], got["len"], world=wid, path=got["path"])
    c.close()
    assert np.array_equal(got["pts"], pts) and np.array_equal(got["parent"], parent)
    assert np.array_equal(got["cost"].view(np.int64), cost.view(np.int64))
    if ell is not None:
        assert np.array_equal(got["ell"].view(np.int64), ell.view(np.int64))
    keep = [i for i, nm in enumerate(_lib.STAT_NAMES) if nm not in ("checks", "cells")]
    assert np.array_equal(got["stats"][:, keep], stats[:, keep]) and np.array_equal(cut["stats"][:, keep], stats[:, keep])
    assert stats[:, 2].sum() > NPLANS // 2                                       # most plans found their goal
    assert_records(got, pts, cost, parent, stats)
    assert np.array_equal(cut["len"], after["len"])
    for key in ("xy", "path"):
        assert np.array_equal(cut[key], after[key]), key
    assert np.array_equal(cut["path_cost"].view(np.int64), after["cost"].view(np.int64))


@pytest.mark.parametrize("model,bits,source", [("dubins", False, "samples"), ("dubins", True, "samples"), ("dubins", False, "states"),
                                               ("dubins", True, "states"), ("informed", True, "states")])
def test_plan2_worlds_reuses_every_slot(model, bits, source):
    ogs, wid, starts, goals, smp, states, balls, rng = case(90)
    nh = 8
    hd = rng.integers(0, nh, (NPLANS, N)).astype(np.uint8)
    s3 = np.concatenate([starts, (np.arange(NPLANS) % nh)[:, None]], axis=1)
    g3 = np.concatenate([goals, ((5 * np.arange(NPLANS)) % nh)[:, None]], axis=1)
    desc = batch.make_desc2(wid, s3, g3)
    if model == "informed":
        cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 20.0, informed=True, r_goal=6.0)
        desc["rot"] = batch.informed_rotations(starts, goals).reshape(NPLANS, 4)
        b, hd = balls, None
    else:
        cfg = _lib.plan2_cfg(_lib.MODEL_DUBINS, True, True, 20.0, nh, 3.0, 1.0)
        b = None
    inp = dict(samples=smp) if source == "samples" else dict(states=states)
    c = _lib.Context()
    c.set_grids(ogs)
    want = c.plan2(cfg, desc, N, heads=hd, balls=b, **inp)
    pts, head, cost, elen, parent, stats = want[:6]
    grids = _lib.pack_grids_host(ogs) if bits else ogs
    got = c.plan2_worlds(cfg, grids, W, H, desc, N, heads=hd, bits=bits, trees=True, paths=True, path_cap=CAP, chunk=CHUNK, balls=b, **inp)
    c.close()
    assert np.array_equal(got["pts"], pts) and np.array_equal(got["head"], head) and np.array_equal(got["parent"], parent)
    assert np.array_equal(got["cost"].view(np.int64), cost.view(np.int64)) and np.array_equal(got["elen"].view(np.int64), elen.view(np.int64))
    if model == "informed":
        assert np.array_equal(got["ell"].view(np.int64), want[6].view(np.int64))
    keep = [i for i, nm in enumerate(_lib.STAT2_NAMES) if nm != "checks"]     # as test_pipelined_worlds_call_equals_the_resident_call
    assert np.array_equal(got["stats"][:, keep], stats[:, keep])
    assert stats[:, 2].sum() > NPLANS // 2
    assert_records(got, pts, cost, parent, stats, head)


@pytest.mark.parametrize("family", ["plan_worlds2", "plan2_worlds"])
def test_close_frees_every_slot_buffer(family):
    """Four contexts, each filling all five slots with 1024-plan chunks of 4096-entry path records, then closed: the device
    memory they used comes back (a context that kept its path-record buffers would hold about 160 MB each)."""
    import torch
    nplans, n, cap = 5120, 16, 4096
    og = np.zeros((1, 32, 32), dtype=np.uint8)
    desc = batch.make_desc(np.zeros(nplans, dtype=np.int64), np.tile([[1, 1]], (nplans, 1)), np.tile([[30, 30]], (nplans, 1)))
    states = batch.seed_states(np.arange(nplans))
    cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 5.0)

    def cycle():
        c = _lib.Context()
        if family == "plan_worlds2":
            c.plan_worlds2(_lib.KIND_STAR, og, 32, 32, desc, n, 5.0, states=states, paths=True, path_cap=cap, chunk=1024)
        else:
            c.plan2_worlds(cfg, og, 32, 32, desc, n, states=states, paths=True, path_cap=cap, chunk=1024)
        c.close()

    torch.cuda.init()
    cycle()                                                                     # module loading and other one-time costs
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(4):
        cycle()
    lost = free0 - torch.cuda.mem_get_info()[0]
    print(f"{family}: {lost / 2**20:.1f} MB of device memory not given back after 4 contexts")
    assert lost < 256 << 20
