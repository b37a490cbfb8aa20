"""Seeded informed batches, the parts that need no GPU: the stacked rotation, and the argument checks of plan_batch(balls="seed"),
rrtk_ball_streams and the RRTK_SEED_BALLS flag (all raised before any device work)."""
import numpy as np
import pytest

from rrtplanner_b200 import _lib, batch, build as build_mod
from rrtplanner_b200.rrt import RRTStarInformed


@pytest.fixture(scope="module")
def lib():
    build_mod.build()
    return _lib.lib()


def test_informed_rotations_equal_the_class_method_bit_for_bit():
    rng = np.random.default_rng(20)
    P = 12000
    starts = rng.integers(0, 2048, size=(P, 2))
    goals = rng.integers(0, 2048, size=(P, 2))
    goals[:1000, 0] = starts[:1000, 0]                    # dx = 0
    goals[1000:2000, 1] = starts[1000:2000, 1]            # dy = 0
    goals[2000:2050] = starts[2000:2050]                  # start == goal
    goals[2050:2100] = starts[2050:2100] + rng.integers(-1, 2, size=(50, 2))     # neighbours (some equal)
    got = batch.informed_rotations(starts, goals)
    assert got.shape == (P, 2, 2) and got.dtype == np.float64
    helper = RRTStarInformed(np.zeros((4, 4)), 8, 1.0, 1.0, pbar=False)
    same = (starts == goals).all(axis=1)
    assert same[2000:2050].all()
    for p in range(P):
        if same[p]:
            assert np.isnan(got[p]).all()
            with pytest.raises(np.linalg.LinAlgError):
                helper.rotation_to_world_frame(starts[p], goals[p])
            continue
        want = np.asarray(helper.rotation_to_world_frame(starts[p], goals[p]), dtype=np.float64)
        assert np.array_equal(got[p].view(np.int64), want.view(np.int64)), p


def test_plan_batch_seed_balls_argument_checks():
    og = np.zeros((1, 32, 32), dtype=np.uint8)
    kw = dict(r_rewire=5.0, r_goal=2.0)
    with pytest.raises(ValueError, match="seeds"):
        batch.plan_batch("informed", og, 50, [[1, 1]], [[20, 20]], balls="seed", **kw)
    with pytest.raises(ValueError, match="samples"):
        batch.plan_batch("informed", og, 50, [[1, 1]], [[20, 20]], balls="seed", seeds=[0],
                         samples=np.zeros((1, 50, 2), dtype=np.int16), **kw)
    with pytest.raises(ValueError, match="balls"):
        batch.plan_batch("star", og, 50, [[1, 1]], [[20, 20]], balls="seed", seeds=[0], **kw)
    with pytest.raises(ValueError, match="balls"):
        batch.plan_batch("informed", og, 50, [[1, 1]], [[20, 20]], balls="disc", seeds=[0], **kw)
    with pytest.raises(ValueError, match="balls"):
        batch.plan_batch("informed", og, 50, [[1, 1]], [[20, 20]], seeds=[0], **kw)


def test_ball_streams_rejects_bad_arguments(lib):
    buf = np.zeros(64, dtype=np.uint64)
    p = _lib.ptr(buf)
    good = [p, 8, p, 1, 10, p, None, p, 12, p, None, None, None]
    for k in (0, 2, 5, 7, 9):                             # each required pointer NULL
        args = list(good)
        args[k] = None
        assert lib.rrtk_ball_streams(*args) == -1, k
    for k, v in ((3, -1), (4, 0), (4, -5), (8, 0), (8, -12), (1, 0), (1, -3)):     # nplans, n, first_stride, W
        args = list(good)
        args[k] = v
        assert lib.rrtk_ball_streams(*args) == -1, (k, v)
    assert b"rrtk_ball_streams" in lib.rrtk_last_error() or b"grid size" in lib.rrtk_last_error()


def test_seed_balls_flag_misuse_is_rejected_without_a_gpu(lib):
    P, n, W = 2, 16, 32
    grids = np.zeros((1, W, W), dtype=np.uint8)
    desc = batch.make_desc([0, 0], [[1, 1], [2, 2]], [[20, 20], [21, 21]])
    states = np.zeros((P, 4), dtype=np.uint64)
    samples = np.zeros((P, n, 2), dtype=np.int16)
    balls = np.zeros((P, n, 2))
    stats = np.zeros((P, _lib.STAT_COUNT), dtype=np.int64)
    flags = _lib.OUT_PATHS | _lib.SEED_BALLS

    def worlds2(kind, smp, st, bl):
        return lib.rrtk_ctx_plan_worlds2(None, kind, _lib.ptr(grids), 1, W, W, _lib.ptr(desc), P, n, 5.0, 2.0, _lib.ptr(smp), _lib.ptr(st),
                                         _lib.ptr(bl), flags, 8, None, None, None, _lib.ptr(stats), None, None, None, None, None, 0)

    for args, what in (((_lib.KIND_INFORMED, samples, None, None), b"h_state"),
                       ((_lib.KIND_INFORMED, None, states, balls), b"h_balls"),
                       ((_lib.KIND_STAR, None, states, None), b"RRTK_INFORMED")):
        assert worlds2(*args) == -1
        err = lib.rrtk_last_error()
        assert b"RRTK_SEED_BALLS" in err and what in err, err

    def plan2_worlds(cfg, smp, st):
        return lib.rrtk_ctx_plan2_worlds(None, _lib.ptr(cfg), _lib.ptr(grids), 1, W, W, _lib.ptr(desc), P, n, _lib.ptr(smp), _lib.ptr(st),
                                         None, flags, 8, None, None, None, None, None, _lib.ptr(stats), None, None, None, None, None, 0)

    informed = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 5.0, informed=True, r_goal=2.0)
    with_balls = informed.copy()
    with_balls["balls"] = balls.ctypes.data
    for args, what in (((informed, samples, None), b"h_state"),
                       ((with_balls, None, states), b"cfg->balls"),
                       ((_lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, 5.0), None, states), b"cfg->informed")):
        assert plan2_worlds(*args) == -1
        err = lib.rrtk_last_error()
        assert b"RRTK_SEED_BALLS" in err and what in err, err
