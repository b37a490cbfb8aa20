"""Path shortcutting, the parts that need no GPU: the specification (oracle/shortcut_oracle.py) on hand-made grids, and the
argument checks of rrtk_shortcut_paths, rrtk_ctx_shortcut, RRTK_OUT_SHORTCUT and batch.shortcut_paths (all raised before
any device work).  tests/test_gpu_shortcut.py runs the same hand-made cases through the kernel."""
import math

import numpy as np
import pytest

from oracle import rrt_oracle as O, shortcut_oracle as S
from rrtplanner_b200 import _lib, batch, build as build_mod


@pytest.fixture(scope="module")
def lib():
    build_mod.build()
    return _lib.lib()


def corridor():
    """10 x 10 walls with an L-shaped corridor: column x = 1 for y = 1..8, then row y = 8 for x = 1..8."""
    og = np.ones((10, 10), dtype=np.uint8)
    og[1, 1:9] = 0
    og[1:9, 8] = 0
    return og


def direction_grid():
    """3 x 3, one obstacle at (1, 0): the walk (0, 0) -> (2, 1) passes (1, 1), the walk (2, 1) -> (0, 0) passes (1, 0)."""
    og = np.zeros((3, 3), dtype=np.uint8)
    og[1, 0] = 1
    return og


def hand_cases():
    """(name, og, points, kept indices) of the hand-made cases."""
    rng = np.random.default_rng(3)
    walk = np.clip(np.cumsum(rng.integers(-3, 4, size=(40, 2)), axis=0) + 60, 0, 119)
    blocked = np.zeros((5, 1), dtype=np.uint8)
    blocked[1, 0] = blocked[3, 0] = 1
    return [
        ("open_world", np.zeros((120, 130), dtype=np.uint8), walk, [0, 39]),
        ("l_corridor", corridor(), [[1, 1], [1, 4], [1, 8], [4, 8], [8, 8]], [0, 2, 4]),
        ("walk_direction_forward", direction_grid(), [[0, 0], [0, 1], [2, 1]], [0, 2]),
        ("walk_direction_reversed", direction_grid(), [[2, 1], [0, 1], [0, 0]], [0, 1, 2]),
        ("blocked_steps_advance_by_one", blocked, [[0, 0], [2, 0], [4, 0]], [0, 1, 2]),
        ("duplicate_points", np.zeros((8, 8), dtype=np.uint8), [[2, 2], [2, 2], [5, 6], [5, 6]], [0, 3]),
    ]


def test_walk_direction_case_is_asymmetric():
    og = direction_grid()
    assert O.collisionfree(og, (0, 0), (2, 1)) and not O.collisionfree(og, (2, 1), (0, 0))


@pytest.mark.parametrize("case", hand_cases(), ids=lambda c: c[0])
def test_hand_made_cases(case):
    _, og, pts, want = case
    pts = np.asarray(pts)
    assert S.shortcut_indices(og, pts) == want
    cap = len(pts) + 3
    xy = np.full((1, cap, 2), -32768, dtype=np.int16)
    xy[0, : len(pts)] = pts
    ids = np.full((1, cap), -1, dtype=np.int32)
    ids[0, : len(pts)] = np.arange(len(pts)) * 7
    got = S.shortcut_records(og, xy, [len(pts)], path=ids)
    t = len(want)
    assert int(got["len"][0]) == t and got["keep"][0, :t].tolist() == want and (got["keep"][0, t:] == -1).all()
    assert np.array_equal(got["xy"][0, :t], pts[want]) and (got["xy"][0, t:] == -32768).all()
    assert got["path"][0, :t].tolist() == [7 * k for k in want] and (got["path"][0, t:] == -1).all()
    kept = pts[want]
    total = 0.0
    for a, b in zip(kept[:-1], kept[1:]):
        total += math.sqrt(float(((b - a) ** 2).sum()))
    assert got["cost"][0] == total


def test_open_world_collapses_to_start_and_goal():
    pts = hand_cases()[0][2]
    got = S.shortcut_records(np.zeros((120, 130), dtype=np.uint8), pts[None], [len(pts)])
    assert got["xy"][0, :2].tolist() == [pts[0].tolist(), pts[-1].tolist()]
    assert got["cost"][0] == math.sqrt(float(((pts[-1] - pts[0]) ** 2).sum()))


def test_rows_outside_one_to_cap_are_untouched():
    og = np.zeros((16, 16), dtype=np.uint8)
    cap = 4
    xy = np.arange(5 * cap * 2, dtype=np.int16).reshape(5, cap, 2) % 16
    ln = np.array([0, 1, 2, cap + 1, -3], dtype=np.int32)
    got = S.shortcut_records(og, xy, ln)
    for p in (0, 3, 4):
        assert np.array_equal(got["xy"][p], xy[p]) and got["len"][p] == ln[p]
        assert (got["keep"][p] == -1).all() and np.isnan(got["cost"][p])
    assert got["len"][1] == 1 and got["keep"][1].tolist() == [0, -1, -1, -1] and got["cost"][1] == 0.0
    assert np.array_equal(got["xy"][1, 0], xy[1, 0]) and (got["xy"][1, 1:] == -32768).all()
    assert got["len"][2] == 2 and got["keep"][2].tolist() == [0, 1, -1, -1]
    d = (xy[2, 1].astype(np.int64) - xy[2, 0]) ** 2
    assert got["cost"][2] == math.sqrt(float(d.sum()))


def test_shortcut_paths_rejects_bad_arguments(lib):
    buf = np.zeros(64, dtype=np.int64)
    p = _lib.ptr(buf)
    good = [p, 32, 32, None, 2, 8, p, p, None, None, None, None]
    for k in (0, 6, 7):                                    # d_bits, d_xy, d_len
        args = list(good)
        args[k] = None
        assert lib.rrtk_shortcut_paths(*args) == -1, k
        assert b"rrtk_shortcut_paths" in lib.rrtk_last_error()
    for k, v, rc in ((4, -1, -1), (5, 0, -1), (5, -4, -1), (5, _lib.SHORTCUT_MAX_CAP + 1, -2), (1, 0, -1), (2, 16385, -1)):
        args = list(good)
        args[k] = v
        assert lib.rrtk_shortcut_paths(*args) == rc, (k, v)
    assert lib.rrtk_ctx_shortcut(None, None, 1, 8, p, p, None, None, None) == -1
    assert b"rrtk_ctx_shortcut" in lib.rrtk_last_error()


def test_shortcut_flag_misuse_is_rejected_without_a_gpu(lib):
    P, n, W = 2, 16, 32
    grids = np.zeros((1, W, W), dtype=np.uint8)
    desc = batch.make_desc([0, 0], [[1, 1], [2, 2]], [[20, 20], [21, 21]])
    states = np.zeros((P, 4), dtype=np.uint64)
    stats = np.zeros((P, _lib.STAT_COUNT), dtype=np.int64)
    path, xy = np.zeros((P, 8), dtype=np.int32), np.zeros((P, 8, 2), dtype=np.int16)
    ln, cost = np.zeros(P, dtype=np.int32), np.zeros(P)

    def worlds2(flags, cap):
        return lib.rrtk_ctx_plan_worlds2(None, _lib.KIND_STAR, _lib.ptr(grids), 1, W, W, _lib.ptr(desc), P, n, 5.0, 0.0, None,
                                         _lib.ptr(states), None, flags, cap, None, None, None, _lib.ptr(stats), None, _lib.ptr(path),
                                         _lib.ptr(xy), _lib.ptr(ln), _lib.ptr(cost), 0)

    assert worlds2(_lib.OUT_SHORTCUT, 8) == -1
    assert b"RRTK_OUT_SHORTCUT needs RRTK_OUT_PATHS" in lib.rrtk_last_error()
    assert worlds2(_lib.OUT_SHORTCUT | _lib.OUT_TREES, 8) == -1
    assert worlds2(_lib.OUT_SHORTCUT | _lib.OUT_PATHS, _lib.SHORTCUT_MAX_CAP + 1) == -2
    assert b"RRTK_SHORTCUT_MAX_CAP" in lib.rrtk_last_error()


def test_host_form_checks_worlds_and_points_before_the_device():
    ogs = np.zeros((2, 20, 12), dtype=np.uint8)
    xy = np.zeros((3, 4, 2), dtype=np.int16)
    ln = np.array([2, 4, 1])
    with pytest.raises(ValueError, match="world index"):
        batch.shortcut_paths(ogs, xy, ln, world_ids=[0, 2, 1])
    with pytest.raises(ValueError, match="world index"):
        batch.shortcut_paths(ogs, xy, ln, world_ids=[0, -1, 1])
    for p, k, pt in ((1, 3, (20, 0)), (0, 1, (0, 12)), (2, 0, (-1, 3))):
        bad = xy.copy()
        bad[p, k] = pt
        with pytest.raises(ValueError, match="outside"):
            batch.shortcut_paths(ogs, bad, ln)
    with pytest.raises(ValueError, match="shape"):
        batch.shortcut_paths(ogs, xy[0], ln)
