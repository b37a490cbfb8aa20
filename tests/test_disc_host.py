"""Configuration space of a disc robot, host side: the radius -> r2 rule, argument checks that need no GPU, and the two scipy
oracles of the contract (dilation with the disc structure, thresholded exact EDT) against each other.  The device kernel
(csrc/disc.cu) is checked against these oracles in tests/test_gpu_disc.py."""
import math

import numpy as np
import pytest
from scipy import ndimage

from rrtplanner_b200 import RRTStandard, RRTStar, _lib, batch, build as build_mod

INT32_MAX = 2 ** 31 - 1


def disc_structure(r2: int) -> np.ndarray:
    R = math.isqrt(r2)
    i = np.arange(-R, R + 1)
    return (i[:, None] ** 2 + i[None, :] ** 2) <= r2


def cspace_dilation(og, r2: int) -> np.ndarray:
    """binary_dilation(og != 0, disc, border_value=0) as uint8; the disc is cut at the grid's diagonal, which no pair of cells
    inside the grid exceeds."""
    W, H = og.shape
    r2 = min(int(r2), (W - 1) ** 2 + (H - 1) ** 2)
    return ndimage.binary_dilation(og != 0, structure=disc_structure(r2), border_value=0).astype(np.uint8)


def sq_dist_to_obstacle(og) -> np.ndarray:
    """Exact integer squared distance of every cell to the nearest obstacle cell of the grid (int64; -1 without obstacles)."""
    og = np.asarray(og) != 0
    if not og.any():
        return np.full(og.shape, -1, dtype=np.int64)
    _, ind = ndimage.distance_transform_edt(~og, return_indices=True)
    X, Y = np.indices(og.shape)
    return (X - ind[0]).astype(np.int64) ** 2 + (Y - ind[1]).astype(np.int64) ** 2


def cspace_edt(og, r2: int, d2=None) -> np.ndarray:
    """The same grid from the distance transform: EDT^2 <= r2 (an obstacle-free world stays free)."""
    d2 = sq_dist_to_obstacle(og) if d2 is None else d2
    return ((d2 >= 0) & (d2 <= int(r2))).astype(np.uint8)


def blobs(W, H, seed, density=900):
    rng = np.random.default_rng(seed)
    og = np.zeros((W, H), dtype=np.uint8)
    X, Y = np.indices((W, H))
    for _ in range(max(2, W * H // density)):
        cx, cy, r = rng.integers(0, W), rng.integers(0, H), rng.integers(0, max(2, min(W, H) // 8) + 1)
        og[(X - cx) ** 2 + (Y - cy) ** 2 <= r * r] = 1
    og[rng.random((W, H)) < 0.01] = 1
    return og


@pytest.mark.parametrize("radius, r2", [(0, 0), (0.0, 0), (1, 1), (2, 4), (3, 9), (7, 49), (100, 10000), (math.sqrt(2), 2),
                                        (1.9999999, 3), (0.5, 0), (0.9999, 0), (3.9999, 15), (46340, 2147395600),
                                        (46341, INT32_MAX), (1e10, INT32_MAX), (1e200, INT32_MAX), (np.finfo(np.float64).max, INT32_MAX)])
def test_r2_rule(radius, r2):
    got = _lib.disc_r2(radius)
    assert got.dtype == np.int32 and int(got) == r2


def test_r2_rule_arrays_and_squared_distances():
    radii = np.array([0, 0.5, 1, math.sqrt(2), 1.5, 2, 3.9999, 7, 33])
    assert _lib.disc_r2(radii).tolist() == [0, 0, 1, 2, 2, 4, 15, 49, 1089]
    # d^2 <= r2 is d^2 <= radius^2 for every integer d^2
    for rho in radii:
        r2 = int(_lib.disc_r2(rho))
        for d2 in range(0, 1200):
            assert (d2 <= r2) == (d2 <= rho * rho)


@pytest.mark.parametrize("bad", [-1, -1e-300, float("nan"), float("inf"), -float("inf")])
def test_bad_radius_raises(bad):
    with pytest.raises(ValueError):
        _lib.disc_r2(bad)
    with pytest.raises(ValueError):
        _lib.disc_r2([1.0, bad])
    og = np.zeros((16, 16))
    with pytest.raises(ValueError):
        RRTStandard(og, 10, pbar=False, robot_radius=bad)
    with pytest.raises(ValueError):
        RRTStar(og, 10, 5.0, pbar=False, robot_radius=bad)
    with pytest.raises(ValueError):
        batch.plan_batch("star", og, 10, [[1, 1]], [[9, 9]], r_rewire=5.0, seeds=[0], robot_radius=bad)


def test_radius_shape_errors():
    og = np.zeros((16, 16))
    with pytest.raises(ValueError):
        RRTStandard(og, 10, pbar=False, robot_radius=[1.0, 2.0])
    with pytest.raises(ValueError):
        batch.plan_batch("star", og, 10, [[1, 1], [2, 2]], [[9, 9], [8, 8]], r_rewire=5.0, seeds=[0, 1], robot_radius=[1.0, 2.0, 3.0])


@pytest.fixture(scope="module")
def lib():
    build_mod.build()
    return _lib.lib()


def test_abi_checks_need_no_gpu(lib):
    assert lib.rrtk_inflate_disc_scratch_bytes(2, 512, 512) == 2 * 512 * 512 * 2
    assert lib.rrtk_inflate_disc_scratch_bytes(1, 43, 100) == 43 * 128 * 2     # rows padded to whole 32-cell words
    assert lib.rrtk_inflate_disc_scratch_bytes(0, 43, 100) == 0
    assert lib.rrtk_inflate_disc_scratch_bytes(1, 0, 100) == 0
    # nothing to write: no device work, no pointer needed
    assert lib.rrtk_inflate_disc(None, 1, 64, 64, None, None, 0, None, None, None) == 0
    assert lib.rrtk_inflate_disc(None, 1, 64, 64, None, None, 1, None, None, None) == -1
    assert b"null" in lib.rrtk_last_error()
    assert lib.rrtk_inflate_disc(None, -1, 64, 64, None, None, 1, None, None, None) == -1
    assert lib.rrtk_inflate_disc(None, 1, 64, 64, None, None, -1, None, None, None) == -1
    assert lib.rrtk_inflate_disc(None, 0, 64, 64, None, None, 1, None, None, None) == -1
    assert lib.rrtk_inflate_disc(None, 1, 0, 64, None, None, 1, None, None, None) == -1
    assert lib.rrtk_inflate_disc(None, 1, 40000, 64, None, None, 1, None, None, None) == -1
    buf = np.zeros(1024, dtype=np.uint32)
    p = _lib.ptr(buf)
    assert lib.rrtk_inflate_disc(p, 1, 32, 32, p, p, 1, p, p, None) == -1           # aliasing
    assert b"alias" in lib.rrtk_last_error()
    assert lib.rrtk_ctx_inflate_disc(None, None, 1, 32, 32, None, None, 1, None) == -1


@pytest.mark.parametrize("shape", [(17, 23), (40, 33), (64, 64), (31, 70)])
def test_scipy_oracles_agree(shape):
    rng = np.random.default_rng(sum(shape))
    W, H = shape
    worlds = [blobs(W, H, 1), (rng.random(shape) < 0.02).astype(np.uint8), (rng.random(shape) < 0.3).astype(np.uint8)]
    single = np.zeros(shape, dtype=np.uint8)
    single[W // 2, H // 3] = 1
    border = np.zeros(shape, dtype=np.uint8)
    border[0, 3] = border[W - 1, H - 5] = border[4, 0] = border[W - 3, H - 1] = 1
    worlds += [single, border, np.ones(shape, dtype=np.uint8)]
    diag = (W - 1) ** 2 + (H - 1) ** 2
    for og in worlds:
        d2 = sq_dist_to_obstacle(og)
        for rho in (0, 0.5, 1, math.sqrt(2), 1.5, 2, 3.9999, 7, 12.5, math.sqrt(diag) + 1):
            r2 = int(_lib.disc_r2(rho))
            want = cspace_dilation(og, r2)
            assert np.array_equal(want, cspace_edt(og, r2, d2)), (shape, rho)
    # the exact disc: one obstacle gives the lattice points of the disc around it
    for rho in (1, math.sqrt(2), 3.9999, 7):
        r2 = int(_lib.disc_r2(rho))
        got = cspace_edt(single, r2)
        X, Y = np.indices(shape)
        assert np.array_equal(got, ((X - W // 2) ** 2 + (Y - H // 3) ** 2 <= r2).astype(np.uint8))
    # an obstacle-free world stays free at every radius, and r2 = 0 is the grid itself
    assert not cspace_edt(np.zeros(shape), INT32_MAX).any()
    assert not cspace_dilation(np.zeros(shape), 50).any()
    assert np.array_equal(cspace_edt(worlds[2], 0), worlds[2])
