"""Bodies with a heading, host side: stencil checks, the run encoding, the heading-layer rule, the car stencils' covering
guarantee, the layered specification (oracle/body_oracle.c) and the scipy reference of the layer grids.  No GPU."""
import math

import numpy as np
import pytest

from oracle import body_oracle as B
from oracle import rewire_oracle as R
from rrtplanner_b200 import RRTDubins, RRTStar, RRTStarDubins
from rrtplanner_b200.body import DM_TWO_PI, body_layer, body_runs, car_body


def _decode(runs, layer_runs, S):
    k = (S - 1) // 2
    out = np.zeros((layer_runs.shape[0] - 1, S, S), dtype=bool)
    for l in range(out.shape[0]):
        for dx, lo, hi in runs[layer_runs[l]:layer_runs[l + 1]]:
            assert not out[l, dx + k, lo + k: hi + k + 1].any()          # runs do not overlap
            out[l, dx + k, lo + k: hi + k + 1] = True
    return out


def _centred(rng, L, S, p):
    s = rng.random((L, S, S)) < p
    s[:, (S - 1) // 2, (S - 1) // 2] = True
    return s


@pytest.mark.parametrize("bad, what", [
    (np.ones((1, 4, 4), bool), "odd"),
    (np.ones((1, 257, 257), bool), "S <= 255"),
    (np.ones((257, 1, 1), bool), "1 .. 256"),
    (np.ones((0, 1, 1), bool), "1 .. 256"),
    (np.ones((1, 3, 5), bool), "odd S x S"),
    (np.ones((3, 3), bool), "shape"),
])
def test_bad_stencils_are_rejected(bad, what):
    with pytest.raises(ValueError, match=what):
        body_runs(bad)


def test_a_layer_without_its_centre_is_rejected():
    s = np.ones((4, 5, 5), bool)
    s[2, 2, 2] = False
    with pytest.raises(ValueError, match="stencil 2 does not contain the centre"):
        body_runs(s)


def test_body_argument_checks_need_no_gpu():
    og = np.zeros((32, 32))
    car = car_body(3, 1, 1, 8)
    with pytest.raises(ValueError, match="either body or robot_radius"):
        RRTDubins(og, 10, 2.0, body=car, robot_radius=2.0)
    with pytest.raises(ValueError, match="either body or robot_radius"):
        RRTStarDubins(og, 10, 5.0, 2.0, body=car, robot_radius=2.0)
    with pytest.raises(ValueError, match="odd"):
        RRTDubins(og, 10, 2.0, body=np.ones((8, 4, 4), bool))
    with pytest.raises(TypeError):
        RRTStar(og, 10, 5.0, body=car)                   # a body needs a heading: only the Dubins planners take one


@pytest.mark.parametrize("L, S, p", [(1, 1, 0.5), (3, 7, 0.5), (16, 23, 0.3), (2, 255, 0.02), (5, 9, 0.9)])
def test_runs_round_trip(L, S, p):
    rng = np.random.default_rng(S * 31 + L)
    s = _centred(rng, L, S, p)
    runs, layer_runs = body_runs(s)
    assert runs.dtype == np.int32 and layer_runs.dtype == np.int32 and layer_runs[0] == 0
    assert np.array_equal(_decode(runs, layer_runs, S), s)
    k = (S - 1) // 2
    assert (np.abs(runs) <= k).all() and (runs[:, 1] <= runs[:, 2]).all()
    if S >= 7 and p <= 0.5:                               # rows with several runs occur
        rows = {(l, int(dx)) for l in range(L) for dx in runs[layer_runs[l]:layer_runs[l + 1], 0]}
        assert len(rows) < runs.shape[0]


def test_runs_are_maximal():
    s = np.zeros((1, 7, 7), bool)
    s[0, 3] = [1, 1, 0, 1, 1, 1, 0]
    s[0, 0] = [0, 0, 0, 0, 0, 0, 1]
    runs, layer_runs = body_runs(s)
    assert runs.tolist() == [[-3, 3, 3], [0, -3, -2], [0, 0, 2]]
    assert layer_runs.tolist() == [0, 3]


@pytest.mark.parametrize("nh", [1, 2, 7, 16, 64, 255])
def test_vertex_headings_map_to_themselves(nh):
    h = np.arange(nh)
    theta = h * (DM_TWO_PI / nh)                           # the angle dubins_track gives heading h
    assert np.array_equal(body_layer(theta, nh), h)
    assert np.array_equal(body_layer(theta + DM_TWO_PI, nh), h)
    assert np.array_equal(body_layer(theta - 2 * DM_TWO_PI, nh), h)


def test_body_layer_wraps_negative_and_large_angles():
    assert body_layer(-DM_TWO_PI / 16, 16) == 15
    assert body_layer(-0.01, 16) == 0
    assert body_layer(DM_TWO_PI - 0.01, 16) == 0
    assert body_layer(3 * DM_TWO_PI + DM_TWO_PI / 4, 8) == 2
    assert body_layer(-5 * DM_TWO_PI - DM_TWO_PI / 4, 8) == 6
    assert body_layer(123.0, 1) == 0


def test_body_layer_at_half_bin_boundaries():
    for L in (2, 4, 16, 64, 256):
        scale = float(L) / DM_TWO_PI
        for k in range(-2 * L, 2 * L):
            t = (k + 0.5) / scale
            x = t * scale                                 # the product the rule rounds
            want = (math.floor(x + 0.5)) % L
            assert body_layer(t, L) == want
            if x == k + 0.5:                              # exactly on the boundary: rounds up to the next layer
                assert want == (k + 1) % L
        # just below / above the boundary
        t = 0.5 / scale
        assert body_layer(t * (1 - 1e-12), L) == 0
        assert body_layer(t * (1 + 1e-12), L) == 1 % L


@pytest.mark.parametrize("shape", [(8, 2, 2.5), (3, 3, 1), (0, 0, 0), (10.5, 0, 4.2), (2, 6, 0.5)])
@pytest.mark.parametrize("L", [1, 4, 8, 16, 32])
@pytest.mark.parametrize("pad", [0.0, math.sqrt(0.5)])
def test_car_body_covers_every_heading_of_its_layer(shape, L, pad):
    front, rear, hw = shape
    s = car_body(front, rear, hw, L, pad)
    S = s.shape[1]
    k = (S - 1) // 2
    assert s.shape == (L, S, S) and S % 2 == 1 and s[:, k, k].all()
    d = np.arange(-k, k + 1, dtype=np.float64)
    dx, dy = np.meshgrid(d, d, indexing="ij")
    rng = np.random.default_rng(L * 7 + S)
    # every layer gets headings from the whole interval that maps to it, its ends included
    thetas = np.concatenate([rng.uniform(-3 * math.pi, 5 * math.pi, 400),
                             (np.arange(L)[:, None] + np.array([-0.5, -0.4999, 0.4999])[None]).ravel() * (DM_TWO_PI / L)])
    for th in thetas:
        c, sn = math.cos(th), math.sin(th)
        along, across = c * dx + sn * dy, -sn * dx + c * dy
        inside = (along >= -rear) & (along <= front) & (np.abs(across) <= hw)
        assert not (inside & ~s[body_layer(th, L)]).any(), th


def test_car_body_matches_the_documented_car():
    s = car_body(8, 2, 2.5, 16)
    assert s.shape == (16, 23, 23)
    assert s.sum() / 16 == pytest.approx(107, abs=1)
    xs, ys = np.nonzero(s[0])
    assert (xs.min() - 11, xs.max() - 11, ys.min() - 11, ys.max() - 11) == (-3, 9, -4, 4)


@pytest.mark.parametrize("L", [1, 5, 16])
def test_symmetric_car_gives_symmetric_stencils(L):
    s = car_body(4, 4, 1.5, L, 0.3)
    assert np.array_equal(s, s[:, ::-1, ::-1])


def test_car_body_checks_its_arguments():
    with pytest.raises(ValueError):
        car_body(-1, 2, 2)
    with pytest.raises(ValueError):
        car_body(1, 2, float("nan"))
    with pytest.raises(ValueError):
        car_body(1, 1, 1, 0)
    with pytest.raises(ValueError):
        car_body(1, 1, 1, 257)
    with pytest.raises(ValueError, match="at most 255"):
        car_body(200, 0, 1, 16)


def test_scipy_layer_oracle_equals_the_definition():
    rng = np.random.default_rng(5)
    og = (rng.random((41, 29)) < 0.08).astype(np.uint8)
    og[0, 5] = og[40, 28] = og[17, 0] = 1                   # obstacles on the border
    asym = np.zeros((7, 7), bool)
    asym[3, 3] = asym[3, 4] = asym[3, 5] = asym[5, 6] = asym[0, 1] = asym[6, 3] = True   # asymmetric, non-convex
    stencils = np.stack([asym, asym.T, car_body(2, 1, 1, 4)[1][2:9, 2:9] | np.eye(7, dtype=bool)])
    got = B.layers_scipy(og, stencils)
    want = B.layers_direct(og, stencils)
    assert np.array_equal(got, want)
    flipped = B.layers_direct(og, stencils[:, ::-1, ::-1])
    assert not np.array_equal(got[0], flipped[0])          # the asymmetric stencil tells the two conventions apart
    assert np.array_equal(B.projection(got), got[0] & got[1] & got[2])


def _world(seed, W=48, H=40, p=0.06):
    rng = np.random.default_rng(seed)
    og = (rng.random((W, H)) < p).astype(np.uint8)
    return rng, og


@pytest.mark.parametrize("star, rewire", [(False, False), (True, False), (True, True)])
def test_layered_specification_with_one_point_layer_is_the_plain_one(star, rewire):
    rng, og = _world(3)
    og[10, 10] = og[30, 20] = 0
    n = 150
    smp = np.stack([rng.integers(0, 48, n), rng.integers(0, 40, n), rng.integers(0, 16, n)], axis=1)
    start, goal = (10, 10, 3), (30, 20, 9)
    want = R.plan("dubins", og, n, start, goal, smp, star=star, rewire=rewire, r_rewire=9.0, nh=16, rho=2.5, ds=0.7)
    got = B.plan_layers(og[None], n, start, goal, smp, star=star, rewire=rewire, r_rewire=9.0, nh=16, rho=2.5, ds=0.7)
    for key in ("pts", "head", "parent"):
        assert np.array_equal(got[key], want[key])
    for key in ("cost", "elen"):
        assert np.array_equal(got[key].view(np.int64), want[key].view(np.int64))
    assert got["stats"] == want["stats"]
    rot = np.eye(2)
    balls = rng.uniform(-0.7, 0.7, (n, 2))
    inf = dict(r_goal=6.0, rot=rot, balls=balls)
    wi = R.plan("dubins", og, n, start, goal, smp, star=True, rewire=rewire, r_rewire=9.0, nh=16, rho=2.5, ds=0.7, informed=inf)
    gi = B.plan_layers(og[None], n, start, goal, smp, star=True, rewire=rewire, r_rewire=9.0, nh=16, rho=2.5, ds=0.7, informed=inf)
    assert np.array_equal(gi["ell"].view(np.int64), wi["ell"].view(np.int64)) and gi["stats"] == wi["stats"]
    assert np.array_equal(gi["cost"].view(np.int64), wi["cost"].view(np.int64))


def test_layered_specification_tests_the_layer_of_each_pose():
    """dubins_free_layers against a host walk: poses from the specification's own dubins_points, layer by body_layer."""
    rng, og = _world(11, 60, 50, 0.04)
    car = car_body(3, 1, 1, 8)
    layers = B.layers_scipy(og, car).astype(np.uint8)
    nh, rho, ds = 16, 3.0, 0.6
    q = np.stack([rng.integers(0, 60, 400), rng.integers(0, 50, 400), rng.integers(0, nh, 400),
                  rng.integers(0, 60, 400), rng.integers(0, 50, 400), rng.integers(0, nh, 400)], axis=1).astype(np.int32)
    got = B.dubins_free_layers(layers, q, nh, rho, ds)
    _, _, ln = R.dubins(q, nh, rho)
    for i in range(q.shape[0]):
        s = np.arange(int(np.floor(ln[i] / ds)) + 1) * ds
        P = R.dubins_points(q[i], nh, rho, s)
        cx, cy = np.floor(P[:, 0] + 0.5), np.floor(P[:, 1] + 0.5)
        ok = bool(((cx >= 0) & (cx < 60) & (cy >= 0) & (cy < 50)).all())
        if ok:
            lay = body_layer(P[:, 2], 8)
            ok = not layers[lay, cx.astype(int), cy.astype(int)].any()
            ok = ok and not layers[body_layer(q[i, 5] * (DM_TWO_PI / nh), 8), q[i, 3], q[i, 4]]
        assert got[i] == ok, i
    assert 0 < got.sum() < got.size
    # one layer of the point body: the plain test
    assert np.array_equal(B.dubins_free_layers(og[None], q, nh, rho, ds), R.dubins_free(og, q, nh, rho, ds))
