"""Dubins primitive and Dubins-vehicle planners, served by librrtk.so (kernel K8, csrc/plan_rewire.cu, csrc/dubins.cuh).

The reference lists a "Dubins Primitive Module", a "Dubins Vehicle RRT Planner" and a "Dubins Vehicle RRT(star)
Planner" as features (README.md:12,18-19 of rland93/rrtplanner) but its tree contains none of them, so there is no
reference signature, behaviour or test to mirror.  The classes here follow the conventions of the reference's
existing planners (rrt.py:375-556): same constructor order ``(og, n[, r_rewire], ..., costfn=None, pbar=True,
seed=0)``, ``plan(xstart, xgoal) -> (nx.DiGraph, goal_vertex)``, same graph attributes (``pt``, ``dist``, ``cost``),
plus what a vehicle with a heading needs.  The specification they are tested against bit for bit is
oracle/rewire_oracle.c (parity UNPINNED: it is this project's own definition).

Model: a configuration is ``(x, y, h)`` -- an integer grid cell and a heading index ``h`` in ``[0, nheadings)``,
heading angle ``h * 2 pi / nheadings`` measured from the +x axis towards +y.  Edges are shortest Dubins paths
(turning radius ``rho`` cells) checked against the grid at points every ``ds`` cells of arc length.  ``robot_radius``
(keyword-only) plans for a disc-shaped vehicle on the configuration-space grid, as for the planners of rrt.py; that footprint
does not depend on the heading.  ``body`` (keyword-only, e.g. ``body.car_body(...)``) plans for a vehicle whose footprint turns
with it: one stencil per heading layer, one configuration-space grid per layer (csrc/body.cu), and every sampled pose of an
edge tests the layer of its own angle (``body.body_layer``), the edge's end cell the layer of the end heading.  Samples are
drawn from the projection, the cells some heading leaves free.  Nearest and rewire-radius queries are Euclidean on ``(x, y)``
exactly as in the reference's planners.
"""
from __future__ import annotations

from typing import Tuple

import networkx as nx
import numpy as np

from . import _lib
from .body import body_runs, inflate_body_host
from .rrt import RRT, _UNFILLED, _as_point

__all__ = ["dubins_path", "dubins_length", "dubins_collisionfree", "dubins_points", "RRTDubins", "RRTStarDubins", "DUBINS_WORDS"]

DUBINS_WORDS = _lib.DUBINS_WORDS


def _as_config(q, shape, nheadings, name) -> np.ndarray:
    a = np.asarray(q)
    if a.shape != (3,):
        raise ValueError(f"{name} must be (x, y, heading index)")
    xy = _as_point(a[:2], shape, name) if shape is not None else a[:2].astype(np.int64)
    h = int(a[2])
    if h != a[2] or not (0 <= h < nheadings):
        raise ValueError(f"{name}: heading index {a[2]} outside [0, {nheadings})")
    return np.array([xy[0], xy[1], h], dtype=np.int64)


def _queries(q0, q1):
    q0 = np.asarray(q0, dtype=np.int64).reshape(-1, 3)
    q1 = np.asarray(q1, dtype=np.int64).reshape(-1, 3)
    return np.concatenate([q0, q1], axis=1).astype(np.int32)


def dubins_path(q0, q1, rho: float, nheadings: int = 16):
    """Shortest Dubins path(s) from configuration(s) q0 to q1: ``(word, (t, p, q), length)`` with the segment
    lengths in units of rho and ``word`` an index into ``DUBINS_WORDS``.  Arrays in, arrays out (one row per pair)."""
    word, tpq, ln = _lib.shared_context().dubins_paths(_queries(q0, q1), nheadings, rho)
    if np.asarray(q0).ndim == 1:
        return int(word[0]), tpq[0], float(ln[0])
    return word, tpq, ln


def dubins_length(q0, q1, rho: float, nheadings: int = 16):
    return dubins_path(q0, q1, rho, nheadings)[2]


def dubins_collisionfree(og, q0, q1, rho: float, nheadings: int = 16, ds: float = 1.0, body=None):
    """True iff the shortest Dubins path q0 -> q1 stays on free cells of ``og`` (points every ``ds`` cells, rounded to
    the nearest cell, end cell included; leaving the grid counts as a collision).  ``body``: (nlayers, S, S) stencils of a body
    with a heading (module ``body``); each pose then tests the heading layer of its own angle, the end cell that of q1's heading."""
    og = np.asarray(og)
    ctx = _lib.shared_context()
    if body is not None:
        runs, layer_runs = body_runs(body)
        ctx.set_body_grids((og != 0).astype(np.uint8)[None], runs, layer_runs)
        RRT._cf_cache = None                 # the shared context no longer holds the grid RRT.collisionfree cached
    else:
        ctx.set_grids((og != 0).astype(np.uint8)[None])
    free = ctx.dubins_collision(_queries(q0, q1), nheadings, rho, ds)
    return bool(free[0]) if np.asarray(q0).ndim == 1 else free


def dubins_points(q0, q1, rho: float, nheadings: int = 16, ds: float = 1.0) -> np.ndarray:
    """Poses ``(x, y, theta)`` of the shortest path q0 -> q1 every ``ds`` cells of arc length (one pair)."""
    q = _queries(q0, q1)
    ctx = _lib.shared_context()
    _, _, ln = ctx.dubins_paths(q, nheadings, rho)
    cap = int(np.floor(ln[0] / ds)) + 1
    xyth, cnt = ctx.dubins_sample(q, nheadings, rho, ds, cap)
    return xyth[0, : int(cnt[0])]


class RRTDubins(RRT):
    """Dubins-vehicle RRT ("Dubins Vehicle RRT Planner", README.md:18): the RRTStandard loop (rrt.py:418-437) with
    Dubins edges.  ``plan(xstart, xgoal)`` takes configurations ``(x, y, heading index)``."""

    _STAR = False

    def __init__(self, og: np.ndarray, n: int, rho: float, nheadings: int = 16, ds: float = 1.0, costfn: callable = None,
                 pbar: bool = True, seed: int = 0, *, robot_radius=None, body=None, sample_weights=None):
        if body is not None and robot_radius is not None:
            raise ValueError("pass either body or robot_radius, not both (a disc is a body whose stencils are all the same disc)")
        self.body = None if body is None else np.asarray(body) != 0
        self._body_runs = None if body is None else body_runs(body)
        super().__init__(og, n, costfn=costfn, pbar=pbar, seed=seed, robot_radius=robot_radius, sample_weights=sample_weights)
        if not (0 < rho <= 16384 and 0.05 <= ds <= 16384):
            raise ValueError("need 0 < rho <= 16384 and 0.05 <= ds <= 16384 (cells)")
        if not (1 <= int(nheadings) <= 255):
            raise ValueError("nheadings must be in [1, 255]")
        self.rho, self.nheadings, self.ds = float(rho), int(nheadings), float(ds)
        self.r_rewire = 0.0
        self.rewire = False

    def _free_cells(self, og) -> np.ndarray:
        """With a body: free cells of its projection of ``og`` (the cells some heading leaves free), computed on the device."""
        if self.body is None:
            return super()._free_cells(og)
        og = np.asarray(og)
        if og.ndim != 2:
            raise ValueError("og must be a 2-D occupancy grid")
        _, proj = inflate_body_host(og, *self._body_runs)
        return np.argwhere(proj[0] == 0)

    def _device(self) -> "_lib.Context":
        if self.body is None:
            return super()._device()
        if self._ctx is None:
            self._ctx = _lib.Context()
            self._dirty = True
        if self._dirty:
            og = np.asarray(self.og)
            if og.ndim != 2:
                raise ValueError("og must be a 2-D occupancy grid")
            self._ctx.set_body_grids((og != 0).astype(np.uint8)[None], *self._body_runs)
            self._dirty = False
        return self._ctx

    def sample_all_free(self):
        """A uniformly random free configuration: cell as RRT.sample_all_free (rrt.py:231-240, weighted with ``sample_weights``),
        then a heading."""
        cell = RRT.sample_all_free(self)
        return np.array([cell[0], cell[1], self.rand_gen.integers(0, self.nheadings)])

    def collisionfree(self, og, a, b) -> bool:  # noqa: D102 -- configurations instead of points
        return dubins_collisionfree(og, a, b, self.rho, self.nheadings, self.ds, body=self.body)

    def _sampler_overridden(self) -> bool:
        return type(self).sample_all_free is not RRTDubins.sample_all_free

    def _draw_configs(self, count: int) -> Tuple[np.ndarray, np.ndarray]:
        """``count`` cells, then ``count`` headings, from the planner's generator; a subclass's own
        ``sample_all_free`` is called ``count`` times instead (one configuration per iteration)."""
        if self._sampler_overridden():
            rows = np.asarray([np.asarray(self.sample_all_free()) for _ in range(count)])
            if rows.ndim != 2 or rows.shape[1] != 3:
                raise TypeError("sample_all_free() must return a configuration (x, y, heading index)")
            heads = rows[:, 2].astype(np.int64)
            if heads.size and (heads.min() < 0 or heads.max() >= self.nheadings):
                raise ValueError("sample_all_free() returned a heading index outside [0, nheadings)")
            return self._as_samples(rows[:, :2]), heads
        cells = RRT._draw_samples(self, count)
        heads = self.rand_gen.integers(0, self.nheadings, size=count)
        return cells, heads

    def plan(self, xstart: np.ndarray, xgoal: np.ndarray) -> Tuple[nx.DiGraph, int]:
        shape = np.asarray(self.og).shape
        xstart = _as_config(xstart, shape, self.nheadings, "xstart")
        xgoal = _as_config(xgoal, shape, self.nheadings, "xgoal")
        ctx = self._device()
        cells, heads = self._draw_configs(self.n)
        desc = self._desc(xstart, xgoal)
        desc["reserved"][0, 0], desc["reserved"][0, 1] = xstart[2], xgoal[2]
        cfg = _lib.plan2_cfg(_lib.MODEL_DUBINS, self._STAR, self.rewire, self.r_rewire, self.nheadings, self.rho, self.ds)
        pts, head, cost, elen, parent, stats = ctx.plan2(cfg, desc, self.n, samples=cells.astype(np.int16)[None],
                                                         heads=heads.astype(np.uint8)[None])
        self._tick()
        return self._finish_dubins(pts[0], head[0], cost[0], elen[0], parent[0], stats[0])

    def _finish_dubins(self, pts, head, cost, elen, parent, stats):
        """Same row / node layout as the reference's planners after go2goal (rrt.py:320-323, 334-369); nodes carry
        ``pt`` and ``heading``, edges ``dist`` (Dubins length), ``cost`` (cost-to-come of the child)."""
        n = self.n
        j, vgoal, found = int(stats[0]), int(stats[1]), bool(stats[2])
        rows = n + 1 if found else n
        points = np.full((rows, 2), _UNFILLED, dtype=np.int64)
        headings = np.full((rows,), -1, dtype=np.int64)
        vcosts = np.full((rows,), np.inf)
        top = j + 1 if found else j
        points[:top], headings[:top], vcosts[:top] = pts[:top], head[:top], cost[:top]
        if found and j < n:
            points[n], headings[n], vcosts[n] = pts[j], head[j], cost[j]
        gv = vgoal if found else np.int64(0)
        T = nx.DiGraph()
        T.add_node(gv, pt=points[gv], heading=int(headings[gv]))
        for i in range(rows):
            T.add_node(i, pt=points[i], heading=int(headings[i]))
        for v in range(1, top):
            T.add_edge(np.int64(parent[v]), v, dist=float(elen[v]), cost=vcosts[v])
        self.last_stats = dict(zip(_lib.STAT2_NAMES, (int(s) for s in stats)))
        return T, gv

    def path_points(self, T: nx.DiGraph, path: list) -> np.ndarray:
        """Poses (x, y, theta) along ``path`` (vertex ids, e.g. from ``route2gv``), every ``ds`` cells per edge."""
        out = []
        for a, b in zip(path[:-1], path[1:]):
            qa = [*T.nodes[a]["pt"], T.nodes[a]["heading"]]
            qb = [*T.nodes[b]["pt"], T.nodes[b]["heading"]]
            out.append(dubins_points(qa, qb, self.rho, self.nheadings, self.ds))
        return np.concatenate(out, axis=0) if out else np.zeros((0, 3))


class RRTStarDubins(RRTDubins):
    """Dubins-vehicle RRT* ("Dubins Vehicle RRT(star) Planner", README.md:19): the RRTStar loop (rrt.py:498-548) with
    Dubins edges; ``rewire=True`` (default) rewires with ``vcosts[vnew] + len(vnew -> vn) < vcosts[vn]`` and keeps
    subtree costs consistent, ``rewire=False`` stops after choose-parent (what the reference's RRTStar computes)."""

    _STAR = True

    def __init__(self, og: np.ndarray, n: int, r_rewire: float, rho: float, nheadings: int = 16, ds: float = 1.0,
                 costfn: callable = None, pbar: bool = True, seed: int = 0, *, rewire: bool = True, robot_radius=None, body=None,
                 sample_weights=None):
        super().__init__(og, n, rho, nheadings=nheadings, ds=ds, costfn=costfn, pbar=pbar, seed=seed, robot_radius=robot_radius,
                         body=body, sample_weights=sample_weights)
        self.r_rewire = r_rewire
        self.rewire = bool(rewire)
