"""Drop-in planner classes: the API of the reference's ``rrtplanner/rrt.py`` served by librrtk.so.

Same names, constructor signatures, attributes and return structures as the reference
(``RRT`` rrt.py:50, ``RRTStandard`` :375, ``RRTStar`` :453, ``RRTStarInformed`` :562, ``r2norm`` :10,
``random_point_og`` :27).  ``plan(xstart, xgoal)`` runs entirely on the GPU (one launch of the
persistent plan kernel, csrc/plan.cu) and returns the reference's ``(nx.DiGraph, goal_vertex)``
built from the downloaded tree arrays.  There is no CPU fallback: without the CUDA extension or a
GPU every kernel-backed call raises.

Documented differences (all at points where the reference is implementation-defined, SURVEY.md
section 0):

* nearest-vertex and goal-connection ties go to the lowest vertex index (the reference uses
  unstable sorts, rrt.py:154,317); an unreachable goal with unfilled slots returns ``gv = 0`` and
  n nodes instead of reading the grid out of bounds (rrt.py:318).
* ``costfn`` other than ``None`` raises ``NotImplementedError``: an arbitrary Python callable cannot
  run on the device and there is deliberately no host fallback.
* the grid is copied to the device in ``__init__`` / ``set_og``; later in-place edits of the
  caller's array are not seen until ``set_og`` is called again (the reference holds ``og`` by
  reference, rrt.py:65).
* ``robot_radius`` (keyword-only, not in the reference): plan for a disc of that radius in cells instead of a point.  The
  planner works on the configuration-space grid, which blocks every cell within squared distance ``floor(radius^2)`` of an
  obstacle cell of ``og`` (csrc/disc.cu, rrtk_inflate_disc); a plan is by definition the same plan on that grid, so the tree
  equals what the class builds when constructed on the inflated grid with the same seed.  ``self.og`` stays the caller's
  object; ``self.free``, the device grid, ``go2goal`` and ``shortcut_path`` use the inflated grid, ``set_og`` inflates again,
  the static ``collisionfree`` is unchanged.  A start or goal inside the inflated obstacles behaves as an occupied one does:
  no growth from the root, or the goal is not found.  ``None`` (default) and radii below 1 (r2 = 0) leave the grid as it is.
* ``sample_weights`` (keyword-only, not in the reference): a (W, H) uint8 map that biases the free-space samples.  A cell's
  effective weight is its weight where the planning grid (the configuration-space grid with ``robot_radius``) leaves it free,
  else 0, and each sample is ``free[searchsorted(cumsum(effective weights), integers(0, T), side="right")]`` with T their sum,
  drawn from the planner's generator (all weights 1 gives the uniform stream exactly).  ``sample_all_free`` and the plans draw
  this way; ``set_og`` masks the weights again.  A subclass that overrides ``sample_all_free`` cannot also take weights.
* points must be integer arrays inside the grid (the reference's Numba kernel rejects float
  points with a TypingError and reads out of bounds for outside points); grids up to
  16384 x 16384, n <= 65534.
* ``within`` answers over the filled rows only.  The reference's unfilled rows hold INT64_MIN, whose
  squared distance wraps around in int64 to |x|^2, so whenever |x| < r it also returns every
  unfilled row (rrt.py:174-181); their cost is inf, so no plan depends on them.
* override points.  ``plan()`` is one fused kernel launch, so of the methods a subclass may replace
  (rrt.py:131,157,183,231) it honours the samplers -- an overridden ``sample_all_free`` (and
  ``unitball`` for RRTStarInformed) is called on the host exactly as often and in the same order as the
  reference's loop calls it, and its results become the device's sample stream -- and it refuses the
  three geometric primitives: a subclass that overrides ``near``, ``within`` or ``collisionfree`` gets a
  ``NotImplementedError`` from ``plan()`` (same reason as ``costfn``), never the stock behaviour silently.
"""
from __future__ import annotations

import copy
import math
from typing import List, Tuple

import networkx as nx
import numpy as np

from . import _lib

__all__ = ["r2norm", "random_point_og", "RRT", "RRTStandard", "RRTStar", "RRTStarInformed"]

_UNFILLED = np.iinfo(np.int64).min      # the reference's int(inf) sentinel (rrt.py:81,408)


def r2norm(x) -> float:
    """2-norm of a length-2 vector (rrt.py:10-24)."""
    return math.sqrt(x[0] * x[0] + x[1] * x[1])


def random_point_og(og: np.ndarray, rnd_gen: np.random.Generator = None) -> np.ndarray:
    """A uniformly random free cell of ``og`` (rrt.py:27-44)."""
    cells = np.argwhere(og == 0)
    draw = np.random.randint if rnd_gen is None else rnd_gen.integers
    return cells[draw(low=0, high=cells.shape[0])]


def _as_point(x, shape, name) -> np.ndarray:
    a = np.asarray(x)
    if a.shape != (2,):
        raise ValueError(f"{name} must be a length-2 array")
    if not np.issubdtype(a.dtype, np.integer):
        if not np.all(a == np.floor(a)):
            raise TypeError(f"{name} must hold integer grid coordinates")   # reference: Numba TypingError
    a = a.astype(np.int64)
    if not (0 <= a[0] < shape[0] and 0 <= a[1] < shape[1]):
        raise ValueError(f"{name}={a.tolist()} lies outside the {shape} grid")
    return a


class RRT(object):
    """Base class: state + device-backed primitives (rrt.py:50-369)."""

    _KIND = None

    def __init__(self, og: np.ndarray, n: int, costfn: callable = None, pbar: bool = True, seed: int = 0, *, robot_radius=None,
                 sample_weights=None):
        if costfn is not None:
            raise NotImplementedError(
                "custom cost functions are Python callables and cannot run on the device; "
                "rrtplanner_b200 has no CPU fallback (pass costfn=None)")
        self.pbar = pbar
        self.n = n
        if sample_weights is not None:
            if self._sampler_overridden():
                raise TypeError(f"{type(self).__name__} overrides sample_all_free, so sample_weights would be ambiguous: "
                                "weight the overriding sampler itself, or drop the override")
            sample_weights = _lib.sample_weights_array(sample_weights, np.shape(og))
        self.sample_weights = sample_weights
        self.robot_radius = robot_radius
        if robot_radius is not None and np.ndim(robot_radius) != 0:
            raise ValueError("robot_radius must be a number (cells)")
        self._r2 = None if robot_radius is None else int(_lib.disc_r2(robot_radius))
        self._ctx = None
        self._cspace = self._inflate(og)
        self.free = self._free_cells(og)
        self._weigh()
        self.og = og

        def costfn(vcosts, points, v, x):
            return vcosts[v] + r2norm(points[v] - x)

        self.cost = costfn
        self.not_a_point = [np.inf, np.inf]
        self.not_a_dist = np.inf
        self.rand_gen = np.random.default_rng(seed)
        self._dirty = True

    # ---- device state ------------------------------------------------------------------------
    def _device(self) -> "_lib.Context":
        if self._ctx is None:
            self._ctx = _lib.Context()
            self._dirty = True
        if self._dirty:
            og = np.asarray(self.og)
            if og.ndim != 2:
                raise ValueError("og must be a 2-D occupancy grid")
            self._ctx.set_grids(((og != 0).astype(np.uint8) if self._cspace is None else self._cspace)[None])
            self._dirty = False
        return self._ctx

    def _inflate(self, og):
        """The configuration-space grid of ``og`` for ``robot_radius`` as (W, H) uint8 of 0 / 1, or None when nothing is
        inflated (no radius, or r2 = 0).  Inflated on the device, downloaded packed (1 bit per cell)."""
        if not self._r2:
            return None
        og = np.asarray(og)
        if og.ndim != 2:
            raise ValueError("og must be a 2-D occupancy grid")
        if self._ctx is None:
            self._ctx = _lib.Context()
            self._dirty = True
        bits = self._ctx.inflate_disc((og != 0).astype(np.uint8)[None], [0], [self._r2])
        return _lib.unpack_grids_host(bits, *og.shape)[0]

    def _free_cells(self, og) -> np.ndarray:
        """Free cells of the planning grid of ``og``, row-major (rrt.py:64)."""
        return np.argwhere((og if self._cspace is None else self._cspace) == 0)

    def _weigh(self):
        """Cumulative effective weights over ``self.free`` (None without weights).  Cells the grid blocks or that weigh 0 never
        end a searchsorted step, so the cumulative sum over the free cells picks the same cells as the one over the whole grid."""
        self._wcum = None
        if self.sample_weights is None:
            return
        cum = np.cumsum(self.sample_weights[self.free[:, 0], self.free[:, 1]].astype(np.int64))
        if not cum.size or cum[-1] == 0:
            raise ValueError("sample_weights put no weight on a free cell of the planning grid: nothing to sample")
        self._wcum = cum

    def _draw_free(self, rng: np.random.Generator, count: int) -> np.ndarray:
        """``count`` free cells from ``rng`` as the stock sampler draws them: uniform (integers(0, nfree)), or weighted."""
        if self._wcum is None:
            return self.free[rng.integers(0, self.free.shape[0], size=count)]
        return self.free[np.searchsorted(self._wcum, rng.integers(0, int(self._wcum[-1]), size=count), side="right")]

    # ---- graph helpers (host, rrt.py:87-129) -----------------------------------------------------
    def route2gv(self, T: nx.DiGraph, gv) -> List[int]:
        """Vertices from the root to ``gv`` (rrt.py:87-107)."""
        return nx.shortest_path(T, source=0, target=gv, weight="dist")

    def vertices_as_ndarray(self, T: nx.DiGraph, path: list) -> np.ndarray:
        """(M-1, 2, 2) array of the path's segments (rrt.py:109-129)."""
        segs = [[T.nodes[a]["pt"], T.nodes[b]["pt"]] for a, b in zip(path[:-1], path[1:])]
        return np.array(segs)

    def shortcut_path(self, T: nx.DiGraph, path: list) -> List[int]:
        """The vertices of ``path`` (a ``route2gv`` list) kept by a greedy line-of-sight shortcut on the planner's current grid:
        from each kept vertex, the farthest later one that ``collisionfree`` sees from it is kept next (walked from the
        earlier vertex to the later one).  ``vertices_as_ndarray(T, shortcut_path(T, path))`` is the pruned polyline.
        Runs on the device (rrtk_ctx_shortcut); paths up to 4096 vertices."""
        path = list(path)
        if not path:
            return []
        pts = np.array([np.asarray(T.nodes[v]["pt"]) for v in path])
        shape = np.asarray(self.og).shape
        if pts.min() < 0 or pts[:, 0].max() >= shape[0] or pts[:, 1].max() >= shape[1]:
            raise ValueError(f"a path vertex lies outside the {shape} grid")
        res = self._device().shortcut(pts.astype(np.int16)[None], [len(path)])
        return [path[int(k)] for k in res["keep"][0, : int(res["len"][0])]]

    # ---- primitives (static in the reference: rrt.py:131,157,183) --------------------------------
    @staticmethod
    def near(points: np.ndarray, x: np.ndarray) -> np.ndarray:
        """All row indices ordered by distance to ``x`` (rrt.py:131-155); equal distances keep
        index order.  Rows holding the reference's unfilled sentinel sort last."""
        points = np.asarray(points)
        x = np.asarray(x)
        ctx = _lib.shared_context()
        if np.issubdtype(points.dtype, np.integer) and np.issubdtype(x.dtype, np.integer):
            hole = points[:, 0] == _UNFILLED
            if hole.any() or np.abs(points[~hole]).max(initial=0) > 2 ** 30:
                live = np.flatnonzero(~hole)
                order = live[ctx.near_order(points[live].astype(np.int32), x)] if live.size else live
                return np.concatenate([order, np.flatnonzero(hole)]).astype(np.int64)
        return ctx.near_order(points, x).astype(np.int64)

    @staticmethod
    def within(points: np.ndarray, x: np.ndarray, r: float) -> np.ndarray:
        """Ascending indices of the rows strictly closer than ``r`` to ``x`` (rrt.py:157-181)."""
        points = np.asarray(points)
        x = np.asarray(x)
        ctx = _lib.shared_context()
        if np.issubdtype(points.dtype, np.integer) and np.issubdtype(x.dtype, np.integer):
            hole = points[:, 0] == _UNFILLED
            if hole.any():
                live = np.flatnonzero(~hole)
                out, ln = ctx.within(points[live].astype(np.int32), x, r)
                return live[out[0, : ln[0]]].astype(np.int64)
        out, ln = ctx.within(points, x, r)
        return out[0, : ln[0]].astype(np.int64)

    # grid the shared context holds for the static collisionfree(): (occupancy as bool, copy)
    _cf_cache = None

    @staticmethod
    def collisionfree(og, a, b) -> bool:
        """True iff the integer line walk a -> b meets no non-zero cell (rrt.py:183-229).

        The reference's function is stateless; a caller looping it over one grid (as go2goal's callers
        do) must not pay an upload and a packing kernel per segment, so the shared context keeps the
        last grid.  The cache is validated by content (one host compare of the occupancy, ~15 us for
        512 x 512), not by identity: in-place edits of ``og`` between calls are seen."""
        og = np.asarray(og)
        a = _as_point(a, og.shape, "a")
        b = _as_point(b, og.shape, "b")
        ctx = _lib.shared_context()
        occ = og != 0
        cached = RRT._cf_cache
        if cached is None or cached[0] is not ctx or cached[1].shape != occ.shape or not np.array_equal(cached[1], occ):
            ctx.set_grids(occ.astype(np.uint8)[None])
            RRT._cf_cache = (ctx, occ)
        return bool(ctx.collision(np.concatenate([a, b])[None])[0])

    def sample_all_free(self):
        """A uniformly random free cell (rrt.py:231-240); with ``sample_weights`` a free cell drawn by weight."""
        if self._wcum is not None:
            return self.free[np.searchsorted(self._wcum, self.rand_gen.integers(0, int(self._wcum[-1])), side="right")]
        return self.free[self.rand_gen.choice(self.free.shape[0])]

    def plan(self, xstart: np.ndarray, xgoal: np.ndarray):
        """Raises on the base class, like the reference (rrt.py:242-259)."""
        raise NotImplementedError("This method is not implemented in the base class.")

    def set_og(self, og_new: np.ndarray):
        """New occupancy grid: refresh free space (rrt.py:261-272) and the device copy."""
        if self.sample_weights is not None and self.sample_weights.shape != np.shape(og_new):
            raise ValueError(f"sample_weights has shape {self.sample_weights.shape}, the new grid {np.shape(og_new)}")
        self.og = og_new
        self._cspace = self._inflate(og_new)
        self.free = self._free_cells(og_new)
        self._weigh()
        self._dirty = True

    def set_n(self, n: int):
        """New number of attempted samples (rrt.py:274-282)."""
        self.n = n

    # ---- goal connection as a stand-alone call (rrt.py:284-332) -----------------------------------
    def go2goal(self, vcosts, points, xgoal, j, children, parents):
        """Connect the goal to the cheapest vertex that sees it.  Inside ``plan()`` this step is
        fused into the plan kernel; this method keeps the reference's signature for callers that
        drive the pieces by hand.  Candidate costs are ordered on the host, the visibility tests
        run on the device (K1) in batches of 256 candidates in (cost, index) order."""
        xgoal = _as_point(xgoal, np.asarray(self.og).shape, "xgoal")
        filled = np.arange(j)
        gap = points[:j] - xgoal
        togo = vcosts[:j] + np.sqrt((gap[:, 0] * gap[:, 0] + gap[:, 1] * gap[:, 1]).astype(np.float64))
        order = filled[np.lexsort((filled, togo))]
        ctx = self._device()
        for lo in range(0, order.size, 256):
            chunk = order[lo: lo + 256]
            segs = np.concatenate([points[chunk], np.broadcast_to(xgoal, (chunk.size, 2))], axis=1)
            ok = ctx.collision(segs)
            if ok.any():
                idx = int(chunk[int(np.argmax(ok))])
                vgoal = j
                points = np.concatenate((points, xgoal[np.newaxis, :]), axis=0)
                vcosts = np.concatenate((vcosts, [togo[idx]]), axis=0)
                points[vgoal] = xgoal
                vcosts[vgoal] = togo[idx]
                children[idx].append(vgoal)
                parents[vgoal] = idx
                return vgoal, children, parents, points, vcosts
        return np.int64(0), children, parents, points, vcosts

    def build_graph(self, vgoal, points, parents, vcosts):
        """nx.DiGraph of the tree with the reference's node / edge attributes (rrt.py:334-369):
        node i for every row (attr ``pt``), the goal node inserted first; one edge per entry of
        ``parents`` with ``dist`` (segment length) and ``cost`` (cost-to-come of the child)."""
        T = nx.DiGraph()
        T.add_node(vgoal, pt=points[vgoal])
        T.add_nodes_from((i, {"pt": points[i]}) for i in range(points.shape[0]))
        # the edges in the order of ``parents`` (insertion order), their lengths in one pass: sqrt of an exact integer sum, the
        # same double math.sqrt gives edge by edge
        children = [c for c, p in parents.items() if p is not None]
        if children:
            pars = [parents[c] for c in children]
            steps = points[np.asarray(children, dtype=np.int64)] - points[np.asarray(pars, dtype=np.int64)]
            dists = np.sqrt((steps[:, 0] * steps[:, 0] + steps[:, 1] * steps[:, 1]).astype(np.float64)).tolist()
            T.add_edges_from((p, c, {"dist": d, "cost": vcosts[c]}) for p, c, d in zip(pars, children, dists))
        return T

    # ---- shared plan() machinery ----------------------------------------------------------------------
    def _check_hooks(self):
        """The reference's override points (rrt.py:131,157,183): the fused plan kernel cannot call back
        into Python, so a subclass that replaces one of the geometric primitives is refused."""
        cls = type(self)
        for name in ("near", "within", "collisionfree"):
            if getattr(cls, name) is not getattr(RRT, name):
                raise NotImplementedError(
                    f"{cls.__name__} overrides RRT.{name}: a Python callable cannot run on the device and "
                    "rrtplanner_b200 has no CPU fallback (plan() uses the stock primitive inside one kernel)")

    def _sampler_overridden(self) -> bool:
        return type(self).sample_all_free is not RRT.sample_all_free

    def _as_samples(self, rows) -> np.ndarray:
        a = np.asarray(rows)
        shape = np.asarray(self.og).shape
        if a.ndim != 2 or a.shape[1] != 2 or not np.issubdtype(a.dtype, np.integer) and not np.all(a == np.floor(a)):
            raise TypeError("sample_all_free() must return integer grid points of shape (2,)")
        a = a.astype(np.int64)
        if a.size and (a.min() < 0 or a[:, 0].max() >= shape[0] or a[:, 1].max() >= shape[1]):
            raise ValueError("sample_all_free() returned a point outside the grid")
        return a

    def _draw_samples(self, count: int) -> np.ndarray:
        """``count`` successive sample_all_free() results.  Stock sampler: numpy's bounded-integer stream
        for size=count equals count scalar choice() calls and leaves the generator in the same state.
        Overridden sampler (the reference's injection point, rrt.py:231): called ``count`` times, as the
        reference's loop does (rrt.py:420,501)."""
        if type(self).sample_all_free is not RRT.sample_all_free and self._sampler_overridden():
            return self._as_samples([np.asarray(self.sample_all_free()) for _ in range(count)])
        return self._draw_free(self.rand_gen, count)

    def _desc(self, xstart, xgoal, rot=None):
        d = np.zeros(1, dtype=_lib.PLAN_DESC)
        d["start_x"], d["start_y"] = int(xstart[0]), int(xstart[1])
        d["goal_x"], d["goal_y"] = int(xgoal[0]), int(xgoal[1])
        if rot is not None:
            d["rot"][0] = np.asarray(rot, dtype=np.float64).reshape(4)
        return d

    def _finish(self, pts, cost, parent, stats):
        """Device rows -> the reference's arrays after go2goal (rrt.py:320-323) -> graph."""
        n = self.n
        j, vgoal, found = int(stats[0]), int(stats[1]), bool(stats[2])
        rows = n + 1 if found else n
        points = np.full((rows, 2), _UNFILLED, dtype=np.int64)
        vcosts = np.full((rows,), np.inf)
        top = j + 1 if found else j
        points[:top] = pts[:top]
        vcosts[:top] = cost[:top]
        if found and j < n:
            points[n] = pts[j]
            vcosts[n] = cost[j]
        parents = {0: None}
        parents.update(zip(range(1, j), np.asarray(parent[1:j]).astype(np.int64)))
        if found:
            parents[vgoal] = np.int64(parent[j])
        gv = vgoal if found else np.int64(0)
        self.last_stats = dict(zip(_lib.STAT_NAMES, (int(s) for s in stats)))
        return self.build_graph(gv, points, parents, vcosts), gv

    def _tick(self):
        if self.pbar:
            from tqdm import tqdm
            bar = tqdm(total=self.n)
            bar.update(self.n)       # one launch covers all n iterations
            bar.close()


class RRTStandard(RRT):
    """Standard RRT (rrt.py:375-447)."""

    _KIND = _lib.KIND_STANDARD

    def __init__(self, og: np.ndarray, n: int, costfn: callable = None, pbar=True, seed: int = 0, *, robot_radius=None,
                 sample_weights=None):
        super().__init__(og, n, costfn=costfn, pbar=pbar, seed=seed, robot_radius=robot_radius, sample_weights=sample_weights)

    def plan(self, xstart: np.ndarray, xgoal: np.ndarray) -> Tuple[nx.DiGraph, int]:
        self._check_hooks()
        shape = np.asarray(self.og).shape
        xstart, xgoal = _as_point(xstart, shape, "xstart"), _as_point(xgoal, shape, "xgoal")
        ctx = self._device()
        samples = self._draw_samples(self.n).astype(np.int16)[None]
        pts, cost, parent, stats, _ = ctx.plan(self._KIND, self._desc(xstart, xgoal), self.n, samples=samples)
        self._tick()
        return self._finish(pts[0], cost[0], parent[0], stats[0])


class RRTStar(RRT):
    """RRT* (rrt.py:453-556).

    ``rewire`` (not in the reference, keyword-only, default = the reference's behaviour):
    ``"reference"`` keeps the reference's rewire block, whose predicate ``cost(vn -> xnew) < vcosts[vn]``
    (rrt.py:532-536) can never hold, i.e. no rewiring; ``"rrtstar"`` rewires with the textbook predicate
    ``vcosts[vnew] + |xnew - xn| < vcosts[vn]`` and keeps the costs of the rewired subtree consistent
    (kernel K8, csrc/plan_rewire.cu; specification oracle/rewire_oracle.c -- there is no reference
    behaviour to match for this mode)."""

    _KIND = _lib.KIND_STAR

    def __init__(self, og: np.ndarray, n: int, r_rewire: float, costfn: callable = None, pbar=True, seed: int = 0, *,
                 rewire: str = "reference", robot_radius=None, sample_weights=None):
        super().__init__(og, n, costfn=costfn, pbar=pbar, seed=seed, robot_radius=robot_radius, sample_weights=sample_weights)
        self.r_rewire = r_rewire
        if rewire not in ("reference", "rrtstar"):
            raise ValueError("rewire must be 'reference' or 'rrtstar'")
        self.rewire = rewire

    def plan(self, xstart: np.ndarray, xgoal: np.ndarray):
        self._check_hooks()
        shape = np.asarray(self.og).shape
        xstart, xgoal = _as_point(xstart, shape, "xstart"), _as_point(xgoal, shape, "xgoal")
        ctx = self._device()
        samples = self._draw_samples(self.n).astype(np.int16)[None]
        if self.rewire == "rrtstar":
            cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, self.r_rewire)
            pts, _, cost, _, parent, stats = ctx.plan2(cfg, self._desc(xstart, xgoal), self.n, samples=samples)
            self._tick()
            T, gv = self._finish(pts[0], cost[0], parent[0], stats[0])
            self.last_stats = dict(zip(_lib.STAT2_NAMES, (int(v) for v in stats[0])))
            return T, gv
        pts, cost, parent, stats, _ = ctx.plan(self._KIND, self._desc(xstart, xgoal), self.n,
                                               r_rewire=self.r_rewire, samples=samples)
        self._tick()
        return self._finish(pts[0], cost[0], parent[0], stats[0])


class RRTStarInformed(RRT):
    """Informed RRT* (rrt.py:562-758).  ``sample_weights`` weight the free-space phase only; the ellipse phase is the reference's.

    ``rewire`` (keyword-only, not in the reference) as for :class:`RRTStar`: ``"reference"`` keeps the reference's rewire
    block, which never fires; ``"rrtstar"`` runs the loop with the rewire that fires (kernel K8 with the informed sampling
    rule; specification oracle/rewire_oracle.c:orc2_plan_informed).  With the rewire off that kernel reproduces the
    reference's informed trees bit for bit (tests/test_gpu_rewire.py), so the sampling rule itself is pinned."""

    _KIND = _lib.KIND_INFORMED

    def __init__(self, og: np.ndarray, n: int, r_rewire: float, r_goal: float, costfn: callable = None,
                 pbar: bool = True, seed: int = 0, *, rewire: str = "reference", robot_radius=None, sample_weights=None):
        super().__init__(og, n, costfn=costfn, pbar=pbar, seed=seed, robot_radius=robot_radius, sample_weights=sample_weights)
        self.r_rewire = r_rewire
        self.r_goal = r_goal
        self.ellipses = {}
        if rewire not in ("reference", "rrtstar"):
            raise ValueError("rewire must be 'reference' or 'rrtstar'")
        self.rewire = rewire               # as for RRTStar: "rrtstar" = the rewire that fires (kernel K8), not in the reference

    def _launch(self, ctx, desc, samples, balls=None):
        """One launch of the plan (balls=None: the probe that stops at the first solution vertex):
        (pts, cost, parent, stats, ell, iteration of the first solution vertex)."""
        if self.rewire == "rrtstar":
            cfg = _lib.plan2_cfg(_lib.MODEL_EUCLID, True, True, self.r_rewire, informed=True, r_goal=self.r_goal)
            pts, _, cost, _, parent, stats, ell = ctx.plan2(cfg, desc, self.n, samples=samples, balls=balls)
            self.last_stats = dict(zip(_lib.STAT2_NAMES, (int(v) for v in stats[0])))
            return pts, cost, parent, stats, ell, int(stats[0][_lib.STAT2_NAMES.index("first_solution_iter")])
        if balls is None:
            pts, cost, parent, stats, ell = ctx.plan(self._KIND, desc, self.n, r_rewire=self.r_rewire, r_goal=self.r_goal, samples=samples)
        else:
            pts, cost, parent, stats, ell = ctx.plan(self._KIND, desc, self.n, r_rewire=self.r_rewire, r_goal=self.r_goal, samples=samples,
                                                     balls=balls)
        return pts, cost, parent, stats, ell, int(stats[0][5])

    # ---- sampler pieces, host-side mirrors of rrt.py:579-651 (the device evaluates the same
    #      formulas inside the plan kernel; these serve callers and the ellipse records) ---------
    def unitball(self):
        """Uniform point of the unit disc from two uniform draws, radius first (rrt.py:579-587)."""
        u = self.rand_gen.uniform(0, 1)
        ang = 2 * np.pi * self.rand_gen.uniform(0, 1)
        return np.array([np.sqrt(u) * np.cos(ang), np.sqrt(u) * np.sin(ang)])

    def rotation_to_world_frame(self, xstart, xgoal):
        """Rotation aligning the x axis with start -> goal via the SVD construction of rrt.py:601-613
        (same numpy calls, so the LAPACK sign convention is inherited)."""
        span = xgoal - xstart
        axis = np.atleast_2d(span / np.linalg.norm(span))
        outer = np.outer(axis, np.atleast_2d([1, 0]))
        try:
            U, _, V = np.linalg.svd(outer)
        except np.linalg.LinAlgError:
            U, _, V = np.linalg.svd(outer, full_matrices=False)
        return U @ np.diag([np.linalg.det(U), np.linalg.det(V)]) @ V.T

    def get_ellipse_xform(self, xstart, xgoal, cmax):
        """Unit disc -> ellipse with foci start/goal and path-length budget cmax (rrt.py:615-625)."""
        rot = self.rotation_to_world_frame(xstart, xgoal)
        gap = xstart - xgoal
        semi_major = cmax / 2
        semi_minor = np.sqrt(abs(cmax * cmax - np.dot(gap.T, gap))) / 2
        return np.dot(rot, np.diag([semi_major, semi_minor]))

    def sample_ellipse(self, xstart, xgoal, c, clamp=True):
        """One integer sample of the informed ellipse (rrt.py:589-599)."""
        centre = (xstart + xgoal) / 2
        x, y = tuple(np.dot(self.get_ellipse_xform(xstart, xgoal, c), self.unitball()) + centre)
        if clamp:
            x = int(max(0, min(self.og.shape[0] - 1, x)))
            y = int(max(0, min(self.og.shape[1] - 1, y)))
        return np.array((x, y))

    @staticmethod
    def least_cost(vcosts, vsoln):
        """Cheapest solution vertex, first one on ties (rrt.py:627-633)."""
        k = 0 if len(vsoln) == 1 else int(np.argmin(vcosts[vsoln]))
        return vsoln[k], vcosts[vsoln[k]]

    @staticmethod
    def rad2deg(a):
        return a * 180 / np.pi

    def get_ellipse_for_plt(self, xstart, xgoal, cmax) -> Tuple[np.ndarray, float, float, float]:
        """(centre, major axis, minor axis, angle in degrees) for plotting (rrt.py:639-651)."""
        centre = (xgoal + xstart) / 2
        xform = self.get_ellipse_xform(xstart, xgoal, cmax)
        ex = np.dot(xform, np.array([1, 0]))
        ey = np.dot(xform, np.array([0, 1]))
        return centre, 2 * np.linalg.norm(ex), 2 * np.linalg.norm(ey), self.rad2deg(np.arctan2(ex[1], ex[0]))

    def plan(self, xstart: np.ndarray, xgoal: np.ndarray):
        """The reference interleaves free-space draws and ellipse draws on ONE generator
        (rrt.py:240,582-583), and where the switch happens depends on the tree.  So the plan runs
        as: (1) a probe launch on a copy of the generator's free-space stream that stops at the
        first solution vertex; (2) the real generator is advanced by exactly the draws the
        reference would have consumed up to there, the ellipse-phase uniforms are drawn from it,
        and the full plan is launched (the first phase replays identically).

        With an overridden ``sample_all_free`` the generator cannot be copied, so the free-space phase
        is drawn call by call instead: a solution vertex can only appear at an iteration whose sample
        lies within ``r_goal`` of the goal (rrt.py:744), so the sampler is called until such a sample
        turns up, a probe launch on the stream so far says whether that iteration produced the first
        solution, and drawing continues if it did not -- the sampler is called exactly as often as
        the reference's loop would call it.  ``unitball`` is always called on the host, once per
        ellipse-phase iteration, overridden or not."""
        self._check_hooks()
        shape = np.asarray(self.og).shape
        xstart, xgoal = _as_point(xstart, shape, "xstart"), _as_point(xgoal, shape, "xgoal")
        ctx = self._device()
        n = self.n
        desc = self._desc(xstart, xgoal)
        if self._sampler_overridden():
            samples = np.zeros((1, n, 2), dtype=np.int16)
            first, drawn = -1, 0
            while drawn < n and first < 0:
                x = self._as_samples([np.asarray(self.sample_all_free())])[0]
                samples[0, drawn] = x
                drawn += 1
                if r2norm(x - xgoal) < self.r_goal:
                    # the probe sees iterations 0 .. drawn-1 only (later rows repeat the last sample: duplicates)
                    samples[0, drawn:] = x
                    f = self._launch(ctx, desc, samples)[5]
                    if 0 <= f < drawn:
                        first = f
        else:
            probe_gen = copy.deepcopy(self.rand_gen)
            samples = self._draw_free(probe_gen, n).astype(np.int16)[None]
            first = self._launch(ctx, desc, samples)[5]
            # advance the real generator by exactly the free-space draws the reference consumes
            self._draw_free(self.rand_gen, n if first < 0 else first + 1)
        balls = np.zeros((1, n, 2))
        if first >= 0:
            rot = self.rotation_to_world_frame(xstart, xgoal)    # LinAlgError if xstart == xgoal, as the reference
            desc = self._desc(xstart, xgoal, rot)
            for i in range(first + 1, n):
                balls[0, i] = self.unitball()
        pts, cost, parent, stats, ell, _ = self._launch(ctx, desc, samples, balls)
        for jj in np.flatnonzero(~np.isnan(ell[0])):
            self.ellipses[int(jj)] = self.get_ellipse_for_plt(xstart, xgoal, ell[0][jj])   # rrt.py:701
        self._tick()
        T, gv = self._finish(pts[0], cost[0], parent[0], stats[0])
        if self.rewire == "rrtstar":
            self.last_stats = dict(zip(_lib.STAT2_NAMES, (int(v) for v in stats[0])))
        return T, gv
