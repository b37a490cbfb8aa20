"""ctypes binding of librrtk.so (C ABI in include/rrtk.h).

There is no CPU fallback: if the library has not been built, or no CUDA device is visible when a
kernel is needed, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RRTK_LIB") or os.path.join(_HERE, "librrtk.so")   # RRTK_LIB: experiment builds

KIND_STANDARD, KIND_STAR, KIND_INFORMED = 0, 1, 2
STAT_NAMES = ("j", "vgoal", "found", "checks", "cells", "first_solution_iter", "ellipse_iters",
              "nn_pairs", "ring_members", "accepted", "reserved0", "reserved1")
STAT_COUNT = len(STAT_NAMES)

MODEL_EUCLID, MODEL_DUBINS = 0, 1
# flags of rrtk_ctx_plan_worlds2 / rrtk_ctx_plan2_worlds
IN_BITS, OUT_TREES, OUT_PATHS, SEED_BALLS, OUT_SHORTCUT, SEED_WEIGHTS = 1, 2, 4, 8, 16, 32
SHORTCUT_MAX_CAP = 4096            # RRTK_SHORTCUT_MAX_CAP: longest path row rrtk_shortcut_paths takes
STAT2_NAMES = ("j", "vgoal", "found", "checks", "accepted", "rewires", "propagated", "ring_members", "len_evals", "overflow",
               "ell_iters", "first_solution_iter")
DUBINS_WORDS = ("LSL", "RSR", "LSR", "RSL", "RLR", "LRL")
# numpy mirror of rrtk_plan2_cfg (80 bytes)
PLAN2_CFG = np.dtype([("model", "<i4"), ("star", "<i4"), ("rewire", "<i4"), ("nheadings", "<i4"), ("r_rewire", "<f8"),
                      ("rho", "<f8"), ("ds", "<f8"), ("dubins_table", "<u8"), ("table_radius", "<i4"), ("informed", "<i4"),
                      ("r_goal", "<f8"), ("balls", "<u8"), ("ell_c", "<u8")], align=True)
assert PLAN2_CFG.itemsize == 80


def plan2_cfg(model, star, rewire, r_rewire=0.0, nheadings=1, rho=1.0, ds=1.0, informed=False, r_goal=0.0) -> np.ndarray:
    """``informed``: the informed sampling rule; the ``balls`` / ``ell_c`` pointers are filled in by the caller that owns the
    arrays (Context.plan2 / plan2_worlds: host arrays; DeviceBatch2: device tensors)."""
    c = np.zeros(1, dtype=PLAN2_CFG)
    c["model"], c["star"], c["rewire"], c["nheadings"] = int(model), int(bool(star)), int(bool(rewire)), int(nheadings)
    c["r_rewire"], c["rho"], c["ds"] = float(r_rewire), float(rho), float(ds)
    c["informed"], c["r_goal"] = int(bool(informed)), float(r_goal)
    return c


# numpy mirror of rrtk_plan_desc (64 bytes)
PLAN_DESC = np.dtype([("world", "<i4"), ("start_x", "<i4"), ("start_y", "<i4"), ("goal_x", "<i4"),
                      ("goal_y", "<i4"), ("reserved", "<i4", (3,)), ("rot", "<f8", (4,))], align=True)
assert PLAN_DESC.itemsize == 64


class RRTKError(RuntimeError):
    pass


_vp, _i, _i64, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_size_t

# name -> (restype, argtypes); every symbol include/rrtk.h declares is listed (tests check this)
SIGNATURES = {
    "rrtk_version": (_i, []),
    "rrtk_last_error": (C.c_char_p, []),
    "rrtk_device_count": (_i, []),
    "rrtk_set_device": (_i, [_i]),
    "rrtk_device_info": (_i, [_vp, _vp]),
    "rrtk_peak_l2_read": (_i, [_vp, _sz, _i, _vp, _vp, _vp]),
    "rrtk_peak_smem_read": (_i, [_i, _i, _vp, _vp, _vp]),
    "rrtk_grid_words": (_sz, [_i, _i]),
    "rrtk_pack_grid": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rrtk_unpack_grid": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rrtk_inflate_grid": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "rrtk_free_rows": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rrtk_inflate_disc_scratch_bytes": (_sz, [_i, _i, _i]),
    "rrtk_inflate_disc": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "rrtk_inflate_body": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "rrtk_gen_worlds": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rrtk_collision_segments": (_i, [_vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "rrtk_clearance_field": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rrtk_collision_segments_cf": (_i, [_vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "rrtk_clearance_field_dir": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "rrtk_collision_segments_cfd": (_i, [_vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "rrtk_clearance_field_dir16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "rrtk_collision_segments_cfd16": (_i, [_vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "rrtk_nearest_batch": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "rrtk_nearest_batch_f64": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "rrtk_within_batch": (_i, [_vp, _i, _vp, _vp, _i, _d, _i, _vp, _vp, _vp]),
    "rrtk_within_batch_f64": (_i, [_vp, _i, _vp, _vp, _i, _d, _i, _vp, _vp, _vp]),
    "rrtk_dist2": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "rrtk_dist_f64": (_i, [_vp, _i, _d, _d, _vp, _vp]),
    "rrtk_argsort_i64": (_i, [_vp, _i, _vp, _vp, _sz, _vp]),
    "rrtk_argsort_scratch_bytes": (_sz, [_i]),
    "rrtk_sample_streams": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "rrtk_sample_streams_carry": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "rrtk_weight_index_bytes": (_sz, [_i, _i, _i]),
    "rrtk_weight_index": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "rrtk_sample_streams_weighted": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "rrtk_ball_streams": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "rrtk_plan_batch": (_i, [_i, _vp, _i, _i, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "rrtk_plan_kernel": (C.c_char_p, [_i, _i, _i, _i, _i]),
    "rrtk_plan_footprint": (_i, [_i, _i, _i, _i, _i, _vp, _vp]),
    "rrtk_extract_paths": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "rrtk_extract_paths_xy": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rrtk_shortcut_paths": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rrtk_create": (_i, [_vp]),
    "rrtk_destroy": (_i, [_vp]),
    "rrtk_ctx_set_grids": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "rrtk_ctx_inflate": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "rrtk_ctx_inflate_disc": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rrtk_ctx_set_sample_weights": (_i, [_vp, _vp, _i, _i, _i]),
    "rrtk_ctx_set_body_grids": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rrtk_ctx_plan": (_i, [_vp, _i, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rrtk_ctx_plan_worlds": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "rrtk_ctx_plan_worlds2": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _vp, _vp, _i]),
    "rrtk_pack_grid_host": (_i, [_vp, _i, _i, _i, _vp]),
    "rrtk_seed_states": (_i, [_vp, _i, _vp]),
    "rrtk_ctx_samples": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "rrtk_ctx_collision": (_i, [_vp, _i, _vp, _i64, _vp, _vp]),
    "rrtk_ctx_shortcut": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rrtk_ctx_nearest": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "rrtk_ctx_nearest_f64": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "rrtk_ctx_within": (_i, [_vp, _vp, _i, _vp, _i, _d, _i, _vp, _vp]),
    "rrtk_ctx_within_f64": (_i, [_vp, _vp, _i, _vp, _i, _d, _i, _vp, _vp]),
    "rrtk_ctx_near_order": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "rrtk_ctx_near_order_f64": (_i, [_vp, _vp, _i, _d, _d, _vp]),
    "rrtk_dubins_table_bytes": (_sz, [_i, _i]),
    "rrtk_dubins_table_build": (_i, [_i, _i, _d, _vp, _vp]),
    "rrtk_plan2_scratch_bytes": (_sz, [_i, _i]),
    "rrtk_plan2_batch": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "rrtk_plan2_batch_layers": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "rrtk_plan2_footprint": (_i, [_i, _i, _vp, _vp]),
    "rrtk_dubins_paths": (_i, [_vp, _i64, _i, _d, _vp, _vp, _vp, _vp]),
    "rrtk_dubins_collision": (_i, [_vp, _i, _i, _vp, _vp, _i64, _i, _d, _d, _vp, _vp]),
    "rrtk_dubins_collision_layers": (_i, [_vp, _i, _i, _i, _vp, _vp, _i64, _i, _d, _d, _vp, _vp]),
    "rrtk_dubins_sample": (_i, [_vp, _i64, _i, _d, _d, _i, _vp, _vp, _vp]),
    "rrtk_ctx_plan2": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rrtk_ctx_plan2_worlds": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _i] + [_vp] * 11 + [_i]),
    "rrtk_ctx_dubins_paths": (_i, [_vp, _vp, _i64, _i, _d, _vp, _vp, _vp]),
    "rrtk_ctx_dubins_collision": (_i, [_vp, _i, _vp, _i64, _i, _d, _d, _vp]),
    "rrtk_ctx_dubins_sample": (_i, [_vp, _vp, _i64, _i, _d, _d, _i, _vp, _vp]),
}

_lib = None


def lib():
    """The loaded library; raises ImportError if it was never built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first (python -m rrtplanner_b200.build). "
                "rrtplanner_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def pack_grids_host(ogs) -> np.ndarray:
    """(nworlds, W, H) occupancy (non-zero = obstacle, rrt.py:218) -> (nworlds, rrtk_grid_words(W, H)) uint32 tiled bit grids
    on the host (rrtk_pack_grid_host): the form RRTK_IN_BITS callers keep their worlds in."""
    og = np.ascontiguousarray((np.asarray(ogs) != 0).astype(np.uint8))
    if og.ndim == 2:
        og = og[None]
    nw, W, H = og.shape
    bits = np.empty((nw, int(lib().rrtk_grid_words(W, H))), dtype=np.uint32)
    check(lib().rrtk_pack_grid_host(ptr(og), nw, W, H, ptr(bits)), "rrtk_pack_grid_host")
    return bits


INT32_MAX = 2 ** 31 - 1


def disc_r2(radius):
    """Squared-distance threshold of a disc robot of radius ``radius`` cells (scalar or array): ``floor(radius * radius)`` in
    float64, clamped to INT32_MAX, as int32.  A cell is blocked iff its squared distance d^2 (an integer) to an obstacle cell is
    <= this, which equals d^2 <= radius^2.  Raises ValueError for a negative, NaN or infinite radius."""
    r = np.asarray(radius, dtype=np.float64)
    if not np.isfinite(r).all() or (r < 0).any():
        raise ValueError("robot_radius must be a finite number >= 0 (cells)")
    with np.errstate(over="ignore"):
        return np.minimum(np.floor(r * r), INT32_MAX).astype(np.int32)


def unpack_grids_host(bits, W: int, H: int) -> np.ndarray:
    """Inverse of pack_grids_host: (nworlds, rrtk_grid_words(W, H)) uint32 tiled bit grids -> (nworlds, W, H) uint8 of 0 / 1."""
    TX, TY = (W + 31) // 32, (H + 31) // 32
    b = np.ascontiguousarray(bits, dtype="<u4").reshape(-1, TX, TY, 32)                 # [world, tx, ty, x & 31]
    cells = np.unpackbits(b.view(np.uint8).reshape(*b.shape, 4), axis=-1, bitorder="little")   # [..., y & 31]
    return cells.transpose(0, 1, 3, 2, 4).reshape(b.shape[0], TX * 32, TY * 32)[:, :W, :H].copy()


def sample_weights_array(weights, shape) -> np.ndarray:
    """A weight map argument as a C-contiguous uint8 array of ``shape`` ((W, H) or (nworlds, W, H)); a single (W, H) map is
    broadcast to every world.  Anything but uint8 is rejected (floats, other integer types, values outside [0, 255]): weights are
    never quantised silently."""
    w = np.asarray(weights)
    if w.dtype != np.uint8:
        raise TypeError(f"sample_weights must be a uint8 array (got {w.dtype}); weights are whole numbers in [0, 255]")
    shape = tuple(int(v) for v in shape)
    if w.shape != shape:
        if len(shape) == 3 and w.shape == shape[1:]:
            w = np.broadcast_to(w, shape)
        else:
            raise ValueError(f"sample_weights has shape {w.shape}, the grids need {shape}" + (f" or {shape[1:]}" if len(shape) == 3 else ""))
    return np.ascontiguousarray(w)


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    msg = lib().rrtk_last_error().decode("utf-8", "replace")
    text = f"{what}: {msg}" if what else msg
    if rc == -1:
        raise ValueError(text)
    if rc == -2:
        raise MemoryError(text)
    raise RRTKError(text)


def ptr(a):
    """void* of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def pcg64_state_words(rng: np.random.Generator) -> np.ndarray:
    """{state_hi, state_lo, inc_hi, inc_lo} of a fresh PCG64 generator, for rrtk_sample_streams."""
    st = rng.bit_generator.state
    if st["bit_generator"] != "PCG64" or st["has_uint32"]:
        raise ValueError("device sampling needs a PCG64 generator with no buffered 32-bit half")
    s, inc = st["state"]["state"], st["state"]["inc"]
    m = (1 << 64) - 1
    return np.array([s >> 64, s & m, inc >> 64, inc & m], dtype=np.uint64)


class Context:
    """Owner of one rrtk_ctx (device scratch + stream).  Created on first use; needs a GPU."""

    def __init__(self):
        self._h = C.c_void_p()
        check(lib().rrtk_create(C.byref(self._h)), "rrtk_create")
        self.shape = None
        self.nworlds = 0
        self.nlayers = 0

    def close(self):
        if self._h:
            lib().rrtk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- grids ---------------------------------------------------------------------------------
    def set_grids(self, og_u8: np.ndarray) -> np.ndarray:
        """og_u8: (nworlds, W, H) uint8, non-zero = obstacle.  Returns nfree per world."""
        og_u8 = np.ascontiguousarray(og_u8, dtype=np.uint8)
        nw, W, H = og_u8.shape
        nfree = np.empty(nw, dtype=np.int32)
        check(lib().rrtk_ctx_set_grids(self._h, ptr(og_u8), nw, W, H, ptr(nfree)), "rrtk_ctx_set_grids")
        self.shape, self.nworlds, self.nlayers = (W, H), nw, 0
        return nfree

    def set_body_grids(self, og_u8: np.ndarray, runs, layer_runs) -> np.ndarray:
        """Worlds for a body with a heading (rrtk_ctx_set_body_grids): ``og_u8`` (nworlds, W, H), non-zero = obstacle; ``runs`` /
        ``layer_runs`` the body's stencils as ``body.body_runs`` encodes them.  The context's worlds become the projections (a
        cell is blocked iff every heading layer blocks it); ``plan2`` (Dubins) and ``dubins_collision`` test the layers until the
        next ``set_grids``.  Returns the free cells per world of the projections."""
        og_u8 = np.ascontiguousarray(og_u8, dtype=np.uint8)
        if og_u8.ndim != 3:
            raise ValueError("og_u8 must have shape (nworlds, W, H)")
        nw, W, H = og_u8.shape
        runs = np.ascontiguousarray(runs, dtype=np.int32).reshape(-1, 3)
        layer_runs = np.ascontiguousarray(layer_runs, dtype=np.int32).reshape(-1)
        nfree = np.empty(nw, dtype=np.int32)
        check(lib().rrtk_ctx_set_body_grids(self._h, ptr(og_u8), nw, W, H, ptr(runs), ptr(layer_runs), layer_runs.shape[0] - 1, ptr(nfree)),
              "rrtk_ctx_set_body_grids")
        self.shape, self.nworlds, self.nlayers = (W, H), nw, layer_runs.shape[0] - 1
        return nfree

    def set_sample_weights(self, weights, shape=None) -> None:
        """Weight maps for RRTK_SEED_WEIGHTS (rrtk_ctx_set_sample_weights): (nworlds, W, H) uint8, or None to clear them.  ``shape``
        (nworlds, W, H), if given, is the shape the maps must have (a single (W, H) map is then used for every world)."""
        if weights is None:
            check(lib().rrtk_ctx_set_sample_weights(self._h, None, 0, 0, 0), "rrtk_ctx_set_sample_weights")
            return
        w = sample_weights_array(weights, np.shape(weights) if shape is None else shape)
        if w.ndim != 3:
            raise ValueError("sample weights must have shape (nworlds, W, H)")
        check(lib().rrtk_ctx_set_sample_weights(self._h, ptr(w), *w.shape), "rrtk_ctx_set_sample_weights")

    def _weights_flag(self, sample_weights, nworlds, W, H) -> int:
        """``sample_weights`` of the pipelined calls: None (uniform), True (the maps set_sample_weights holds) or maps to set now."""
        if sample_weights is None or sample_weights is False:
            return 0
        if sample_weights is not True:
            self.set_sample_weights(sample_weights, (nworlds, W, H))
        return SEED_WEIGHTS

    # -- plans ---------------------------------------------------------------------------------
    def plan(self, kind, desc, n, r_rewire=0.0, r_goal=0.0, samples=None, states=None, balls=None, out=None):
        """``out``: optional preallocated (pts, cost, parent, stats, ell) host arrays (e.g. pinned)."""
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        if out is not None:
            pts, cost, parent, stats, ell = out
            assert pts.shape == (nplans, n + 1, 2) and pts.dtype == np.int16 and cost.shape == (nplans, n + 1)
            assert parent.dtype == np.int32 and stats.shape == (nplans, STAT_COUNT)
        else:
            pts = np.empty((nplans, n + 1, 2), dtype=np.int16)
            cost = np.empty((nplans, n + 1), dtype=np.float64)
            parent = np.empty((nplans, n + 1), dtype=np.int32)
            stats = np.empty((nplans, STAT_COUNT), dtype=np.int64)
            ell = np.empty((nplans, n + 1), dtype=np.float64) if kind == KIND_INFORMED else None
        if samples is not None:
            samples = np.ascontiguousarray(samples, dtype=np.int16)
            assert samples.shape == (nplans, n, 2), samples.shape
        if states is not None:
            states = np.ascontiguousarray(states, dtype=np.uint64)
            assert states.shape == (nplans, 4)
        if balls is not None:
            balls = np.ascontiguousarray(balls, dtype=np.float64)
            assert balls.shape == (nplans, n, 2)
        check(lib().rrtk_ctx_plan(self._h, kind, ptr(desc), nplans, n, float(r_rewire), float(r_goal), ptr(samples),
                                  ptr(states), ptr(balls), ptr(pts), ptr(cost), ptr(parent), ptr(stats), ptr(ell)),
              "rrtk_ctx_plan")
        return pts, cost, parent, stats, ell

    def plan_worlds(self, kind, og_u8, desc, n, r_rewire=0.0, r_goal=0.0, samples=None, states=None, balls=None, out=None,
                    chunk=0):
        """Upload + plan + download, pipelined over chunks of plans (plans ordered by world index)."""
        og_u8 = np.ascontiguousarray(og_u8, dtype=np.uint8)
        nw, W, H = og_u8.shape
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        if out is not None:
            pts, cost, parent, stats, ell = out
        else:
            pts = np.empty((nplans, n + 1, 2), dtype=np.int16)
            cost = np.empty((nplans, n + 1), dtype=np.float64)
            parent = np.empty((nplans, n + 1), dtype=np.int32)
            stats = np.empty((nplans, STAT_COUNT), dtype=np.int64)
            ell = np.empty((nplans, n + 1), dtype=np.float64) if kind == KIND_INFORMED else None
        samples = None if samples is None else np.ascontiguousarray(samples, dtype=np.int16)
        states = None if states is None else np.ascontiguousarray(states, dtype=np.uint64)
        balls = None if balls is None else np.ascontiguousarray(balls, dtype=np.float64)
        check(lib().rrtk_ctx_plan_worlds(self._h, kind, ptr(og_u8), nw, W, H, ptr(desc), nplans, n, float(r_rewire), float(r_goal),
                                         ptr(samples), ptr(states), ptr(balls), ptr(pts), ptr(cost), ptr(parent), ptr(stats),
                                         ptr(ell), int(chunk)), "rrtk_ctx_plan_worlds")
        return pts, cost, parent, stats, ell

    def plan_worlds2(self, kind, grids, W, H, desc, n, r_rewire=0.0, r_goal=0.0, samples=None, states=None, balls=None,
                     bits=False, trees=False, paths=True, path_cap=256, out=None, chunk=0, seed_balls=False, shortcut=False,
                     sample_weights=None):
        """rrtk_ctx_plan_worlds2: ``grids`` is (nworlds, W, H) uint8, or with ``bits=True`` the (nworlds, words) uint32 tiled
        bit grids of pack_grids_host.  Returns a dict with ``stats`` and, as requested, the trees (``pts``, ``cost``,
        ``parent``, ``ell``) and / or the path records (``path``, ``xy``, ``len``, ``path_cost``).  ``out``: optional dict of
        preallocated (e.g. pinned) host arrays under the same names.  ``seed_balls`` (informed, with ``states``, no ``balls``):
        the ellipse phase draws from each plan's own generator, as a seeded RRTStarInformed object does (RRTK_SEED_BALLS).
        ``shortcut`` (with ``paths``): the path records come back pruned by line of sight (RRTK_OUT_SHORTCUT, see shortcut()).
        ``sample_weights`` (seed mode): each plan draws its cells from its world's weight map (RRTK_SEED_WEIGHTS): (nworlds, W, H)
        or (W, H) uint8 maps, uploaded by this call, or True for the maps ``set_sample_weights`` already holds."""
        grids = np.ascontiguousarray(grids, dtype=np.uint32 if bits else np.uint8)
        nw = grids.shape[0]
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        out = dict(out or {})
        def buf(name, shape, dtype):
            if name not in out:
                out[name] = np.empty(shape, dtype=dtype)
            return out[name]
        buf("stats", (nplans, STAT_COUNT), np.int64)
        flags = (1 if bits else 0) | (2 if trees else 0) | (4 if paths else 0) | (SEED_BALLS if seed_balls else 0) | (OUT_SHORTCUT if shortcut else 0)
        flags |= self._weights_flag(sample_weights, nw, W, H)
        if trees:
            buf("pts", (nplans, n + 1, 2), np.int16); buf("cost", (nplans, n + 1), np.float64); buf("parent", (nplans, n + 1), np.int32)
            if kind == KIND_INFORMED:
                buf("ell", (nplans, n + 1), np.float64)
        if paths:
            buf("path", (nplans, path_cap), np.int32); buf("xy", (nplans, path_cap, 2), np.int16)
            buf("len", (nplans,), np.int32); buf("path_cost", (nplans,), np.float64)
        samples = None if samples is None else np.ascontiguousarray(samples, dtype=np.int16)
        states = None if states is None else np.ascontiguousarray(states, dtype=np.uint64)
        balls = None if balls is None else np.ascontiguousarray(balls, dtype=np.float64)
        g = out.get
        check(lib().rrtk_ctx_plan_worlds2(self._h, kind, ptr(grids), nw, W, H, ptr(desc), nplans, n, float(r_rewire), float(r_goal),
                                          ptr(samples), ptr(states), ptr(balls), flags, int(path_cap), ptr(g("pts")), ptr(g("cost")),
                                          ptr(g("parent")), ptr(out["stats"]), ptr(g("ell")), ptr(g("path")), ptr(g("xy")), ptr(g("len")),
                                          ptr(g("path_cost")), int(chunk)), "rrtk_ctx_plan_worlds2")
        return out

    def samples(self, desc, n, states):
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        states = np.ascontiguousarray(states, dtype=np.uint64)
        out = np.empty((nplans, n, 2), dtype=np.int16)
        check(lib().rrtk_ctx_samples(self._h, ptr(desc), nplans, n, ptr(states), ptr(out)), "rrtk_ctx_samples")
        return out

    def inflate(self, og_u8: np.ndarray, iterations: int, holes=None) -> np.ndarray:
        """anim.py:79-87 for one (W,H) grid: (nout, W, H) uint8, one inflated grid per (px, py, size) row of ``holes``."""
        og_u8 = np.ascontiguousarray(og_u8, dtype=np.uint8)
        W, H = og_u8.shape
        h = None if holes is None else np.ascontiguousarray(holes, dtype=np.int32).reshape(-1, 3)
        nout = 1 if h is None else h.shape[0]
        out = np.empty((nout, W, H), dtype=np.uint8)
        check(lib().rrtk_ctx_inflate(self._h, ptr(og_u8), W, H, int(iterations), ptr(h), nout, ptr(out)), "rrtk_ctx_inflate")
        return out

    def inflate_disc(self, og_u8: np.ndarray, src, r2) -> np.ndarray:
        """Configuration-space grids of a disc robot (rrtk_ctx_inflate_disc): ``og_u8`` (nworlds, W, H), non-zero = obstacle;
        output o blocks every cell within squared distance ``r2[o]`` (``disc_r2(radius)``) of an obstacle cell of world
        ``src[o]``.  Returns (nout, rrtk_grid_words(W, H)) uint32 tiled bit grids, the form ``plan_worlds2(bits=True)`` takes."""
        og_u8 = np.ascontiguousarray(og_u8, dtype=np.uint8)
        if og_u8.ndim != 3:
            raise ValueError("og_u8 must have shape (nworlds, W, H)")
        nw, W, H = og_u8.shape
        src = np.ascontiguousarray(src, dtype=np.int32).reshape(-1)
        r2 = np.ascontiguousarray(r2, dtype=np.int32).reshape(-1)
        if src.shape != r2.shape:
            raise ValueError("src and r2 need one entry per output")
        out = np.empty((src.shape[0], int(lib().rrtk_grid_words(W, H))), dtype=np.uint32)
        check(lib().rrtk_ctx_inflate_disc(self._h, ptr(og_u8), nw, W, H, ptr(src), ptr(r2), src.shape[0], ptr(out)),
              "rrtk_ctx_inflate_disc")
        return out

    # -- K8: rewire / Dubins planners, Dubins primitive ---------------------------------------
    def plan2(self, cfg, desc, n, samples=None, states=None, heads=None, out=None, balls=None):
        """rrtk_ctx_plan2: returns (pts, head, cost, elen, parent, stats); desc["reserved"][:, :2] = start / goal heading.
        ``out``: optional preallocated host arrays in that order (e.g. pinned).  With ``cfg["informed"]`` set, ``balls`` is the
        (nplans, n, 2) array of unit-disc draws (None = probe run) and a seventh array, the (nplans, n + 1) ellipse budgets, is
        appended to the result."""
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        cfg = np.ascontiguousarray(cfg, dtype=PLAN2_CFG).copy()
        ell = None
        if int(cfg["informed"][0]):
            if balls is not None:
                balls = np.ascontiguousarray(balls, dtype=np.float64)
                assert balls.shape == (nplans, n, 2), balls.shape
            ell = np.empty((nplans, n + 1), dtype=np.float64)
            cfg["balls"], cfg["ell_c"] = (0 if balls is None else balls.ctypes.data), ell.ctypes.data
        if out is not None:
            pts, head, cost, elen, parent, stats = out
            assert pts.shape == (nplans, n + 1, 2) and pts.dtype == np.int16 and head.dtype == np.uint8
            assert cost.shape == elen.shape == (nplans, n + 1) and parent.dtype == np.int32 and stats.shape == (nplans, STAT_COUNT)
        else:
            pts = np.empty((nplans, n + 1, 2), dtype=np.int16)
            head = np.empty((nplans, n + 1), dtype=np.uint8)
            cost = np.empty((nplans, n + 1), dtype=np.float64)
            elen = np.empty((nplans, n + 1), dtype=np.float64)
            parent = np.empty((nplans, n + 1), dtype=np.int32)
            stats = np.empty((nplans, STAT_COUNT), dtype=np.int64)
        if samples is not None:
            samples = np.ascontiguousarray(samples, dtype=np.int16)
            assert samples.shape == (nplans, n, 2), samples.shape
        if states is not None:
            states = np.ascontiguousarray(states, dtype=np.uint64)
            assert states.shape == (nplans, 4)
        if heads is not None:
            heads = np.ascontiguousarray(heads, dtype=np.uint8)
            assert heads.shape == (nplans, n), heads.shape
        check(lib().rrtk_ctx_plan2(self._h, ptr(cfg), ptr(desc), nplans, n, ptr(samples), ptr(states), ptr(heads), ptr(pts), ptr(head),
                                   ptr(cost), ptr(elen), ptr(parent), ptr(stats)), "rrtk_ctx_plan2")
        if ell is not None:
            return pts, head, cost, elen, parent, stats, ell
        return pts, head, cost, elen, parent, stats

    def plan2_worlds(self, cfg, grids, W, H, desc, n, samples=None, states=None, heads=None, bits=False, trees=False, paths=True,
                     path_cap=256, out=None, chunk=0, balls=None, seed_balls=False, sample_weights=None):
        """rrtk_ctx_plan2_worlds: K8 plans with their worlds in one pipelined call.  ``grids`` as for plan_worlds2.  Returns a
        dict with ``stats`` and, as requested, the trees (``pts``, ``head``, ``cost``, ``elen``, ``parent``) and / or the path
        records (``path``, ``xy``, ``path_head``, ``len``, ``path_cost``); informed plans (``cfg["informed"]``, ``balls`` as for
        plan2) also return ``ell``.  ``seed_balls`` and ``sample_weights`` as for plan_worlds2."""
        grids = np.ascontiguousarray(grids, dtype=np.uint32 if bits else np.uint8)
        nw = grids.shape[0]
        nplans = desc.shape[0]
        desc = np.ascontiguousarray(desc, dtype=PLAN_DESC)
        cfg = np.ascontiguousarray(cfg, dtype=PLAN2_CFG).copy()
        out = dict(out or {})
        def buf(name, shape, dtype):
            if name not in out:
                out[name] = np.empty(shape, dtype=dtype)
            return out[name]
        buf("stats", (nplans, STAT_COUNT), np.int64)
        if int(cfg["informed"][0]):
            if balls is not None:
                balls = np.ascontiguousarray(balls, dtype=np.float64)
                assert balls.shape == (nplans, n, 2), balls.shape
            cfg["balls"], cfg["ell_c"] = (0 if balls is None else balls.ctypes.data), buf("ell", (nplans, n + 1), np.float64).ctypes.data
        flags = (1 if bits else 0) | (2 if trees else 0) | (4 if paths else 0) | (SEED_BALLS if seed_balls else 0)
        flags |= self._weights_flag(sample_weights, nw, W, H)
        if trees:
            buf("pts", (nplans, n + 1, 2), np.int16); buf("head", (nplans, n + 1), np.uint8); buf("cost", (nplans, n + 1), np.float64)
            buf("elen", (nplans, n + 1), np.float64); buf("parent", (nplans, n + 1), np.int32)
        if paths:
            buf("path", (nplans, path_cap), np.int32); buf("xy", (nplans, path_cap, 2), np.int16); buf("path_head", (nplans, path_cap), np.uint8)
            buf("len", (nplans,), np.int32); buf("path_cost", (nplans,), np.float64)
        samples = None if samples is None else np.ascontiguousarray(samples, dtype=np.int16)
        states = None if states is None else np.ascontiguousarray(states, dtype=np.uint64)
        heads = None if heads is None else np.ascontiguousarray(heads, dtype=np.uint8)
        g = out.get
        check(lib().rrtk_ctx_plan2_worlds(self._h, ptr(cfg), ptr(grids), nw, W, H, ptr(desc), nplans, n, ptr(samples), ptr(states), ptr(heads),
                                          flags, int(path_cap), ptr(g("pts")), ptr(g("head")), ptr(g("cost")), ptr(g("elen")), ptr(g("parent")),
                                          ptr(out["stats"]), ptr(g("path")), ptr(g("xy")), ptr(g("path_head")), ptr(g("len")), ptr(g("path_cost")),
                                          int(chunk)), "rrtk_ctx_plan2_worlds")
        return out

    def dubins_paths(self, q, nheadings, rho):
        """q: (nq, 6) (x0, y0, h0, x1, y1, h1) -> (word, tpq, length)."""
        q = np.ascontiguousarray(q, dtype=np.int32).reshape(-1, 6)
        word = np.empty(q.shape[0], dtype=np.int32)
        tpq = np.empty((q.shape[0], 3), dtype=np.float64)
        ln = np.empty(q.shape[0], dtype=np.float64)
        check(lib().rrtk_ctx_dubins_paths(self._h, ptr(q), q.shape[0], int(nheadings), float(rho), ptr(word), ptr(tpq), ptr(ln)),
              "rrtk_ctx_dubins_paths")
        return word, tpq, ln

    def dubins_collision(self, q, nheadings, rho, ds, world=0):
        q = np.ascontiguousarray(q, dtype=np.int32).reshape(-1, 6)
        free = np.empty(q.shape[0], dtype=np.uint8)
        check(lib().rrtk_ctx_dubins_collision(self._h, int(world), ptr(q), q.shape[0], int(nheadings), float(rho), float(ds), ptr(free)),
              "rrtk_ctx_dubins_collision")
        return free.astype(bool)

    def dubins_sample(self, q, nheadings, rho, ds, cap):
        """Poses every ds cells: (xyth (nq, cap, 3), count (nq,))."""
        q = np.ascontiguousarray(q, dtype=np.int32).reshape(-1, 6)
        xyth = np.empty((q.shape[0], cap, 3), dtype=np.float64)
        cnt = np.empty(q.shape[0], dtype=np.int32)
        check(lib().rrtk_ctx_dubins_sample(self._h, ptr(q), q.shape[0], int(nheadings), float(rho), float(ds), int(cap), ptr(xyth),
                                           ptr(cnt)), "rrtk_ctx_dubins_sample")
        return xyth, cnt

    def shortcut(self, xy, ln, world=None, path=None):
        """Greedy line-of-sight shortcut of path rows on the context's worlds (rrtk_ctx_shortcut): ``xy`` (P, cap, 2) points root
        first, ``ln`` (P,) their counts, ``world`` (P,) world per row (None = world 0), ``path`` (P, cap) vertex ids or None.
        From each kept point the farthest later point the walk of RRT.collisionfree (rrt.py:183-229) reaches is kept next.
        Returns a new dict: ``xy``, ``len``, ``path`` (None without one) with the kept entries compacted to the front, ``keep``
        (P, cap) their indices in the input row and ``cost`` (P,) the summed segment lengths.  Rows with ``len`` outside
        [1, cap] are not processed: their ``keep`` is -1 and their ``cost`` NaN, the rest as given."""
        xy = np.array(xy, dtype=np.int16, order="C")
        if xy.ndim != 3 or xy.shape[2] != 2:
            raise ValueError("xy must have shape (npaths, cap, 2)")
        P, cap = xy.shape[0], xy.shape[1]
        ln = np.array(ln, dtype=np.int32, order="C").reshape(P)
        w = None if world is None else np.ascontiguousarray(world, dtype=np.int32).reshape(P)
        path = None if path is None else np.array(path, dtype=np.int32, order="C").reshape(P, cap)
        keep = np.full((P, cap), -1, dtype=np.int32)
        cost = np.full(P, np.nan)
        check(lib().rrtk_ctx_shortcut(self._h, ptr(w), P, cap, ptr(xy), ptr(ln), ptr(path), ptr(keep), ptr(cost)), "rrtk_ctx_shortcut")
        return dict(xy=xy, len=ln, path=path, keep=keep, cost=cost)

    # -- queries -------------------------------------------------------------------------------
    def collision(self, segs, world=0, cells=False):
        segs = np.ascontiguousarray(segs, dtype=np.int32).reshape(-1, 4)
        free = np.empty(segs.shape[0], dtype=np.uint8)
        ncell = np.empty(segs.shape[0], dtype=np.int32) if cells else None
        check(lib().rrtk_ctx_collision(self._h, world, ptr(segs), segs.shape[0], ptr(free), ptr(ncell)), "rrtk_ctx_collision")
        return (free.astype(bool), ncell) if cells else free.astype(bool)

    def nearest(self, pts, queries):
        if np.issubdtype(pts.dtype, np.integer) and np.issubdtype(queries.dtype, np.integer):
            p = np.ascontiguousarray(pts, dtype=np.int32)
            q = np.ascontiguousarray(queries, dtype=np.int32).reshape(-1, 2)
            idx = np.empty(q.shape[0], dtype=np.int32)
            key = np.empty(q.shape[0], dtype=np.int64)
            check(lib().rrtk_ctx_nearest(self._h, ptr(p), p.shape[0], ptr(q), q.shape[0], ptr(idx), ptr(key)), "rrtk_ctx_nearest")
        else:
            p = np.ascontiguousarray(pts, dtype=np.float64)
            q = np.ascontiguousarray(queries, dtype=np.float64).reshape(-1, 2)
            idx = np.empty(q.shape[0], dtype=np.int32)
            key = np.empty(q.shape[0], dtype=np.float64)
            check(lib().rrtk_ctx_nearest_f64(self._h, ptr(p), p.shape[0], ptr(q), q.shape[0], ptr(idx), ptr(key)),
                  "rrtk_ctx_nearest_f64")
        return idx, key

    def within(self, pts, queries, r, cap=None):
        integer = np.issubdtype(pts.dtype, np.integer) and np.issubdtype(np.asarray(queries).dtype, np.integer)
        p = np.ascontiguousarray(pts, dtype=np.int32 if integer else np.float64)
        q = np.ascontiguousarray(queries, dtype=p.dtype).reshape(-1, 2)
        cap = p.shape[0] if cap is None else cap
        out = np.empty((q.shape[0], cap), dtype=np.int32)
        ln = np.empty(q.shape[0], dtype=np.int32)
        fn = lib().rrtk_ctx_within if integer else lib().rrtk_ctx_within_f64
        check(fn(self._h, ptr(p), p.shape[0], ptr(q), q.shape[0], float(r), cap, ptr(out), ptr(ln)), "rrtk_ctx_within")
        return out, ln

    def near_order(self, pts, x):
        integer = np.issubdtype(pts.dtype, np.integer) and np.issubdtype(np.asarray(x).dtype, np.integer)
        p = np.ascontiguousarray(pts, dtype=np.int32 if integer else np.float64)
        perm = np.empty(p.shape[0], dtype=np.int32)
        if integer:
            check(lib().rrtk_ctx_near_order(self._h, ptr(p), p.shape[0], int(x[0]), int(x[1]), ptr(perm)), "rrtk_ctx_near_order")
        else:
            check(lib().rrtk_ctx_near_order_f64(self._h, ptr(p), p.shape[0], float(x[0]), float(x[1]), ptr(perm)),
                  "rrtk_ctx_near_order_f64")
        return perm


_shared_ctx = None


def shared_context() -> Context:
    """Process-wide context used by the static-method wrappers (near / within / collisionfree)."""
    global _shared_ctx
    if _shared_ctx is None:
        _shared_ctx = Context()
    return _shared_ctx
