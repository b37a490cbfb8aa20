"""References for a body with a heading -- TEST INFRASTRUCTURE ONLY.  Nothing in ``rrtplanner_b200`` imports this module.

Layer grids (include/rrtk.h, rrtk_inflate_body): layer l of a world blocks cell c iff some offset d of stencil l (entry [l, i, j]
= offset (i - k, j - k)) has c + d inside the grid on an obstacle; cells outside the grid are free.  ``layers_scipy`` states it
through scipy's dilation, which mirrors its structure element (hence the reflected stencil); ``layers_direct`` states it
literally, as the test of the two agrees.

Planners on the layers (rrtk_plan2_batch_layers, rrtk_dubins_collision_layers): ``plan_layers`` and ``dubins_free_layers`` are
the ctypes front-end of oracle/body_oracle.c, the specification the device is tested against bit for bit.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
from scipy import ndimage

from . import rewire_oracle as R

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "body_oracle.c")
_OUT = os.path.join(_HERE, "_build", "liborcbody.so")
_lib = None


def layers_scipy(og, stencils) -> np.ndarray:
    """(L, W, H) bool: layer[l] = binary_dilation(og != 0, structure=S_l[::-1, ::-1], border_value=0)."""
    occ = np.asarray(og) != 0
    s = np.asarray(stencils) != 0
    return np.stack([ndimage.binary_dilation(occ, structure=m[::-1, ::-1], border_value=0) for m in s])


def layers_direct(og, stencils) -> np.ndarray:
    """The definition itself: OR over the set offsets d of stencil l of og[c + d] (False outside the grid)."""
    occ = np.asarray(og) != 0
    s = np.asarray(stencils) != 0
    W, H = occ.shape
    k = (s.shape[1] - 1) // 2
    padded = np.zeros((W + 2 * k, H + 2 * k), dtype=bool)
    padded[k:k + W, k:k + H] = occ
    out = np.zeros((s.shape[0], W, H), dtype=bool)
    for l in range(s.shape[0]):
        for i, j in zip(*np.nonzero(s[l])):
            out[l] |= padded[i:i + W, j:j + H]           # og[x + (i - k), y + (j - k)]
    return out


def projection(layers) -> np.ndarray:
    """A cell of the projection is blocked iff every layer blocks it."""
    return np.logical_and.reduce(np.asarray(layers) != 0, axis=0)


def build(force: bool = False) -> str:
    deps = (_SRC, os.path.join(_HERE, "rewire_oracle.c"))
    if force or not os.path.exists(_OUT) or any(os.path.getmtime(_OUT) < os.path.getmtime(d) for d in deps):
        os.makedirs(os.path.dirname(_OUT), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", _OUT, _SRC, "-lm"])
    return _OUT


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_OUT)
        vp, i, d, lg = C.c_void_p, C.c_int, C.c_double, C.c_long
        L.orc2_plan_layers.restype = i
        L.orc2_plan_layers.argtypes = [i, i, vp, i, i, i, i, d, i, d, d] + [vp] * 9
        L.orc2_plan_informed_layers.restype = i
        L.orc2_plan_informed_layers.argtypes = [i, i, vp, i, i, i, i, d, i, d, d] + [vp] * 9 + [d, vp, vp, vp]
        L.orc2_dubins_free_layers.restype = None
        L.orc2_dubins_free_layers.argtypes = [vp, i, i, i, vp, lg, i, d, d, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _layers(layers):
    g = np.ascontiguousarray(np.asarray(layers) != 0, dtype=np.uint8)
    if g.ndim != 3:
        raise ValueError("layers must have shape (L, W, H)")
    return g


def dubins_free_layers(layers, q, nh, rho, ds):
    """rewire_oracle.dubins_free on heading-layer grids ``layers`` (L, W, H): a sampled pose tests the layer of its own angle, the
    end cell the layer of the end heading."""
    g = _layers(layers)
    q = np.ascontiguousarray(q, dtype=np.int32).reshape(-1, 6)
    out = np.empty(q.shape[0], dtype=np.uint8)
    lib().orc2_dubins_free_layers(_p(g), g.shape[0], g.shape[1], g.shape[2], _p(q), q.shape[0], int(nh), float(rho), float(ds), _p(out))
    return out.astype(bool)


def plan_layers(layers, n, start, goal, samples, star=True, rewire=True, r_rewire=0.0, nh=16, rho=1.0, ds=1.0, informed=None):
    """rewire_oracle.plan("dubins", ...) on heading-layer grids ``layers`` (L, W, H) instead of one grid; same arguments and
    result otherwise."""
    g = _layers(layers)
    L, W, H = g.shape
    s = np.ascontiguousarray(samples, dtype=np.int32)
    assert s.shape == (n, 3), s.shape
    st = np.ascontiguousarray(start, dtype=np.int32).reshape(3)
    gl = np.ascontiguousarray(goal, dtype=np.int32).reshape(3)
    pts = np.empty((n + 1, 2), dtype=np.int32)
    head = np.empty(n + 1, dtype=np.int32)
    cost, elen = np.empty(n + 1), np.empty(n + 1)
    par = np.empty(n + 1, dtype=np.int32)
    stats = np.zeros(len(R.ST_NAMES), dtype=np.int64)
    args = (int(bool(star)), int(bool(rewire)), _p(g), L, W, H, n, float(r_rewire), int(nh), float(rho), float(ds), _p(st), _p(gl), _p(s),
            _p(pts), _p(head), _p(cost), _p(elen), _p(par), _p(stats))
    ell = None
    if informed is None:
        rc = lib().orc2_plan_layers(*args)
    else:
        rot = np.ascontiguousarray(informed["rot"], dtype=np.float64).reshape(4)
        balls = None if informed.get("balls") is None else np.ascontiguousarray(informed["balls"], dtype=np.float64).reshape(n, 2)
        ell = np.empty(n + 1)
        rc = lib().orc2_plan_informed_layers(*args, float(informed["r_goal"]), _p(rot), _p(balls), _p(ell))
    if rc:
        raise MemoryError("orc2_plan_layers")
    out = dict(pts=pts, head=head, cost=cost, elen=elen, parent=par, stats=dict(zip(R.ST_NAMES, (int(v) for v in stats))))
    if ell is not None:
        out["ell"] = ell
    return out
