"""Greedy line-of-sight shortcut of path records  --  TEST INFRASTRUCTURE ONLY.

The specification of ``rrtk_shortcut_paths`` (include/rrtk.h), restated on ``rrt_oracle.first_hit`` (the reference's
``collisionfree``, rrt.py:183-229, pinned to its golden collision fixtures) with Python floats for the cost::

    keep = [0]; i = 0
    while i < m - 1:
        k = max({k in (i, m-1] : collisionfree(og, q_i, q_k)} | {i + 1})     # walk q_i -> q_k, earlier point first
        keep.append(k); i = k
    cost = 0.0; for consecutive (a, b) of q[keep]: cost = cost + sqrt(float(|b - a|^2))

Rows are laid out as ``rrtk_extract_paths_xy`` writes them; rows with ``len <= 0`` or ``len > cap`` are not processed.
"""
from __future__ import annotations

import math

import numpy as np

from .rrt_oracle import first_hit


def shortcut_indices(og: np.ndarray, pts) -> list:
    """Indices of the kept points of one polyline ``pts`` (m, 2), root first."""
    m = len(pts)
    keep, i = [0], 0
    while i < m - 1:
        k = i + 1
        for cand in range(m - 1, i + 1, -1):
            if first_hit(og, pts[i], pts[cand])[0]:
                k = cand
                break
        keep.append(k)
        i = k
    return keep


def shortcut_cost(pts) -> float:
    cost = 0.0
    for a, b in zip(pts[:-1], pts[1:]):
        dx, dy = int(b[0]) - int(a[0]), int(b[1]) - int(a[1])
        cost = cost + math.sqrt(float(dx * dx + dy * dy))
    return cost


def shortcut_records(ogs, xy, ln, world=None, path=None) -> dict:
    """Expected outputs of ``_lib.Context.shortcut`` for (P, cap, 2) rows ``xy`` with counts ``ln`` on grids ``ogs``
    ((nworlds, W, H), or one (W, H) grid); unprocessed rows keep their entries, with ``keep`` -1 and ``cost`` NaN."""
    ogs = np.asarray(ogs)
    if ogs.ndim == 2:
        ogs = ogs[None]
    xy = np.array(xy, dtype=np.int16)
    P, cap = xy.shape[0], xy.shape[1]
    ln = np.array(ln, dtype=np.int32).reshape(P)
    path = None if path is None else np.array(path, dtype=np.int32).reshape(P, cap)
    keep = np.full((P, cap), -1, dtype=np.int32)
    cost = np.full(P, np.nan)
    for p in range(P):
        m = int(ln[p])
        if m <= 0 or m > cap:
            continue
        og = ogs[0 if world is None else int(world[p])]
        pts = xy[p, :m].astype(np.int64)
        kp = shortcut_indices(og, pts)
        t = len(kp)
        keep[p, :t] = kp
        cost[p] = shortcut_cost(pts[kp])
        xy[p, :t] = pts[kp]
        xy[p, t:] = -32768
        if path is not None:
            path[p, :t] = path[p, kp]
            path[p, t:] = -1
        ln[p] = t
    return dict(xy=xy, len=ln, path=path, keep=keep, cost=cost)
