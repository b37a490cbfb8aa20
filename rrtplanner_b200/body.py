"""Bodies with a heading for the Dubins planners: per-heading stencils, their run encoding and the heading-layer rule.

A body is given as ``L`` stencils, one per heading layer ``l = 0 .. L - 1``: an odd ``S x S`` boolean mask centred on offset
``(0, 0)`` whose entry ``[l, i, j]`` is the offset ``(i - k, j - k)``, ``k = (S - 1) // 2``, in grid index coordinates (x = first
index of ``og``).  Layer ``l`` blocks a cell iff some offset of stencil ``l`` lands on an obstacle cell inside the grid
(include/rrtk.h, ``rrtk_inflate_body``); a pose with heading angle ``theta`` tests layer ``body_layer(theta, L)``.
``car_body`` builds stencils for a rectangle that cover every heading mapped to each layer.
"""
from __future__ import annotations

import math
from typing import Tuple

import numpy as np

from . import _lib

__all__ = ["car_body", "body_runs", "body_layer", "inflate_body_host", "MAX_LAYERS", "MAX_STENCIL"]

MAX_LAYERS = 256
MAX_STENCIL = 255
DM_TWO_PI = 6.28318530717958647692      # the double of 2 pi the device and the specification use


def body_layer(theta, nlayers: int):
    """Heading layer of angle(s) ``theta`` (radians, any real) on ``nlayers`` layers:
    ``floor(theta * (nlayers / 2 pi) + 1/2) mod nlayers``, with the device's double operations."""
    th = np.asarray(theta, dtype=np.float64)
    f = np.floor(th * (float(nlayers) / DM_TWO_PI) + 0.5)
    out = np.mod(f.astype(np.int64), int(nlayers))
    return int(out) if out.ndim == 0 else out


def _check_stencils(stencils) -> np.ndarray:
    s = np.asarray(stencils)
    if s.ndim != 3:
        raise ValueError("body stencils must have shape (nlayers, S, S)")
    L, S, S2 = s.shape
    if not 1 <= L <= MAX_LAYERS:
        raise ValueError(f"a body needs 1 .. {MAX_LAYERS} heading layers (got {L})")
    if S != S2 or S % 2 == 0 or not 1 <= S <= MAX_STENCIL:
        raise ValueError(f"body stencils must be odd S x S masks with S <= {MAX_STENCIL} (got {S} x {S2})")
    s = s != 0
    k = (S - 1) // 2
    empty = np.flatnonzero(~s[:, k, k])
    if empty.size:
        raise ValueError(f"stencil {int(empty[0])} does not contain the centre cell")
    return s


def body_runs(stencils) -> Tuple[np.ndarray, np.ndarray]:
    """Encode ``(nlayers, S, S)`` stencils for the device: ``runs`` (n, 3) int32 ``(dx, dy_lo, dy_hi)``, one per maximal run of
    set cells of a stencil row, grouped by layer, and ``layer_runs`` (nlayers + 1,) int32 prefix offsets.  Raises ValueError for
    anything the device rejects: not 1 <= nlayers <= 256, an even or non-square mask, S > 255, a layer without its centre."""
    s = _check_stencils(stencils)
    L, S, _ = s.shape
    k = (S - 1) // 2
    # a run starts where a set cell follows a clear one along the row (dy) and ends where a clear one follows
    pad = np.zeros((L, S, S + 2), dtype=np.int8)
    pad[:, :, 1:-1] = s
    d = np.diff(pad, axis=2)
    lay, row, lo = np.nonzero(d == 1)
    _, _, hi = np.nonzero(d == -1)                   # same (layer, row) order, one end per start
    runs = np.stack([row - k, lo - k, hi - 1 - k], axis=1).astype(np.int32)
    layer_runs = np.zeros(L + 1, dtype=np.int32)
    np.cumsum(np.bincount(lay, minlength=L), out=layer_runs[1:])
    return np.ascontiguousarray(runs), layer_runs


def car_body(front: float, rear: float, half_width: float, nlayers: int = 16, pad: float = 0.0) -> np.ndarray:
    """Stencils ``(nlayers, S, S)`` of a rectangle reaching ``front`` cells ahead of the reference point, ``rear`` behind and
    ``half_width`` to each side.  Layer ``l`` has angle ``l * 2 pi / nlayers``; an offset is set iff its body coordinates
    ``(along, across) = (c dx + s dy, -s dx + c dy)`` lie within ``m`` (+1e-9) of the rectangle, where the margin
    ``m = 2 R sin(pi / (2 nlayers)) + pad`` (R = farthest corner) covers every heading that maps to the layer.  So every integer
    offset that the rectangle turned by any angle theta covers is in stencil ``body_layer(theta, nlayers)``.  ``pad`` widens the
    margin further, e.g. by sqrt(1/2) to cover a pose's rounding to its cell.  ``S = 2 ceil(R + m) + 1`` must stay <= 255."""
    vals = np.array([front, rear, half_width, pad], dtype=np.float64)
    if not np.isfinite(vals).all() or (vals < 0).any():
        raise ValueError("front, rear, half_width and pad must be finite numbers >= 0 (cells)")
    L = int(nlayers)
    if L != nlayers or not 1 <= L <= MAX_LAYERS:
        raise ValueError(f"nlayers must be an integer in [1, {MAX_LAYERS}]")
    R = math.hypot(max(front, rear), half_width)
    m = 2.0 * R * math.sin(math.pi / (2 * L)) + pad
    k = int(math.ceil(R + m))
    if 2 * k + 1 > MAX_STENCIL:
        raise ValueError(f"the body needs {2 * k + 1} x {2 * k + 1} stencils (at most {MAX_STENCIL})")
    d = np.arange(-k, k + 1, dtype=np.float64)
    dx, dy = d[:, None], d[None, :]
    th = np.arange(L, dtype=np.float64) * (2.0 * math.pi / L)
    c, s = np.cos(th)[:, None, None], np.sin(th)[:, None, None]
    along, across = c * dx + s * dy, -s * dx + c * dy
    ex = np.maximum(np.maximum(-rear - along, along - front), 0.0)
    ey = np.maximum(np.abs(across) - half_width, 0.0)
    return np.hypot(ex, ey) <= m + 1e-9


def inflate_body_host(ogs, runs, layer_runs) -> Tuple[np.ndarray, np.ndarray]:
    """Heading layers and projection of ``ogs`` (nworlds, W, H) (or one (W, H) grid), non-zero = obstacle, computed on the
    device (rrtk_inflate_body) and downloaded: ``layers`` (nworlds, nlayers, W, H) and ``proj`` (nworlds, W, H), uint8 of 0 / 1."""
    import torch

    og = np.ascontiguousarray(np.asarray(ogs) != 0, dtype=np.uint8)
    if og.ndim == 2:
        og = og[None]
    if og.ndim != 3:
        raise ValueError("ogs must have shape (nworlds, W, H)")
    if not torch.cuda.is_available():
        raise RuntimeError("inflate_body_host needs a CUDA device (no CPU fallback)")
    nw, W, H = og.shape
    runs = np.ascontiguousarray(runs, dtype=np.int32).reshape(-1, 3)
    layer_runs = np.ascontiguousarray(layer_runs, dtype=np.int32).reshape(-1)
    L = layer_runs.shape[0] - 1
    lib = _lib.lib()
    words = int(lib.rrtk_grid_words(W, H))
    dev = torch.device("cuda", torch.cuda.current_device())
    st = torch.cuda.current_stream(dev).cuda_stream
    d_og = torch.from_numpy(og).to(dev)
    d_runs = torch.from_numpy(np.concatenate([runs.reshape(-1), np.zeros(1, np.int32)])).to(dev)
    d_lr = torch.from_numpy(layer_runs).to(dev)
    bits = torch.empty((nw, words), dtype=torch.int32, device=dev)
    layers = torch.empty((nw * L, words), dtype=torch.int32, device=dev)
    proj = torch.empty((nw, words), dtype=torch.int32, device=dev)
    out_l = torch.empty((nw * L, W, H), dtype=torch.uint8, device=dev)
    out_p = torch.empty((nw, W, H), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.rrtk_pack_grid(d_og.data_ptr(), nw, W, H, bits.data_ptr(), st), "pack")
        _lib.check(lib.rrtk_inflate_body(bits.data_ptr(), nw, W, H, d_runs.data_ptr(), d_lr.data_ptr(), L, layers.data_ptr(),
                                         proj.data_ptr(), st), "rrtk_inflate_body")
        _lib.check(lib.rrtk_unpack_grid(layers.data_ptr(), nw * L, W, H, out_l.data_ptr(), st), "unpack")
        _lib.check(lib.rrtk_unpack_grid(proj.data_ptr(), nw, W, H, out_p.data_ptr(), st), "unpack")
    return out_l.cpu().numpy().reshape(nw, L, W, H), out_p.cpu().numpy()
