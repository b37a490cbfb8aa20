"""Specification of the weighted sample streams (test infrastructure; nothing under rrtplanner_b200/ imports it).

A weight map is (W, H) uint8, w[x, y].  The effective weight of a cell is w where the planning grid leaves it free, else 0;
T is their sum.  A plan's stream of n samples is, exactly:

    cum = np.cumsum(e.ravel().astype(np.int64))
    k   = np.searchsorted(cum, rng.integers(0, T, size=n), side="right")
    samples = np.stack(np.divmod(k, H), axis=1)        # (x, y)

with the plan's numpy PCG64 generator: ``default_rng(seed)``, or a generator resumed from PCG64 state words
{state_hi, state_lo, inc_hi, inc_lo} and numpy's buffered 32-bit half (carry = (has_uint32, uinteger)).
"""
from __future__ import annotations

import numpy as np

_M64 = (1 << 64) - 1


def effective_weights(weights, free) -> np.ndarray:
    """(W, H) int64: the weight where ``free`` is true, else 0."""
    return np.where(np.asarray(free, dtype=bool), np.asarray(weights).astype(np.int64), 0)


def generator(seed=None, state=None, carry=None) -> np.random.Generator:
    """``default_rng(seed)``, or a PCG64 generator at ``state`` (4 uint64 words) with ``carry`` (has_uint32, uinteger)."""
    if state is None:
        return np.random.default_rng(seed)
    s = [int(v) for v in np.asarray(state, dtype=np.uint64)]
    c = (0, 0) if carry is None else [int(v) for v in np.asarray(carry, dtype=np.uint32)]
    bg = np.random.PCG64()
    bg.state = {"bit_generator": "PCG64", "state": {"state": (s[0] << 64) | s[1], "inc": (s[2] << 64) | s[3]},
                "has_uint32": int(c[0] != 0), "uinteger": int(c[1])}
    return np.random.Generator(bg)


def generator_words(rng: np.random.Generator):
    """(state words (4,) uint64, carry (2,) uint32) of a PCG64 generator."""
    st = rng.bit_generator.state
    s, inc = st["state"]["state"], st["state"]["inc"]
    words = np.array([s >> 64, s & _M64, inc >> 64, inc & _M64], dtype=np.uint64)
    return words, np.array([st["has_uint32"], st["uinteger"]], dtype=np.uint32)


def weighted_stream(weights, free, n, seed=None, state=None, carry=None):
    """(samples (n, 2) int64, state words after the draws, carry after the draws) of one plan.  Raises ValueError when T == 0,
    as numpy does for integers(0, 0)."""
    e = effective_weights(weights, free)
    H = e.shape[1]
    cum = np.cumsum(e.ravel())
    T = int(cum[-1]) if cum.size else 0
    rng = generator(seed, state, carry)
    k = np.searchsorted(cum, rng.integers(0, T, size=n), side="right")
    samples = np.stack(np.divmod(k, H), axis=1).astype(np.int64)
    words, c = generator_words(rng)
    return samples, words, c


def brute_force_stream(weights, free, n, seed=None):
    """The same stream by a linear walk over the cells per draw (an independent statement of the rank -> cell rule)."""
    e = effective_weights(weights, free)
    W, H = e.shape
    flat = e.ravel()
    T = int(flat.sum())
    rng = np.random.default_rng(seed)
    out = np.empty((n, 2), dtype=np.int64)
    for i in range(n):
        k = int(rng.integers(0, T))
        acc = 0
        for c in range(flat.size):
            acc += int(flat[c])
            if k < acc:
                out[i] = divmod(c, H)
                break
    return out
