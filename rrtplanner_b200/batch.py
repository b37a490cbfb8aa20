"""Batched planning: thousands of independent plans (worlds x start/goal pairs) per launch.

Not in the reference (its ``plan()`` handles one query); this is the batched driver the north star
asks for.  Every plan is what ``RRTStandard / RRTStar / RRTStarInformed(og, n, ...).plan(xstart, xgoal)``
(rrt.py:386-447, 466-556, 653-758) would compute for its world and sample stream; plans never
interact, so a batch shards across GPUs by plan index with no collective (``shard`` below).

Two layers:

* ``DeviceBatch`` -- buffers resident in HBM (torch owns the memory and the stream), kernels
  enqueued through the device-pointer entry points of the C ABI.  Used by ``bench.py`` for the
  kernel-side throughput and by the multi-GPU driver.
* ``plan_batch`` -- host arrays in, host arrays out, through the host-buffer C-ABI call
  ``rrtk_ctx_plan_worlds`` (the end-to-end path: chunked, copies overlapped with kernels).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _lib

KINDS = {"standard": _lib.KIND_STANDARD, "star": _lib.KIND_STAR, "informed": _lib.KIND_INFORMED,
         "RRTStandard": _lib.KIND_STANDARD, "RRTStar": _lib.KIND_STAR, "RRTStarInformed": _lib.KIND_INFORMED}


def make_desc(world_ids, starts, goals, rots=None) -> np.ndarray:
    """Array of rrtk_plan_desc from per-plan world index, start (P,2), goal (P,2), rotation (P,2,2)."""
    starts = np.asarray(starts).reshape(-1, 2)
    goals = np.asarray(goals).reshape(-1, 2)
    d = np.zeros(starts.shape[0], dtype=_lib.PLAN_DESC)
    d["world"] = np.asarray(world_ids, dtype=np.int32)
    d["start_x"], d["start_y"] = starts[:, 0], starts[:, 1]
    d["goal_x"], d["goal_y"] = goals[:, 0], goals[:, 1]
    if rots is not None:
        d["rot"] = np.asarray(rots, dtype=np.float64).reshape(-1, 4)
    return d


def informed_rotations(starts, goals) -> np.ndarray:
    """(P, 2, 2) ``RRTStarInformed.rotation_to_world_frame`` of every start / goal pair (rrt.py:601-613), stacked: the same
    numpy calls (unit axis, outer product with [1, 0], SVD, determinants) on a stack of matrices, which gives the per-pair
    results bit for bit.  Rows where start == goal, whose axis is undefined and where the reference raises, are NaN."""
    starts = np.asarray(starts).reshape(-1, 2)
    goals = np.asarray(goals).reshape(-1, 2)
    span = goals - starts
    out = np.full((span.shape[0], 2, 2), np.nan)
    ok = (span != 0).any(axis=1)
    if ok.any():
        s = span[ok].astype(np.float64)
        axis = s / np.sqrt(s[:, 0] * s[:, 0] + s[:, 1] * s[:, 1])[:, None]     # squares and sum are exact integers
        outer = axis[:, :, None] * np.array([1, 0])[None, None, :]                # np.outer(axis, [1, 0])
        U, _, V = np.linalg.svd(outer)
        D = np.zeros_like(U)
        D[:, 0, 0], D[:, 1, 1] = np.linalg.det(U), np.linalg.det(V)
        out[ok] = U @ D @ np.swapaxes(V, 1, 2)
    return out


_M32 = np.uint64(0xFFFFFFFF)


def _mul64_wide(a, b):
    """(hi, lo) of the 128-bit product of two uint64 arrays."""
    a0, a1, b0, b1 = a & _M32, a >> np.uint64(32), b & _M32, b >> np.uint64(32)
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (p00 >> np.uint64(32)) + (p01 & _M32) + (p10 & _M32)
    lo = (p00 & _M32) | (mid << np.uint64(32))
    hi = p11 + (p01 >> np.uint64(32)) + (p10 >> np.uint64(32)) + (mid >> np.uint64(32))
    return hi, lo


def seed_states(seeds: Sequence[int]) -> np.ndarray:
    """PCG64 start states {state_hi, state_lo, inc_hi, inc_lo} of ``np.random.default_rng(seed)``
    (rrt.py:85) for an array of non-negative integer seeds < 2**64 (rrtk_seed_states: host code of librrtk.so)."""
    seeds = np.asarray(seeds)
    if seeds.ndim != 1 or (seeds.size and (seeds.min() < 0)):
        raise ValueError("seeds must be a 1-D array of non-negative integers")
    s64 = np.ascontiguousarray(seeds.astype(np.uint64))
    out = np.empty((s64.shape[0], 4), dtype=np.uint64)
    _lib.check(_lib.lib().rrtk_seed_states(_lib.ptr(s64), int(s64.shape[0]), _lib.ptr(out)), "rrtk_seed_states")
    return out


def seed_states_numpy(seeds: Sequence[int]) -> np.ndarray:
    """The same in vectorised numpy (kept as an independent statement for the tests).

    Restates numpy's published seeding path (numpy/random/bit_generator.pyx ``SeedSequence``:
    hashmix / mix over a 4-word pool, ``generate_state(4, uint64)``; numpy/random/_pcg64.pyx +
    pcg64.h ``pcg_setseq_128_srandom_r``).  tests/test_host_logic.py checks it against numpy."""
    seeds = np.asarray(seeds)
    if seeds.ndim != 1 or (seeds.size and (seeds.min() < 0)):
        raise ValueError("seeds must be a 1-D array of non-negative integers")
    seeds = seeds.astype(np.uint64)
    u32 = np.uint32
    sh = u32(16)
    with np.errstate(over="ignore"):
        ent = [(seeds & _M32).astype(u32), (seeds >> np.uint64(32)).astype(u32)]
        hc = np.full(seeds.shape, 0x43B0D7E5, dtype=u32)

        def hashmix(v):
            nonlocal hc
            v = v ^ hc
            hc = hc * u32(0x931E8875)
            v = v * hc
            return v ^ (v >> sh)

        def mix(x, y):
            r = u32(0xCA01F9DD) * x - u32(0x4973F715) * y
            return r ^ (r >> sh)

        pool = [hashmix(ent[i] if i < 2 else np.zeros_like(ent[0])) for i in range(4)]
        for src in range(4):
            for dst in range(4):
                if src != dst:
                    pool[dst] = mix(pool[dst], hashmix(pool[src]))
        hb = np.full(seeds.shape, 0x8B51F9DD, dtype=u32)
        words = []
        for i in range(8):
            v = pool[i % 4] ^ hb
            hb = hb * u32(0x58F38DED)
            v = v * hb
            words.append((v ^ (v >> sh)).astype(np.uint64))
        w = [words[2 * i] | (words[2 * i + 1] << np.uint64(32)) for i in range(4)]
        # pcg_setseq_128_srandom_r: state = 0; inc = (initseq << 1) | 1; step; state += initstate; step
        init_hi, init_lo, seq_hi, seq_lo = w
        inc_hi = (seq_hi << np.uint64(1)) | (seq_lo >> np.uint64(63))
        inc_lo = (seq_lo << np.uint64(1)) | np.uint64(1)
        mh, ml = np.uint64(0x2360ED051FC65DA4), np.uint64(0x4385DF649FCCF645)

        def step(hi, lo):
            phi, plo = _mul64_wide(lo, np.full_like(lo, ml))
            phi = phi + hi * ml + lo * mh
            nlo = plo + inc_lo
            return phi + inc_hi + (nlo < plo).astype(np.uint64), nlo

        hi, lo = step(np.zeros_like(init_hi), np.zeros_like(init_lo))
        nlo = lo + init_lo
        hi = hi + init_hi + (nlo < lo).astype(np.uint64)
        hi, lo = step(hi, nlo)
    return np.stack([hi, lo, inc_hi, inc_lo], axis=1)


def shard(nplans: int, rank: int, world_size: int) -> range:
    """Contiguous plan-index range of ``rank`` (plans are independent: no data-path collective)."""
    per = (nplans + world_size - 1) // world_size
    return range(min(rank * per, nplans), min((rank + 1) * per, nplans))


@dataclass
class BatchResult:
    """Host copies of the trees: rows 0..n per plan, laid out as rrtk_plan_batch documents."""
    pts: np.ndarray        # (P, n+1, 2) int16, (-32768, -32768) in unfilled rows
    cost: np.ndarray       # (P, n+1) float64, inf in unfilled rows
    parent: np.ndarray     # (P, n+1) int32, -1 for root / unfilled
    stats: np.ndarray      # (P, STAT_COUNT) int64
    ell_c: Optional[np.ndarray] = None

    def stat(self, name: str) -> np.ndarray:
        return self.stats[:, _lib.STAT_NAMES.index(name)]

    def path(self, p: int):
        """Vertex ids root -> goal vertex of plan p."""
        v = int(self.stats[p, 1])
        out = [v]
        while v > 0:
            v = int(self.parent[p, v])
            out.append(v)
        return out[::-1]

    def path_cost(self, p: int) -> float:
        return float(self.cost[p, int(self.stats[p, 1])])


def plan_batch(kind, ogs, n, starts, goals, world_ids=None, r_rewire=0.0, r_goal=0.0, samples=None, seeds=None,
               balls=None, rots=None, ctx: Optional[_lib.Context] = None) -> BatchResult:
    """End-to-end batched plan() from host arrays through ``rrtk_ctx_plan_worlds``.

    ogs: (nworlds, W, H) array, non-zero = obstacle.  Either ``samples`` (P, n, 2) -- the explicit
    sample streams -- or ``seeds`` (P,) -- plan p's free-space stream is what a planner built with
    seed=seeds[p] draws (``default_rng(seed).integers(0, nfree, n)``, rrt.py:85,240).

    Informed plans take their ellipse phase either from pre-generated streams: ``balls`` (P, n, 2), the unit-disc
    point iteration i would use (rrt.py:579-587), and ``rots`` (P, 2, 2), ``rotation_to_world_frame`` of each
    pair (rrt.py:601-613).  Both are required: without ``balls`` the kernel runs as a probe that stops at the
    first solution vertex, and without ``rots`` every ellipse sample collapses onto the centre, so neither is
    accepted silently.

    Or, with ``seeds`` and ``balls="seed"``, from each plan's own generator, as a seeded planner object interleaves
    its free-space and unit-disc draws on one generator (rrt.py:85,240,579-587): plan p is then what
    ``RRTStarInformed(ogs[world_ids[p]], n, r_rewire, r_goal, seed=seeds[p]).plan(starts[p], goals[p])`` computes.  The
    device runs a probe to each plan's first solution vertex and draws the unit-disc stream past it (RRTK_SEED_BALLS of
    ``rrtk_ctx_plan_worlds2``), so nothing per iteration is uploaded.  ``rots`` defaults to ``informed_rotations``; a plan
    with start == goal that reaches the ellipse phase raises ``np.linalg.LinAlgError``, as the class does.
    """
    k = KINDS[kind] if isinstance(kind, str) else int(kind)
    seed_balls = isinstance(balls, str)
    if seed_balls:
        if balls != "seed" or k != _lib.KIND_INFORMED:
            raise ValueError("balls='seed' is the only string option, and it is for informed plans")
        if seeds is None or samples is not None:
            raise ValueError("balls='seed' draws the ellipse phase from the plans' generators: pass seeds, not samples")
        if rots is None:
            rots = informed_rotations(starts, goals)
    elif k == _lib.KIND_INFORMED and (balls is None or rots is None):
        raise ValueError("plan_batch('informed', ...) needs both balls (P, n, 2) and rots (P, 2, 2), or seeds with "
                         "balls='seed'; see the docstring")
    ogs = np.asarray(ogs)
    if ogs.ndim == 2:
        ogs = ogs[None]
    starts = np.asarray(starts).reshape(-1, 2)
    nplans = starts.shape[0]
    if seed_balls and len(seeds) != nplans:
        raise ValueError("balls='seed' needs one seed per plan")
    if world_ids is None:
        world_ids = np.arange(nplans) % ogs.shape[0]
    own = ctx is None
    ctx = ctx or _lib.Context()
    try:
        og_u8 = ogs if ogs.dtype == np.uint8 else (ogs != 0).astype(np.uint8)
        desc = make_desc(world_ids, starts, goals, rots)
        states = None if seeds is None else seed_states(seeds)
        order = np.argsort(desc["world"], kind="stable")          # the pipelined call wants plans grouped by world
        sorted_ = bool((np.diff(desc["world"]) >= 0).all())
        if sorted_:
            order = np.arange(nplans)
        if seed_balls:
            d = desc[order]
            stats = np.empty((nplans, _lib.STAT_COUNT), dtype=np.int64)
            try:
                o = ctx.plan_worlds2(k, og_u8, og_u8.shape[1], og_u8.shape[2], d, n, r_rewire, r_goal, states=states[order],
                                     trees=True, paths=False, seed_balls=True, out={"stats": stats})
            except ValueError as e:
                bad = (stats[:, 5] >= 0) & ~np.isfinite(d["rot"]).all(axis=1)
                if "start == goal" not in str(e) or not bad.any():
                    raise
                raise np.linalg.LinAlgError(f"plan {int(order[np.argmax(bad)])}: start == goal, so the ellipse of the informed phase "
                                            "has no axis (rotation_to_world_frame, rrt.py:601-613)") from None
            res = (o["pts"], o["cost"], o["parent"], o["stats"], o["ell"])
        elif sorted_:
            res = ctx.plan_worlds(k, og_u8, desc, n, r_rewire, r_goal, samples=samples, states=states, balls=balls)
        else:
            take = lambda a: None if a is None else np.asarray(a)[order]          # noqa: E731
            res = ctx.plan_worlds(k, og_u8, desc[order], n, r_rewire, r_goal, samples=take(samples), states=take(states),
                                  balls=take(balls))
        if sorted_:
            pts, cost, parent, stats, ell = res
        else:
            inv = np.empty_like(order)
            inv[order] = np.arange(order.size)
            pts, cost, parent, stats, ell = (None if a is None else a[inv] for a in res)
    finally:
        if own:
            ctx.close()
    return BatchResult(pts, cost, parent, stats, ell)


class DeviceBatch:
    """HBM-resident batch on one GPU.  torch is plumbing only: allocation, stream, copies."""

    def __init__(self, kind, W: int, H: int, n: int, r_rewire=0.0, r_goal=0.0, device=None, threads: int = 0):
        import torch

        self.torch = torch
        if not torch.cuda.is_available():
            raise RuntimeError("DeviceBatch needs a CUDA device (no CPU fallback)")
        self.dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.kind = KINDS[kind] if isinstance(kind, str) else int(kind)
        self.W, self.H, self.n = W, H, n
        self.r_rewire, self.r_goal, self.threads = float(r_rewire), float(r_goal), threads
        self.L = _lib.lib()
        self.words = int(self.L.rrtk_grid_words(W, H))
        self.og = self.bits = self.rowcum = None
        self.desc = self.samples = self.balls = None
        self.state_out = self.carry_out = None     # seed_informed: the generators after plan()
        self.nplans = 0
        self.out = None

    # -- helpers -------------------------------------------------------------------------------
    def _stream(self):
        return self.torch.cuda.current_stream(self.dev).cuda_stream

    def _empty(self, shape, dtype):
        return self.torch.empty(shape, dtype=dtype, device=self.dev)

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    # -- worlds --------------------------------------------------------------------------------
    def set_worlds_u8(self, og_u8):
        """og_u8: torch uint8 tensor (nworlds, W, H) already on the device."""
        t = self.torch
        assert og_u8.dtype == t.uint8 and og_u8.is_cuda and tuple(og_u8.shape[1:]) == (self.W, self.H)
        self.og = og_u8.contiguous()
        nw = self.og.shape[0]
        self.bits = self._empty((nw, self.words), t.int32)
        self.rowcum = self._empty((nw, self.W + 1), t.int32)
        with t.cuda.device(self.dev):
            _lib.check(self.L.rrtk_pack_grid(self._p(self.og), nw, self.W, self.H, self._p(self.bits), self._stream()), "pack")
            _lib.check(self.L.rrtk_free_rows(self._p(self.bits), nw, self.W, self.H, self._p(self.rowcum), self._stream()), "free_rows")
        return self

    def set_worlds_host(self, ogs: np.ndarray):
        t = self.torch
        h = t.from_numpy(np.ascontiguousarray((np.asarray(ogs) != 0).astype(np.uint8)))
        return self.set_worlds_u8(h.to(self.dev))

    def gen_worlds(self, seeds: Sequence[int], thresh: float = 0.33, chunk: int = 256):
        """Synthetic worlds on the device (bit-identical to worlds.perlin_occupancygrid)."""
        t = self.torch
        seeds = np.asarray(seeds, dtype=np.int32)
        nw = seeds.shape[0]
        og = self._empty((nw, self.W, self.H), t.uint8)
        scratch = self._empty((chunk * self.W * self.H + 2 * chunk,), t.int32)
        d_seeds = t.from_numpy(seeds).to(self.dev)
        with t.cuda.device(self.dev):
            for lo in range(0, nw, chunk):
                m = min(chunk, nw - lo)
                _lib.check(self.L.rrtk_gen_worlds(self._p(d_seeds[lo:]), m, self.W, self.H, int(round(thresh * 1000)),
                                                  self._p(scratch), self._p(og[lo:]), self._stream()), "gen_worlds")
        return self.set_worlds_u8(og)

    def nfree(self) -> np.ndarray:
        return self.rowcum[:, self.W].cpu().numpy()

    def _require_free_cells(self):
        """Seed mode draws free[choice(nfree)] (rrt.py:240): a world without a free cell has nothing to draw (numpy raises)."""
        if self.rowcum is not None and (self.nfree() <= 0).any():
            raise ValueError("world %d has no free cell to sample" % int(np.flatnonzero(self.nfree() <= 0)[0]))

    # -- plans ---------------------------------------------------------------------------------
    def set_plans(self, desc: np.ndarray):
        t = self.torch
        desc = np.ascontiguousarray(desc, dtype=_lib.PLAN_DESC)
        self.nplans = desc.shape[0]
        self.desc = t.from_numpy(desc.view(np.uint8).reshape(self.nplans, 64)).to(self.dev)
        P, n = self.nplans, self.n
        self.out = dict(pts=self._empty((P, n + 1, 2), t.int16), cost=self._empty((P, n + 1), t.float64),
                        parent=self._empty((P, n + 1), t.int32), stats=self._empty((P, _lib.STAT_COUNT), t.int64),
                        ell=self._empty((P, n + 1), t.float64) if self.kind == _lib.KIND_INFORMED else None)
        return self

    def set_samples_host(self, samples: np.ndarray):
        s = np.ascontiguousarray(samples, dtype=np.int16)
        assert s.shape == (self.nplans, self.n, 2)
        self.samples = self.torch.from_numpy(s).to(self.dev)
        return self

    def set_balls_host(self, balls: np.ndarray):
        b = np.ascontiguousarray(balls, dtype=np.float64)
        assert b.shape == (self.nplans, self.n, 2)
        self.balls = self.torch.from_numpy(b).to(self.dev)
        return self

    def seed_samples(self, seeds: Sequence[int]):
        """Sample streams on the device from numpy-compatible PCG64 (rrt.py:85,231-240)."""
        t = self.torch
        self._require_free_cells()
        st = t.from_numpy(seed_states(seeds).view(np.int64)).to(self.dev)
        self.samples = self._empty((self.nplans, self.n, 2), t.int16)
        with t.cuda.device(self.dev):
            _lib.check(self.L.rrtk_sample_streams(self._p(self.bits), self._p(self.rowcum), self.W, self.H, self._p(self.desc),
                                                  self.nplans, self._p(st), self.n, self._p(self.samples), self._stream()),
                       "sample_streams")
        return self

    def _words(self, a, cols, dtype, name):
        """(nplans, cols) generator words as a fresh device tensor: a numpy array (uint64 / uint32) or a torch tensor."""
        t = self.torch
        if isinstance(a, t.Tensor):
            w = a.to(self.dev, dtype).clone()
        else:
            a = np.ascontiguousarray(a)
            w = t.from_numpy(a.view(np.int64 if dtype == t.int64 else np.int32).copy()).to(self.dev)
        if tuple(w.shape) != (self.nplans, cols):
            raise ValueError(f"{name} must have shape ({self.nplans}, {cols})")
        return w.contiguous()

    def _is_informed(self) -> bool:
        return self.kind == _lib.KIND_INFORMED

    def _first_sol_col(self) -> int:
        return _lib.STAT_NAMES.index("first_solution_iter")

    def _use_balls(self, balls):
        self.balls = balls

    def seed_informed(self, states, carry=None):
        """Informed plans from each plan's own generator, as a seeded RRTStarInformed object draws them (rrt.py:85,240,
        579-587): ``states`` (nplans, 4) PCG64 words (``seed_states(seeds)``, or the ``state_out`` of an earlier batch) and
        ``carry`` (nplans, 2) numpy's has_uint32 / uinteger (None = a fresh generator).  Enqueues the sample streams, the
        probe launch (stops at each plan's first solution vertex) and rrtk_ball_streams, which fills the unit-disc stream
        from the generator past that iteration; ``run()`` then plans.  ``state_out`` / ``carry_out`` (device tensors) hold
        the generators as the planner objects hold them after plan(), for a next batch.  The descriptors carry the rotation
        (``make_desc(..., rots=informed_rotations(starts, goals))``)."""
        t = self.torch
        if not self._is_informed():
            raise ValueError("seed_informed is for informed batches")
        self._require_free_cells()
        P, n = self.nplans, self.n
        st = self._words(states, 4, t.int64, "states")
        cr = t.zeros((P, 2), dtype=t.int32, device=self.dev) if carry is None else self._words(carry, 2, t.int32, "carry")
        st_s, cr_s = st.clone(), cr.clone()                # the sampler advances its copy past the n free-space draws
        self.samples = self._empty((P, n, 2), t.int16)
        balls = self._empty((P, n, 2), t.float64)
        self.state_out, self.carry_out = t.empty_like(st), t.empty_like(cr)
        with t.cuda.device(self.dev):
            _lib.check(self.L.rrtk_sample_streams_carry(self._p(self.bits), self._p(self.rowcum), self.W, self.H, self._p(self.desc), P,
                                                        self._p(st_s), self._p(cr_s), n, self._p(self.samples), self._stream()),
                       "sample_streams_carry")
            self._use_balls(None)
            self.run()                                      # probe
            first = self.out["stats"][:, self._first_sol_col()]
            _lib.check(self.L.rrtk_ball_streams(self._p(self.rowcum), self.W, self._p(self.desc), P, n, self._p(st), self._p(cr),
                                                first.data_ptr(), _lib.STAT_COUNT, self._p(balls), self._p(self.state_out),
                                                self._p(self.carry_out), self._stream()), "ball_streams")
        self._use_balls(balls)
        return self

    def run(self):
        """Enqueue the plan kernel on torch's current stream (asynchronous)."""
        o = self.out
        with self.torch.cuda.device(self.dev):
            _lib.check(self.L.rrtk_plan_batch(self.kind, self._p(self.bits), self.W, self.H, self._p(self.desc), self.nplans, self.n,
                                              self.r_rewire, self.r_goal, self._p(self.samples), self._p(self.balls),
                                              self._p(o["pts"]), self._p(o["cost"]), self._p(o["parent"]), self._p(o["stats"]),
                                              self._p(o["ell"]), self.threads, self._stream()), "plan_batch")
        return self

    def paths(self, cap: int):
        t = self.torch
        path = self._empty((self.nplans, cap), t.int32)
        ln = self._empty((self.nplans,), t.int32)
        with t.cuda.device(self.dev):
            _lib.check(self.L.rrtk_extract_paths(self._p(self.out["parent"]), self._p(self.out["stats"]), self.nplans, self.n, cap,
                                                 self._p(path), self._p(ln), self._stream()), "extract_paths")
        return path, ln

    def path_records(self, cap: int = 256):
        """Fixed-size per-plan records on the device -- what a caller of the reference keeps of a plan (rrt.py:87-129):
        path vertex ids, their points, path length, path cost -- plus the statistics row.  Dict of torch tensors with
        leading dimension nplans; the unit multigpu.gather_tensors moves."""
        t = self.torch
        P = self.nplans
        rec = dict(path=self._empty((P, cap), t.int32), xy=self._empty((P, cap, 2), t.int16), len=self._empty((P,), t.int32),
                   path_cost=self._empty((P,), t.float64), stats=self.out["stats"])
        with t.cuda.device(self.dev):
            _lib.check(self.L.rrtk_extract_paths_xy(self._p(self.out["parent"]), self._p(self.out["pts"]), self._p(self.out["cost"]),
                                                    self._p(self.out["stats"]), P, self.n, cap, self._p(rec["path"]), self._p(rec["xy"]),
                                                    self._p(rec["len"]), self._p(rec["path_cost"]), self._stream()), "extract_paths_xy")
        return rec

    def footprint(self):
        import ctypes as C
        smem, blocks = C.c_int(0), C.c_int(0)
        with self.torch.cuda.device(self.dev):
            _lib.check(self.L.rrtk_plan_footprint(self.kind, self.W, self.H, self.n, self.threads, C.byref(smem), C.byref(blocks)),
                       "plan_footprint")
        return smem.value, blocks.value

    def download(self) -> BatchResult:
        o = self.out
        self.torch.cuda.synchronize(self.dev)
        return BatchResult(o["pts"].cpu().numpy(), o["cost"].cpu().numpy(), o["parent"].cpu().numpy(), o["stats"].cpu().numpy(),
                           None if o["ell"] is None else o["ell"].cpu().numpy())


@dataclass
class Batch2Result:
    """Host copies of K8 trees (rrtk_plan2_batch layout)."""
    pts: np.ndarray        # (P, n+1, 2) int16
    head: np.ndarray       # (P, n+1) uint8, 255 in unfilled rows
    cost: np.ndarray       # (P, n+1) float64
    elen: np.ndarray       # (P, n+1) float64 length of the edge from the parent
    parent: np.ndarray     # (P, n+1) int32
    stats: np.ndarray      # (P, STAT_COUNT) int64, slots named by _lib.STAT2_NAMES

    def stat(self, name: str) -> np.ndarray:
        return self.stats[:, _lib.STAT2_NAMES.index(name)]


def make_desc2(world_ids, starts, goals) -> np.ndarray:
    """Descriptors for K8: starts / goals are (P, 3) configurations (x, y, heading index)."""
    starts = np.asarray(starts).reshape(-1, 3)
    goals = np.asarray(goals).reshape(-1, 3)
    d = make_desc(world_ids, starts[:, :2], goals[:, :2])
    d["reserved"][:, 0], d["reserved"][:, 1] = starts[:, 2], goals[:, 2]
    return d


class DeviceBatch2(DeviceBatch):
    """HBM-resident batch of K8 plans (RRT* with a firing rewire, Dubins RRT / RRT*; include/rrtk.h rrtk_plan2_batch)."""

    def __init__(self, model, W: int, H: int, n: int, r_rewire=0.0, star=True, rewire=True, nheadings=16, rho=6.0, ds=1.0,
                 device=None, threads: int = 0, use_table: bool = True, informed: bool = False, r_goal: float = 0.0):
        super().__init__("star" if star else "standard", W, H, n, r_rewire=r_rewire, device=device, threads=threads)
        m = {"euclid": _lib.MODEL_EUCLID, "dubins": _lib.MODEL_DUBINS}[model] if isinstance(model, str) else int(model)
        self.cfg = _lib.plan2_cfg(m, star, rewire, r_rewire, nheadings if m == _lib.MODEL_DUBINS else 1, rho, ds, informed, r_goal)
        self.informed = bool(informed)
        self.balls2 = None
        self.nheadings = int(self.cfg["nheadings"][0])
        self.heads = None
        self.scratch = None
        self.table = None
        if use_table and m == _lib.MODEL_DUBINS and star and 1.0 <= float(r_rewire) <= 1024.0:
            # memo of the Dubins primitive over the rewire radius, shared by every plan of the batch
            R = int(np.ceil(float(r_rewire)))
            nbytes = int(self.L.rrtk_dubins_table_bytes(R, self.nheadings))
            if 0 < nbytes <= (256 << 20):
                self.table = self._empty((nbytes,), self.torch.uint8)
                with self.torch.cuda.device(self.dev):
                    _lib.check(self.L.rrtk_dubins_table_build(R, self.nheadings, float(rho), self._p(self.table), self._stream()),
                               "dubins_table_build")
                self.cfg["dubins_table"], self.cfg["table_radius"] = self.table.data_ptr(), R

    def set_plans(self, desc: np.ndarray):
        t = self.torch
        desc = np.ascontiguousarray(desc, dtype=_lib.PLAN_DESC)
        self.nplans = desc.shape[0]
        self.desc = t.from_numpy(desc.view(np.uint8).reshape(self.nplans, 64)).to(self.dev)
        P, n = self.nplans, self.n
        self.out = dict(pts=self._empty((P, n + 1, 2), t.int16), head=self._empty((P, n + 1), t.uint8),
                        cost=self._empty((P, n + 1), t.float64), elen=self._empty((P, n + 1), t.float64),
                        parent=self._empty((P, n + 1), t.int32), stats=self._empty((P, _lib.STAT_COUNT), t.int64))
        self.scratch = self._empty((int(self.L.rrtk_plan2_scratch_bytes(P, n)),), t.uint8)
        if self.informed:
            self.out["ell"] = self._empty((P, n + 1), t.float64)
            self.cfg["ell_c"] = self.out["ell"].data_ptr()
            self.cfg["balls"] = 0                          # probe until set_balls_host
        return self

    def set_balls_host(self, balls: np.ndarray):
        """Informed plans: (nplans, n, 2) unit-disc draws, row i used by iteration i (rrt.py:579-587); the descriptors carry the
        rotation (make_desc(..., rots=...)).  Without this call an informed batch runs as the probe (stops at the first solution)."""
        b = np.ascontiguousarray(balls, dtype=np.float64)
        assert self.informed and b.shape == (self.nplans, self.n, 2), b.shape
        self._use_balls(self.torch.from_numpy(b).to(self.dev))
        return self

    def _is_informed(self) -> bool:
        return self.informed

    def _first_sol_col(self) -> int:
        return _lib.STAT2_NAMES.index("first_solution_iter")

    def _use_balls(self, balls):
        self.balls2 = balls
        self.cfg["balls"] = 0 if balls is None else balls.data_ptr()

    def set_heads_host(self, heads: np.ndarray):
        h = np.ascontiguousarray(heads, dtype=np.uint8)
        assert h.shape == (self.nplans, self.n) and (h.size == 0 or h.max() < self.nheadings)
        self.heads = self.torch.from_numpy(h).to(self.dev)
        return self

    def seed_heads(self, seeds: Sequence[int]):
        """Heading stream of plan p = default_rng(seeds[p]).integers(0, nheadings, n), drawn on the host."""
        return self.set_heads_host(np.stack([np.random.default_rng(int(s)).integers(0, self.nheadings, self.n) for s in seeds]))

    def run(self):
        o = self.out
        with self.torch.cuda.device(self.dev):
            _lib.check(self.L.rrtk_plan2_batch(_lib.ptr(self.cfg), self._p(self.bits), self.W, self.H, self._p(self.desc), self.nplans,
                                               self.n, self._p(self.samples), self._p(self.heads), self._p(o["pts"]), self._p(o["head"]),
                                               self._p(o["cost"]), self._p(o["elen"]), self._p(o["parent"]), self._p(o["stats"]),
                                               self._p(self.scratch), self.threads, self._stream()), "plan2_batch")
        return self

    def footprint(self):
        import ctypes as C
        smem, blocks = C.c_int(0), C.c_int(0)
        with self.torch.cuda.device(self.dev):
            _lib.check(self.L.rrtk_plan2_footprint(self.n, self.threads, C.byref(smem), C.byref(blocks)), "plan2_footprint")
        return smem.value, blocks.value

    def download(self) -> Batch2Result:
        o = self.out
        self.torch.cuda.synchronize(self.dev)
        return Batch2Result(*(o[k].cpu().numpy() for k in ("pts", "head", "cost", "elen", "parent", "stats")))
