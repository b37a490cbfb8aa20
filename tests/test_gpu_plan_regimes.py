"""Every kernel variant the K7 dispatch (csrc/plan.cu) can reach, against the C oracle bit for bit.

The dispatch picks one of three kernels -- the bucket kernel (plan_grid.cuh), the packed-key scan kernel (plan_scan.cuh) and
the 32-bit-distance wide kernel (plan_wide.cu) -- and, within each, a block shape, a membership-word layout and a key width.
This file restates that choice in Python (``dispatch``), checks the restatement against the library (kernel name and shared
memory) on every table row before the row runs, and then compares every tree with ``oracle.c_oracle.plan_raw``.  A change of
the dispatch thresholds fails ``test_dispatch_restatement`` with the row's id, so the tables get new rows instead of silently
testing other variants.  Fields the library does not report (T, K, membership words, tail bytes, key width) come from the
restatement; each row states the values it is meant to exercise, and the rows at a limit sit on both sides of it.

All environment overrides are read by plan.cu at each launch, so ``monkeypatch.setenv`` switches them per test."""
import ctypes as C
import functools
import math
import os

import numpy as np
import pytest

from oracle import rrt_oracle as O
from rrtplanner_b200 import _lib, batch, worlds
from tests.test_gpu_parity import assert_same_as_oracle, edge_cases, oracle_tree, run_edge_case

pytestmark = pytest.mark.gpu

KIND = {"standard": 0, "star": 1, "informed": 2}
OVERRIDES = ("RRTK_PLAN_IMPL", "RRTK_PLAN_K", "RRTK_PLAN_T", "RRTK_PLAN_CAP", "RRTK_GRID_K", "RRTK_GRID_SMEM", "RRTK_GRID_BSX",
             "RRTK_GRID_BSY", "RRTK_GRID_KEY32")
KEY_LIMIT = 1 << 29          # scan keys: (2 side^2) << sbits must not exceed this (plan.cu, scan_shape)
WIDE_LIST_CAP = 256          # kWideListCap, plan_wide.cu


# ---- the dispatch of csrc/plan.cu, restated ----------------------------------------------------------------------------------
def _env_int(name, dflt):
    s = os.environ.get(name, "")
    return int(s) if s else dflt


def _bits_for(v):
    b = 0
    while (1 << b) <= v:
        b += 1
    return b


def grid_shape(kind, W, H, n, threads, optin):
    """plan.cu grid_shape: the bucket kernel's shape, or None when it does not take the plan."""
    impl = os.environ.get("RRTK_PLAN_IMPL", "")[:1]
    if impl in ("w", "s") or kind not in (KIND["standard"], KIND["star"]) or threads not in (0, 128):
        return None
    if _env_int("RRTK_PLAN_T", 0) != 0 or (n < 256 and impl != "g"):
        return None
    K = _env_int("RRTK_GRID_K", 16)
    if K not in (8, 16):
        return None
    ib = 32 - _bits_for(W - 1) - _bits_for(H - 1)
    if ib < 1 or ib > 31 or n >= (1 << ib) - 1:                  # ids 0 .. n beside the packed coordinates, one word
        return None
    bsx, bsy = _env_int("RRTK_GRID_BSX", 5), _env_int("RRTK_GRID_BSY", 2)
    while True:
        nbx, nby = -(-W // (1 << bsx)), -(-H // (1 << bsy))
        if nbx * nby <= 2048 and nbx * nby + 1 <= n:
            break
        if bsx >= 15:
            return None
        if bsy < bsx:
            bsy += 1
        else:
            bsx += 1
    need = (n + 1 + 31) & ~31
    list_cap = 0 if kind == KIND["standard"] else min(_env_int("RRTK_PLAN_CAP", 256), need)
    smem = 4 * need + 16 * list_cap + ((2 * (nbx * nby + 1) + 15) & ~15)
    kb = _bits_for(n)
    d2max = (W - 1) ** 2 + (H - 1) ** 2
    if kb >= 32 or d2max >= (1 << (32 - kb)) - 1 or _env_int("RRTK_GRID_KEY32", 1) == 0:
        kb = 0                                                    # two-word (distance, id) keys
    if smem > optin - 4096:
        return None
    return dict(kernel="grid", T=128, K=K, list_cap=list_cap, kb=kb, key_words=1 if kb else 2, smem=smem)


def scan_shape(kind, W, H, n, threads, optin, sm_smem):
    """plan.cu scan_shape: the packed-key scan kernel's shape, or None."""
    if os.environ.get("RRTK_PLAN_IMPL", "")[:1] == "w" or n + 1 > 65535:
        return None
    K = _env_int("RRTK_PLAN_K", 8)
    if K not in (4, 8, 16):
        return None
    T = threads if threads > 0 else _env_int("RRTK_PLAN_T", 0)
    if T <= 0:
        T = 64 if n < 2048 else 128 if n < 5120 else 256 if n < 32768 else 512
    if T not in (64, 128, 160, 256, 512):
        return None
    rows = -(-(n + 1) // T)
    hw = -(-rows // 32)
    if hw > 4:
        return None
    sbits = 5 if hw == 1 else 6 if hw == 2 else 7
    side = max(W, H)
    if (2 * side * side) << sbits > KEY_LIMIT:
        return None
    steps_max = (rows + 3) // 4
    need = (n + 1 + 31) & ~31
    list_cap = 0 if kind == KIND["standard"] else min(_env_int("RRTK_PLAN_CAP", 448 if kind == KIND["informed"] else 256), need)
    tail_rows = rows - 32 * (hw - 1)
    tail = 1 if tail_rows <= 8 else 2 if tail_rows <= 16 else 4
    smem = 16 * T * steps_max
    if kind != KIND["standard"]:
        smem += 4 * (hw - 1) * K * T + ((tail * K * T + 3) & ~3) + 2 * (T // 32) * list_cap
    smem = (smem + 15) & ~15
    if smem > optin - 2048:
        return None
    two = int(T == 256 and sm_smem // (smem + 2048) <= 2)
    return dict(kernel="scan", T=T, K=K, hit_words=hw, tail_bytes=tail, sbits=sbits, list_cap=list_cap, two_per_sm=two, smem=smem)


def wide_shape(kind, W, H, n, threads, optin, sm_smem):
    """plan_wide.cu wide_plan_footprint / choose_grid_smem."""
    T = 0 if threads in (160, 512) else threads
    if T <= 0:
        T = 128 if n >= 512 else 64
    npad = (n + 1 + 3) & ~3
    hw = (-(-(npad >> 2) // T) + 7) >> 3

    def size(grid):
        b = npad * 4 + (T // 32) * hw * T * 4 + (T // 32) * WIDE_LIST_CAP * 2 + 16
        if grid:
            b += -(-W // 32) * -(-H // 32) * 32 * 4
        return (b + 15) & ~15

    def per_sm(b):
        return max(1, min(sm_smem // (b + 2048), 2048 // T, 32))

    budget = optin - 2048
    in_smem = size(True) <= budget and per_sm(size(True)) >= per_sm(size(False))
    force = os.environ.get("RRTK_GRID_SMEM", "")[:1]
    if force == "0":
        in_smem = False
    if force == "1" and size(True) <= budget:
        in_smem = True
    smem = size(in_smem)
    if smem > budget:
        return None
    return dict(kernel="wide", T=T, K=T // 32, list_cap=0 if kind == KIND["standard"] else WIDE_LIST_CAP, grid_smem=int(in_smem),
                smem=smem)


def dispatch(kind, W, H, n, threads, optin, sm_smem):
    return (grid_shape(kind, W, H, n, threads, optin) or scan_shape(kind, W, H, n, threads, optin, sm_smem)
            or wide_shape(kind, W, H, n, threads, optin, sm_smem))


@functools.lru_cache(maxsize=None)
def device_limits():
    """(opt-in shared memory per block, shared memory per SM) of the device the library plans on."""
    import torch
    sms, optin = C.c_int(0), C.c_int(0)
    _lib.check(_lib.lib().rrtk_device_info(C.byref(sms), C.byref(optin)), "device_info")
    return optin.value, torch.cuda.get_device_properties(torch.cuda.current_device()).shared_memory_per_multiprocessor


def checked_shape(row, kind, W, H, n, threads=0, expect=None):
    """The restated shape of a plan under the current environment, after checking it against the library: the kernel
    rrtk_plan_kernel names and the shared memory rrtk_plan_footprint reports.  ``expect``: the fields the row is meant to
    exercise."""
    k = KIND[kind]
    shape = dispatch(k, W, H, n, threads, *device_limits())
    assert shape is not None, f"row {row}: no kernel takes this plan in the restated dispatch"
    L = _lib.lib()
    got = L.rrtk_plan_kernel(k, W, H, n, threads).decode()
    assert got == shape["kernel"], (f"row {row}: the library runs the {got} kernel, the restated dispatch says {shape['kernel']}: "
                                    "the dispatch changed, update the restatement and the table rows")
    smem, per_sm = C.c_int(0), C.c_int(0)
    _lib.check(L.rrtk_plan_footprint(k, W, H, n, threads, C.byref(smem), C.byref(per_sm)), "plan_footprint")
    assert smem.value == shape["smem"], (f"row {row}: the library's {got} kernel takes {smem.value} bytes of shared memory, the "
                                         f"restated dispatch says {shape['smem']}: update the restatement and the table rows")
    for f, v in (expect or {}).items():
        assert shape.get(f) == v, f"row {row}: {f} = {shape.get(f)} in the restated dispatch, the row is meant for {v}"
    return shape


# ---- plans --------------------------------------------------------------------------------------------------------------------
def unit_disc(rng, n):
    u = rng.uniform(0, 1, size=(n, 2))
    return np.stack([np.sqrt(u[:, 0]) * np.cos(2 * np.pi * u[:, 1]), np.sqrt(u[:, 0]) * np.sin(2 * np.pi * u[:, 1])], axis=-1)


def plan_vs_oracle(kind, ogs, starts, goals, samples, r, rg, threads=0, seed=0):
    """One launch of len(starts) plans (plan p on world p), every tree compared with the C oracle; returns the oracle's."""
    P = len(starts)
    _, W, H = ogs.shape
    n = samples.shape[1]
    inf = kind == "informed"
    rots = np.stack([O.ellipse_rotation(a, b) for a, b in zip(starts, goals)]) if inf else None
    balls = np.stack([unit_disc(np.random.default_rng(seed + p), n) for p in range(P)]) if inf else None
    db = batch.DeviceBatch(kind, W, H, n, r, rg, threads=threads).set_worlds_host(ogs)
    db.set_plans(batch.make_desc(np.arange(P), starts, goals, rots))
    db.set_samples_host(samples)
    if inf:
        db.set_balls_host(balls)
    res = db.run().download()
    wants = []
    for p in range(P):
        want = oracle_tree(kind, ogs[p], n, starts[p], goals[p], samples[p], r, rg, None if balls is None else balls[p],
                           None if rots is None else rots[p])
        assert_same_as_oracle(res, p, want)
        wants.append(want)
    return wants


def perlin_plans(kind, W, H, n, r, rg, plans, seed, threads=0):
    ogs = np.stack([worlds.perlin_occupancygrid(W, H, seed=seed + p) for p in range(plans)]).astype(np.uint8)
    pairs = [worlds.start_goal(ogs[p], seed + p) for p in range(plans)]
    samples = np.stack([O.sample_stream(ogs[p], n, seed + p) for p in range(plans)])
    return plan_vs_oracle(kind, ogs, [a for a, _ in pairs], [b for _, b in pairs], samples, r, rg, threads, seed)


def set_env(monkeypatch, env):
    for k in OVERRIDES:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))


def row(kind, W, H, n, expect, env=None, threads=0, plans=2, r=50.0, rg=20.0):
    env = dict(env or {})
    parts = [expect["kernel"]] + [f"{k}{v}" for k, v in expect.items() if k != "kernel"] + [kind, f"{W}x{H}", f"n{n}"]
    parts += ([f"threads{threads}"] if threads else []) + [f"{k[5:].lower()}={v}" for k, v in env.items()]
    return pytest.param(kind, W, H, n, env, threads, expect, plans, r, rg, id="-".join(parts))


def max_radius_set(pts, j, r):
    """max over the tree's sampled vertices i of |{v < i : d2(v, i) < r^2}|: the radius set vertex i was connected with."""
    p = pts[:j].astype(np.int64)
    best = 0
    for i in range(1, j):
        d2 = ((p[:i] - p[i]) ** 2).sum(1)
        best = max(best, int((d2 < r * r).sum()))
    return best


# ---- 2. regimes of the scan and wide kernels, default dispatch and forced variants ---------------------------------------------
# Worlds the bucket kernel refuses for standard / star (bits(W-1) + bits(H-1) + bits(n+1) > 32):
#   2400 x 1100: 12 + 11 bits, n >= 511 (scan: one membership word only, side > 2048)
#   2048 x 1200: 11 + 11 bits, n >= 1023
#   1024 x 1024: 10 + 10 bits, n >= 4095
def scan(T, hw, tail, K=8, **kw):
    return dict(kernel="scan", T=T, K=K, hit_words=hw, tail_bytes=tail, **kw)


REGIME_ROWS = []
for _k in ("standard", "star", "informed"):
    REGIME_ROWS += [
        row(_k, 2400, 1100, 200, scan(64, 1, 1)),
        row(_k, 2400, 1100, 700, scan(64, 1, 2)),
        row(_k, 2048, 1200, 1023, scan(64, 1, 2)),                 # n + 1 = 1024: the bucket kernel's id limit on this grid
        row(_k, 2400, 1100, 1500, scan(64, 1, 4)),
        row(_k, 2400, 1100, 3000, scan(128, 1, 4)),
        row(_k, 2048, 1200, 4500, scan(128, 2, 1), plans=1),
        row(_k, 1024, 1024, 6000, scan(256, 1, 4, two_per_sm=0), plans=1),
        row(_k, 1024, 1024, 8300, scan(256, 2, 1, two_per_sm=0), plans=1),
        row(_k, 1024, 1024, 12000, scan(256, 2, 2, two_per_sm=0), plans=1),
        row(_k, 1024, 1024, 20000, scan(256, 3, 2, two_per_sm=1), plans=1),
        row(_k, 1024, 1024, 30000, scan(256, 4, 4, two_per_sm=1), plans=1),
        row(_k, 1024, 1024, 34000, scan(512, 3, 1), plans=1),
        # forced: samples per round, 160 threads
        row(_k, 2400, 1100, 700, scan(64, 1, 2, K=4), env={"RRTK_PLAN_K": 4}),
        row(_k, 1024, 1024, 12000, scan(256, 2, 2, K=4, two_per_sm=0), env={"RRTK_PLAN_K": 4}, plans=1),
        row(_k, 2400, 1100, 700, scan(64, 1, 2, K=16), env={"RRTK_PLAN_K": 16}),
        row(_k, 2048, 1200, 4500, scan(128, 2, 1, K=16), env={"RRTK_PLAN_K": 16}, plans=1),
        row(_k, 1024, 1024, 20000, scan(256, 3, 2, K=16, two_per_sm=1), env={"RRTK_PLAN_K": 16}, plans=1),
        row(_k, 1024, 1024, 3000, scan(160, 1, 4), env={"RRTK_PLAN_T": 160}),
        row(_k, 1024, 1024, 6000, scan(160, 2, 1), env={"RRTK_PLAN_T": 160}, plans=1),
        # the wide kernel: 64 / 128 / 256 threads, grid in shared or global memory
        row(_k, 1024, 1024, 400, dict(kernel="wide", T=64, grid_smem=1), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 1}),
        row(_k, 1024, 1024, 400, dict(kernel="wide", T=64, grid_smem=0), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 0}),
        row(_k, 1024, 1024, 3000, dict(kernel="wide", T=128, grid_smem=1), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 1}),
        row(_k, 1024, 1024, 3000, dict(kernel="wide", T=128, grid_smem=0), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 0}),
        row(_k, 1024, 1024, 3000, dict(kernel="wide", T=256, grid_smem=1), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 1},
            threads=256),
        row(_k, 1024, 1024, 3000, dict(kernel="wide", T=256, grid_smem=0), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 0},
            threads=256),
    ]
# T = 512 with four membership words: the tree alone takes 200 KB, so only RRTStandard (no membership words in shared memory)
REGIME_ROWS.append(row("standard", 1024, 1024, 50000, scan(512, 4, 1), plans=1))


@pytest.mark.parametrize("kind,W,H,n,env,threads,expect,plans,r,rg", REGIME_ROWS)
def test_kernel_regimes(monkeypatch, request, kind, W, H, n, env, threads, expect, plans, r, rg):
    set_env(monkeypatch, env)
    checked_shape(request.node.callspec.id, kind, W, H, n, threads, expect)
    perlin_plans(kind, W, H, n, r, rg, plans, seed=100 + n % 97, threads=threads)


# ---- 3. radius sets larger than the list -------------------------------------------------------------------------------------
OVERFLOW_ROWS = []
for _k, _kern in (("star", "scan"), ("informed", "scan"), ("star", "wide"), ("informed", "wide")):
    OVERFLOW_ROWS.append(row(_k, 256, 256, 2000, dict(kernel=_kern), env={"RRTK_PLAN_IMPL": _kern}, r=120.0, rg=10.0))
for _K in (8, 16):
    OVERFLOW_ROWS.append(row("star", 256, 256, 2000, dict(kernel="grid", K=_K), env={"RRTK_GRID_K": _K}, r=120.0))
# a 32-entry list: overflows at small n
OVERFLOW_ROWS += [
    row("star", 128, 128, 300, dict(kernel="scan", list_cap=32), env={"RRTK_PLAN_CAP": 32, "RRTK_PLAN_IMPL": "scan"}, r=40.0),
    row("informed", 128, 128, 300, dict(kernel="scan", list_cap=32), env={"RRTK_PLAN_CAP": 32}, r=40.0, rg=10.0),
    row("star", 128, 128, 300, dict(kernel="grid", K=8, list_cap=32), env={"RRTK_PLAN_CAP": 32, "RRTK_GRID_K": 8}, r=40.0),
    row("star", 128, 128, 300, dict(kernel="grid", K=16, list_cap=32), env={"RRTK_PLAN_CAP": 32}, r=40.0),
]


@pytest.mark.parametrize("kind,W,H,n,env,threads,expect,plans,r,rg", OVERFLOW_ROWS)
def test_list_overflow(monkeypatch, request, kind, W, H, n, env, threads, expect, plans, r, rg):
    """A radius r so large that some radius sets exceed the kernel's candidate list: the exact brute-force (scan), sparse (wide)
    or all-slot (bucket) path runs, and the assertion on the oracle's tree shows that it did."""
    set_env(monkeypatch, env)
    shape = checked_shape(request.node.callspec.id, kind, W, H, n, threads, expect)
    wants = perlin_plans(kind, W, H, n, r, rg, plans, seed=300 + n % 89, threads=threads)
    most = max(max_radius_set(w[0], w[3]["j"], r) for w in wants)
    assert most > shape["list_cap"], f"largest radius set {most} fits the {shape['list_cap']}-entry list: the overflow path did not run"


# ---- 4. key-range limits in the worst geometry ---------------------------------------------------------------------------------
def corner_stream(W, H, n, seed):
    """Samples for an empty W x H grid: the four corners first, then corners, cells near a corner and uniform cells."""
    rng = np.random.default_rng(seed)
    cx = np.array([0, W - 1, W - 1, 0])
    cy = np.array([0, H - 1, 0, H - 1])
    c = rng.integers(0, 4, n)
    near = np.stack([np.abs(cx[c] - rng.integers(0, min(W, 24), n)), np.abs(cy[c] - rng.integers(0, min(H, 24), n))], 1)
    uni = np.stack([rng.integers(0, W, n), rng.integers(0, H, n)], 1)
    mode = rng.random(n)
    s = np.where((mode < 0.15)[:, None], np.stack([cx[c], cy[c]], 1), np.where((mode < 0.6)[:, None], near, uni))
    s[:4] = np.stack([cx, cy], 1)[[1, 2, 3, 0]]               # far corner, the other two, the root's own cell
    return s


def corner_plans(kind, W, H, n, threads=0, seed=0):
    """Root in corner (0, 0), goal in the opposite corner; r at least the diagonal (every threshold clamped) and r just below
    it (every vertex but the opposite corner's is a member)."""
    diag = math.hypot(W - 1, H - 1)
    og = np.zeros((1, W, H), dtype=np.uint8)
    starts, goals = [np.array([0, 0])], [np.array([W - 1, H - 1])]
    samples = corner_stream(W, H, n, seed)[None]
    for r in (math.ceil(diag) + 1.0, max(diag - 0.5, 0.0)):
        plan_vs_oracle(kind, og, starts, goals, samples, r, 2.0, threads, seed)


KEY_ROWS = []
for _k in ("standard", "star", "informed"):
    KEY_ROWS += [
        # scan: (2 side^2) << sbits <= 2^29 at 2896 / 2048 / 1448 cells a side for 1 / 2 / 3-4 words; one cell more -> wide
        row(_k, 2896, 2896, 2000, scan(64, 1, 4, sbits=5)),
        row(_k, 2897, 2897, 2000, dict(kernel="wide")),
        row(_k, 2048, 2048, 4500, scan(128, 2, 1, sbits=6)),
        row(_k, 2049, 2049, 4500, dict(kernel="wide")),
        row(_k, 1448, 1448, 17000, scan(256, 3, 1, sbits=7)),
        row(_k, 1449, 1449, 17000, dict(kernel="wide")),
        row(_k, 1448, 1448, 30000, scan(256, 4, 4, sbits=7)),
        # non-square at the limit (RRTStandard / RRTStar would take the bucket kernel here: forced onto the scan kernel)
        row(_k, 2896, 8, 1500, scan(64, 1, 4, sbits=5), env={"RRTK_PLAN_IMPL": "scan"}),
        row(_k, 8, 2897, 1500, dict(kernel="wide"), env={"RRTK_PLAN_IMPL": "scan"}),
        # the 16384-cell limit of the packed vertex format
        row(_k, 16384, 4, 2000, dict(kernel="wide", grid_smem=0), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 0}),
        row(_k, 16384, 4, 2000, dict(kernel="wide", grid_smem=1), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 1}),
        row(_k, 4, 16384, 2000, dict(kernel="wide", grid_smem=0), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 0}),
        row(_k, 4, 16384, 2000, dict(kernel="wide", grid_smem=1), env={"RRTK_PLAN_IMPL": "wide", "RRTK_GRID_SMEM": 1}),
    ]
for _k in ("standard", "star"):
    KEY_ROWS += [
        # bucket: one-word (d2 << kb | id) keys while d2max < 2^(32 - kb) - 1
        row(_k, 512, 512, 8191, dict(kernel="grid", kb=13, key_words=1)),    # d2max 522242 < 524287
        row(_k, 512, 512, 8192, dict(kernel="grid", kb=0, key_words=2)),     # kb = 14: 522242 >= 262143
        row(_k, 512, 513, 8190, dict(kernel="grid", kb=13, key_words=1)),    # d2max 523265, and n + 1 at the 13-bit id limit
        row(_k, 512, 514, 8190, dict(kernel="grid", kb=0, key_words=2)),     # d2max 524290 >= 524287
        # 16384 cells: ids still fit (14 + 2 bits of coordinates), keys take two words
        row(_k, 16384, 4, 2000, dict(kernel="grid", key_words=2)),
        row(_k, 4, 16384, 2000, dict(kernel="grid", key_words=2)),
    ]


@pytest.mark.parametrize("kind,W,H,n,env,threads,expect,plans,r,rg", KEY_ROWS)
def test_key_range_limits(monkeypatch, request, kind, W, H, n, env, threads, expect, plans, r, rg):
    set_env(monkeypatch, env)
    checked_shape(request.node.callspec.id, kind, W, H, n, threads, expect)
    corner_plans(kind, W, H, n, threads, seed=W * 7 + H + n)


@pytest.mark.parametrize("W,H", [(16385, 4), (4, 16385), (16385, 16385)])
def test_grid_beyond_the_vertex_format_is_refused_before_launch(W, H):
    db = batch.DeviceBatch("star", W, H, 300, 50.0).set_worlds_host(np.zeros((1, W, H), dtype=np.uint8))
    db.set_plans(batch.make_desc([0], [[0, 0]], [[W - 1, H - 1]]))
    db.set_samples_host(np.zeros((1, 300, 2), dtype=np.int16))
    for t in db.out.values():
        if t is not None:
            t.fill_(-7)
    with pytest.raises(ValueError, match="out of range"):
        db.run()
    with pytest.raises(ValueError, match="out of range"):
        db.footprint()
    res = db.download()
    assert (res.stats == -7).all() and (res.parent == -7).all()          # nothing was launched


# ---- 5. the edge cases on every kernel -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = _lib.Context()
    yield c
    c.close()


@pytest.mark.parametrize("impl,kind", [("grid", "standard"), ("grid", "star"), ("scan", "standard"), ("scan", "star"),
                                       ("scan", "informed"), ("wide", "standard"), ("wide", "star"), ("wide", "informed")])
def test_edge_cases_on_every_kernel(ctx, monkeypatch, impl, kind):
    set_env(monkeypatch, {"RRTK_PLAN_IMPL": impl})
    ran = {}
    for case in edge_cases():
        name, og, n = case[:3]
        ran[name] = checked_shape(f"edge-{impl}-{kind}-{name}", kind, og.shape[0], og.shape[1], n)["kernel"]
        run_edge_case(ctx, kind, case)
    # the bucket kernel needs a bucket per vertex beside the root (nbx * nby + 1 <= n): one bucket covers these grids, so
    # only n = 1 falls back to the scan kernel
    want = {name: ("scan" if impl == "grid" and n == 1 else impl) for name, _, n, *_ in edge_cases()}
    assert ran == want


# ---- 6. a seeded random sweep --------------------------------------------------------------------------------------------------
def _sweep_cases(count=40, seed=20261020):
    rng = np.random.default_rng(seed)
    sides = [1, 2, 5, 31, 64, 97, 128, 300, 513, 1000, 1500]
    cases = []
    while len(cases) < count:
        kind = ["standard", "star", "informed"][rng.integers(3)]
        W, H = int(rng.choice(sides)), int(rng.choice(sides))
        n = int(rng.choice([1, 2, 40, 255, 256, 511, 700, 1500, 2047, 2600, 4100, 5200]))
        r = float(rng.choice([0.0, 1.5, 7.5, 30.0, 77.25, 1e4]))
        rg = float(rng.choice([0.0, 2.5, 10.0, 40.0]))
        impl = str(rng.choice(["auto", "auto", "grid", "scan", "wide"]))
        threads = int(rng.choice([0, 0, 64, 128, 160, 256, 512]))
        K = int(rng.choice([4, 8, 16]))
        if W * H < 4 or n * W * H > 4e9:
            continue
        cases.append(pytest.param(len(cases), kind, W, H, n, r, rg, impl, threads, K,
                                  id=f"{len(cases):02d}-{kind}-{W}x{H}-n{n}-r{r:g}-rg{rg:g}-{impl}-threads{threads}-K{K}"))
    return cases


@pytest.mark.parametrize("i,kind,W,H,n,r,rg,impl,threads,K", _sweep_cases())
def test_random_sweep(monkeypatch, request, i, kind, W, H, n, r, rg, impl, threads, K):
    env = {"RRTK_PLAN_K": K}
    if impl != "auto":
        env["RRTK_PLAN_IMPL"] = impl
    if K in (8, 16):
        env["RRTK_GRID_K"] = K
    set_env(monkeypatch, env)
    checked_shape(request.node.callspec.id, kind, W, H, n, threads)
    rng = np.random.default_rng(9000 + i)
    if min(W, H) >= 16:
        og = worlds.perlin_occupancygrid(W, H, seed=9000 + i).astype(np.uint8)
    else:
        og = (rng.random((W, H)) < 0.15).astype(np.uint8)
    free = np.argwhere(og == 0)
    if len(free) < 2:
        og[:] = 0
        free = np.argwhere(og == 0)
    a, b = rng.choice(len(free), 2, replace=False)
    samples = free[rng.integers(0, len(free), n)]
    plan_vs_oracle(kind, og[None], [free[a]], [free[b]], samples[None], r, rg, threads, seed=9000 + i)


# ---- 1. the restatement itself, on every row -----------------------------------------------------------------------------------
DISPATCH_ONLY_ROWS = [
    row("star", 1024, 1024, 50000, dict(kernel="wide", T=128)),           # T = 512 with four words does not fit a star tree
    row("informed", 1024, 1024, 50000, dict(kernel="wide", T=128)),
    row("star", 512, 512, 5000, dict(kernel="grid", K=16, kb=13)),        # cfg3
    row("informed", 1024, 1024, 20000, scan(256, 3, 2, two_per_sm=1)),    # cfg4
    row("star", 1024, 1024, 4094, dict(kernel="grid")),                   # 1024^2: bucket ids end at n = 4094
    row("star", 1024, 1024, 4095, scan(128, 1, 4)),
    row("star", 1024, 1024, 255, scan(64, 1, 1)),                         # n < 256 stays with the scan kernel
    row("star", 1024, 1024, 255, dict(kernel="grid"), env={"RRTK_PLAN_IMPL": "grid"}),
    row("star", 512, 512, 5000, scan(128, 2, 1), env={"RRTK_GRID_K": 4}),  # no bucket kernel with 4 samples per round
    row("star", 512, 512, 6000, scan(160, 2, 1), env={"RRTK_PLAN_T": 160}),
    row("star", 512, 512, 5000, scan(256, 1, 4), threads=256),
]


@pytest.mark.parametrize("kind,W,H,n,env,threads,expect,plans,r,rg",
                         REGIME_ROWS + OVERFLOW_ROWS + KEY_ROWS + DISPATCH_ONLY_ROWS)
def test_dispatch_restatement(monkeypatch, request, kind, W, H, n, env, threads, expect, plans, r, rg):
    """The Python restatement of the dispatch equals the library on every table row (kernel and shared memory), and each row
    sits in the regime it is meant for."""
    set_env(monkeypatch, env)
    checked_shape(request.node.callspec.id, kind, W, H, n, threads, expect)
