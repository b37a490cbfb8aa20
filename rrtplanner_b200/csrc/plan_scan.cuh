// K7 (default form): one thread block per plan, K samples per round, packed-key scan.
//
// Replaces the three plan() loops of the reference (rrt.py:418-437, 498-548, 690-748), go2goal
// (rrt.py:284-332) and the primitives they call (near :131-155, within :157-181, collisionfree
// :183-229, default costfn :70-78, informed sampler :579-633).  Results are identical to the
// reference run on the same sample stream with its two unstable argsorts pinned to "lowest index
// first" (SURVEY.md section 8(c)); tests/test_gpu_parity.py checks that bit for bit.
//
// The reference's loop is sequential (iteration i sees the tree iteration i-1 left).  A round takes
// the next K samples and keeps that semantics exactly:
//
//   scan     all threads, brute force over the whole tree (north star: no spatial index).  The tree
//            lives in shared memory as packed vertices x | y << 16, laid out so that thread t owns
//            the vertices v = row * T + t ("column t"): one LDS.128 = rows 4s .. 4s+3 of the
//            column, conflict free, and the filled part of the tree is always spread evenly over
//            the threads.  For vertex v and sample q the scan needs d2 = |v - q|^2 only up to a
//            per-sample constant, so it evaluates
//                key = S * (|v|^2 - 2 v.q) + row - S * (r^2 - |q|^2)          S = 2^sbits > row
//            with two IMADs (S |v|^2 + row is per vertex, shared by the K samples; -2 S q per
//            sample), then  key < 0  <=>  d2 < r^2  (one funnel shift appends the sign bit to the
//            thread's membership word) and  min key  <=>  (min d2, lowest row)  (half a 3-input
//            minimum per pair).  Everything is exact integer arithmetic: |key| < 2^31 is checked
//            on the host as (2 side^2) << sbits <= 2^29 (grids up to 2896 / 2048 / 1448 cells a side
//            for 1 / 2 / 3-4 membership words); larger grids use the 32-bit-distance kernel of plan_wide.cu.
//   barrier
//   owner    the warps take the samples one at a time, first come first served (a sample costs
//            anything between a duplicate test and several walks), and evaluate each against the
//            round-start tree: combine the per-warp minima, duplicate test, walk nearest -> sample
//            (rrt.py:424/506/706; its first grid word and the nearest vertex's cost are requested
//            before the radius set is compacted), FP64 cost via the nearest vertex, compaction of
//            the membership words into a dense list, choose-parent (rrt.py:510-521) cheapest first:
//            up to three members per lane are costed together, the cheapest one of the warp that beats
//            the nearest vertex is walked, and the first free one wins (ties: lowest index).
//   barrier
//   commit   one warp (the duty rotates, see cw) replays the K results in sample order against the vertices accepted earlier in
//            the same round (one per lane): equal cell -> duplicate; inside the radius -> extra
//            candidate (cost, walk); strictly nearer than the recorded nearest vertex, or a change
//            of the informed sampler's state -> the round is cut there and the remaining samples
//            are redone next round (rare).  Accepted vertices are appended in order, and the next
//            round's samples (free-space stream or informed ellipse) are staged.
//   barrier
//
// so every decision is the one the sequential loop would take.  The reference's "rewire" block
// (rrt.py:532-546, 732-742) tests vcosts[vn] + d < vcosts[vn] and can never fire with the default
// cost function (oracle/rrt_oracle.py counts it: always 0), so it has no device counterpart.
#pragma once
#include <type_traits>

#include "plan_common.cuh"

namespace rrtk {

constexpr int kKeyDead = 0x20000400;        // key of a masked-out slot: above every real key and every threshold
constexpr int kKeyNever = -0x20000400;      // threshold of an inactive sample: below every real key

// position of vertex v in the on-chip tree: quad (step, column) holds rows 4*step .. 4*step+3
template <int T>
__device__ __forceinline__ int tree_slot(int v)
{
    const int row = v / T, col = v - row * T;
    return ((((row >> 2) * T) + col) << 2) | (row & 3);
}

#ifndef RRTK_MINB128
#define RRTK_MINB128 7
#endif
#ifndef RRTK_MINB256
#define RRTK_MINB256 3
#endif
template <int KIND, int K, int T>
struct ScanCfg {
    // resident blocks per SM the register allocation aims for
    static constexpr int kMinBlocks = (T <= 64) ? 12 : (T <= 128) ? RRTK_MINB128 : (T <= 160) ? 5 : (T <= 256) ? RRTK_MINB256 : 1;
};

// MB: resident blocks per SM the registers are bounded for.  Blocks of 256 threads come in two builds: 3 per SM (80 registers) and,
// for trees so large that shared memory admits only two blocks anyway (cfg4: n = 20000), 2 per SM with 128 registers -- the
// informed kernel spills at 80 (cfg4: 2.27 k -> 2.63 k plans/s).
template <int KIND, int K, int T, int MB = ScanCfg<KIND, K, T>::kMinBlocks>
__global__ void __launch_bounds__(T, MB) plan_scan_kernel(PlanParams P)
{
    constexpr int NW = T / 32;
    static_assert(T % 32 == 0 && K <= 16 && K >= 1, "block shape");
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ int2 s_near[K][NW];                    // [sample][warp] (min key >> sbits, vertex)
    __shared__ SampleRec s_rec[K];
    __shared__ RoundSummary s_sum;
    __shared__ short2 s_q[K];                         // samples of the round
    __shared__ int4 s_qk[K];                          // their scan constants (ax, ay, thr, 0), staged with the samples
    __shared__ int s_next;                            // owner phase: next sample nobody has taken yet
    __shared__ double s_qc[K];                        // informed: cbest each ellipse sample was drawn with
    __shared__ unsigned long long s_goalc;
    __shared__ int s_goalv;
    __shared__ unsigned long long s_checks, s_cells;

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int plan = blockIdx.x;
    const int n = P.n;
    const int sbits = P.sbits;
    const int S = 1 << sbits;
    const int cap = P.list_cap;
    const int HW = P.hit_words;

    const int npts = 4 * T * P.steps_max;
    uint32_t *s_pts = smem;                                               // npts words
    // thread-private membership words: [HW - 1][K][T] full words, then the last word of every (sample, thread) stored in
    // tail_bytes bytes -- a tree of n + 1 vertices fills only its first rows (8 of 32 for n = 5000, T = 128), and the 3 KB
    // this saves are what lets an eighth plan fit on the SM
    uint32_t *s_hits = smem + npts;
    const int tailb = P.tail_bytes;                                       // 1, 2 or 4
    uint8_t *s_tail = reinterpret_cast<uint8_t *>(s_hits + (HW - 1) * K * T);
    uint16_t *s_list = reinterpret_cast<uint16_t *>(KIND == RRTK_STANDARD ? (uint8_t *)s_hits : s_tail + ((tailb * K * T + 3) & ~3));   // [NW][cap]: one list per owner warp
    auto hit_store = [&](int w, int k, int t, uint32_t word) {            // word: left-aligned (row r of the word in bit 31 - r)
        if (w < HW - 1 || tailb == 4) s_hits[(w * K + k) * T + t] = word;
        else if (tailb == 1) s_tail[k * T + t] = (uint8_t)(word >> 24);
        else reinterpret_cast<uint16_t *>(s_tail)[k * T + t] = (uint16_t)(word >> 16);
    };
    auto hit_load = [&](int w, int k, int t) -> uint32_t {
        if (w < HW - 1 || tailb == 4) return s_hits[(w * K + k) * T + t];
        if (tailb == 1) return (uint32_t)s_tail[k * T + t] << 24;
        return (uint32_t)reinterpret_cast<uint16_t *>(s_tail)[k * T + t] << 16;
    };

    const rrtk_plan_desc *dsc = P.plans + plan;
    const uint32_t *gbits = P.bits + (size_t)dsc->world * P.words_per_grid;
    const int sx = dsc->start_x, sy = dsc->start_y, gx = dsc->goal_x, gy = dsc->goal_y;
    const uint32_t startp = pack_xy(sx, sy);

    double *cost = P.cost + (size_t)plan * (n + 1);
    int *parent = P.parent + (size_t)plan * (n + 1);
    const short2 *samples = P.samples + (size_t)plan * n;
    const double2 *balls = (KIND == RRTK_INFORMED && P.balls) ? P.balls + (size_t)plan * n : nullptr;
    double *ell_c = (KIND == RRTK_INFORMED) ? P.ell_c + (size_t)plan * (n + 1) : nullptr;
    const uint32_t r2x = P.r2_excl;

    // scan constants of a sample (see the header): key = vx * ax + vy * ay + (S |v|^2 + row),  key < thr  <=>  d2 < r2x
    auto scan_consts = [&](short2 q, bool act) {
        const int qq = q.x * q.x + q.y * q.y;
        long long t = (long long)S * ((long long)r2x - qq);
        t = t > (long long)kKeyDead ? (long long)kKeyDead : t;
        int thr = (act && KIND != RRTK_STANDARD) ? (int)t : kKeyNever;
        if (KIND == RRTK_STANDARD && act) thr = 0;                            // any constant: bits unused
        return make_int4(act ? -2 * S * q.x : 0, act ? -2 * S * q.y : 0, thr, 0);
    };
    for (int i = tid; i < npts; i += T) s_pts[i] = startp;                // slot 0 = the root; the rest is never read unmasked
    if (tid < K) {
        const short2 q0 = samples[min(tid, n - 1)];
        s_q[tid] = q0;
        s_qk[tid] = scan_consts(q0, tid < min(min(K, n), 1));                 // first round: j = 1 -> one sample
        if (tid == 0) s_next = NW;
    }
    if (tid == 0) { s_checks = s_cells = 0ull; cost[0] = 0.0; parent[0] = -1; }
    if (KIND == RRTK_INFORMED)
        for (int i = tid; i <= n; i += T) ell_c[i] = CUDART_NAN;
    __syncthreads();

    GlobalGrid gg{gbits};
    const int TY = P.TY;
#define WALK(ax_, ay_, bx_, by_) warp_first_hit(gg, TY, ax_, ay_, bx_, by_, lane)

    // block-uniform state, replicated in every thread (refreshed from s_sum after each round)
    int j = 1, it0 = 0, kwant = 1;
    // The commit duty rotates over the warps: warp w of every resident block sits on scheduler w mod 4 of the SM, so a
    // fixed commit warp would load one scheduler with all the serial work of every block (-DRRTK_FIXED_COMMIT: warp 0).
    int cw = 0;
    __shared__ unsigned long long s_cnt[4];           // commit-phase counters of all warps, summed at the end
    if (tid < 4) s_cnt[tid] = 0ull;
    bool have_sol = false;              // INFORMED: running least_cost over vsoln (rrt.py:627-633)
    int vsol = 0;
    double csol = 0.0;
    long long first_sol = -1;
    // counters kept by the committing warp (every warp takes its turn) / per warp (walks)
    long long ell_iters = 0, nn_pairs = 0, ring_members = 0, accepted = 0;
    unsigned my_checks = 0, my_cells = 0;

    // -DRRTK_PHASE_CLOCKS (experiment builds, scripts/phase_clocks.py): cycles per phase in spare stats slots
#ifdef RRTK_PHASE_CLOCKS
    long long clk_scan = 0, clk_owner = 0, clk_commit = 0, clk_ownwork = 0, rounds = 0;
#define PHASE_T(var) const long long var = clock64()
#define PHASE_ADD(acc, a, b) acc += (b) - (a)
#else
#define PHASE_T(var)
#define PHASE_ADD(acc, a, b)
#endif
    while (it0 < n) {
        PHASE_T(t_0);
        if (KIND != RRTK_INFORMED && j == n) break;                       // tree full: every later sample is rejected
        if (KIND == RRTK_INFORMED && have_sol && balls == nullptr) break; // probe run: stop at first solution
        const bool ellipse_mode = (KIND == RRTK_INFORMED) && have_sol;
        // Samples of this round.  How many a round takes changes the speed, never the result (the commit replays them in order):
        // the count doubles after every round that consumed all of its samples and halves after a round that was cut short (but
        // not below 1 + j / 8) -- few while the tree is tiny and a new vertex is often the nearest one to the next sample, K once
        // it has grown, and K as well for a plan whose tree does not grow at all (a walled-in start: 5000 one-sample rounds made such plans the
        // stragglers of every batch, 19 M cycles against a mean of 13.7 M at 444 plans per launch).
        const int kact = min(min(K, n - it0), kwant);

        // ---- scan: nearest + radius-set bits for K samples over vertices 0 .. j-1 ---------------
        const int rows = (j + T - 1) / T;
        const int steps = (rows + 3) >> 2;
        const int nwords = (steps + 7) >> 3;
        // fold the running minima of a warp into (distance key, vertex) per sample; col = the column each lane scanned
        auto fold_near = [&](int col, const int (&thr)[K], const int (&best)[K], int2 (*dst)[NW]) {
#pragma unroll
            for (int k = 0; k < K; ++k) {   // warp minimum, lowest index among equals
                const bool any = best[k] != 0x7fffffff;
                const int key = best[k] + thr[k];
                const int dp = any ? (key >> sbits) : 0x7fffffff;
                const int v = (key & (S - 1)) * T + col;
                const int wd = __reduce_min_sync(RRTK_FULL, dp);
                const unsigned wi = __reduce_min_sync(RRTK_FULL, (any && dp == wd) ? (unsigned)v : 0xffffffffu);
                if (lane == 0) dst[k][warp] = make_int2(wd, (int)wi);
            }
        };
        {
            int ax[K], ay[K], thr[K], best[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int4 c = s_qk[k];                                       // staged by the commit warp for this round's kact
                ax[k] = c.x; ay[k] = c.y; thr[k] = c.z;
                best[k] = 0x7fffffff;
            }
            // column tid of the tree, one quad (LDS.128 = rows 4s .. 4s+3) per step; the last, partly empty quad is masked
            // and done in halves (rows 4s, 4s+1 always; 4s+2, 4s+3 only if the tree reaches them)
            const uint4 *q4 = reinterpret_cast<const uint4 *>(s_pts) + tid;
            auto pair_step = [&](const uint32_t w0, const uint32_t w1, int row0, uint32_t (&h)[K], auto masked_c) {
                constexpr bool masked = decltype(masked_c)::value;
                int vx[2], vy[2], nvs[2];
                const uint32_t wv[2] = {w0, w1};
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    vx[u] = px(wv[u]); vy[u] = py(wv[u]);
                    nvs[u] = (vx[u] * vx[u] + vy[u] * vy[u]) * S + (row0 + u);
                    if (masked && (row0 + u) * T + tid >= j) { vx[u] = 0; vy[u] = 0; nvs[u] = kKeyDead; }
                }
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int d0 = vx[0] * ax[k] + (vy[0] * ay[k] + nvs[0]) - thr[k];
                    const int d1 = vx[1] * ax[k] + (vy[1] * ay[k] + nvs[1]) - thr[k];
                    if (KIND != RRTK_STANDARD) {
                        h[k] = __funnelshift_l((uint32_t)d0, h[k], 1);
                        h[k] = __funnelshift_l((uint32_t)d1, h[k], 1);
                    }
                    best[k] = min(best[k], min(d0, d1));
                }
            };
            for (int w = 0; w < nwords; ++w) {          // one membership word = 32 rows = 8 quads; row r of the word -> bit 31 - r
                uint32_t h[K];
#pragma unroll
                for (int k = 0; k < K; ++k) h[k] = 0u;
                const int s_end = min(steps, 8 * w + 8);
                const int s_full = (s_end == steps) ? s_end - 1 : s_end;
                int s = 8 * w;
                for (; s < s_full; ++s) {
                    const uint4 q = q4[s * T];
                    pair_step(q.x, q.y, 4 * s, h, std::false_type{});
                    pair_step(q.z, q.w, 4 * s + 2, h, std::false_type{});
                }
                int nrow = 4 * (s - 8 * w);
                if (s < s_end) {
                    const uint4 q = q4[s * T];
                    pair_step(q.x, q.y, 4 * s, h, std::true_type{});
                    nrow += 2;
                    if (rows > 4 * s + 2) { pair_step(q.z, q.w, 4 * s + 2, h, std::true_type{}); nrow += 2; }
                }
                if (KIND != RRTK_STANDARD) {
#pragma unroll
                    for (int k = 0; k < K; ++k) hit_store(w, k, tid, h[k] << (32 - nrow));   // 2 <= nrow <= 32
                }
            }
            fold_near(tid, thr, best, s_near);
        }
        __syncthreads();                                                   // ---- barrier: scan results visible
        PHASE_T(t_1);

        // the stream samples the next round can start with (it0 + consumed + k, consumed <= kact <= K): requested by the
        // committing warp before its owner work, so that the load is long done when the commit phase stages them
        short2 ahead = make_short2(0, 0);
        if (warp == cw && lane < 2 * K) ahead = samples[min(it0 + lane, n - 1)];

        // ---- owner phase: warp (k mod NW) evaluates sample k against the round-start tree ---------
        // a sample costs anything between a duplicate test and several walks: warps take the next free one as they finish
        for (int k = warp; k < K;) {
            if (k >= kact) {
                if (lane == 0) s_rec[k].flags = 0;
                int nk = 0;
                if (lane == 0) nk = atomicAdd(&s_next, 1);
                k = __shfl_sync(RRTK_FULL, nk, 0);
                continue;
            }
            const short2 smp = s_q[k];
            const int x = smp.x, y = smp.y;
            uint32_t bd;
            int vnear;
            {
                const int2 e = lane < NW ? s_near[k][lane] : make_int2(0x7fffffff, 0x7fffffff);
                const int md = __reduce_min_sync(RRTK_FULL, e.x);
                vnear = (int)__reduce_min_sync(RRTK_FULL, e.x == md ? (unsigned)e.y : 0xffffffffu);
                bd = (uint32_t)(md + x * x + y * y);
            }
            // `sampled` holds accepted samples only, not xstart (rrt.py:410,426): a sample on the root's cell is a
            // duplicate only if some vertex >= 1 sits there too (the scan reports the lowest index)
            bool dup = bd == 0 && vnear >= 1;
            if (bd == 0 && vnear == 0) {
                bool f = false;
                for (int v = 1 + lane; v < j; v += 32) f |= s_pts[tree_slot<T>(v)] == startp;
                dup = __any_sync(RRTK_FULL, f);
            }
            const uint32_t pnear = s_pts[tree_slot<T>(vnear)];
            int flags = 1 | (dup ? 2 : 0);
            double c0 = 0.0, wc = CUDART_INF;
            int wv = 0x7fffffff, ring = 0;
            // the reference walks nearest -> sample before looking at the duplicate test
            // (rrt.py:424-425 / 506-507 / 706-707); the verdicts are independent, so skip the walk
            if (!dup) {
                // long-latency operands first: the nearest vertex's cost and the first chunk of the walk
                // nearest -> sample are in flight while the radius set is compacted
                const double cnear = cost[vnear];
                WalkState wk = walk_begin(gg, TY, px(pnear), py(pnear), x, y, lane);
                int total = 0;
                uint16_t *list = s_list + warp * cap;
                if (KIND != RRTK_STANDARD) {
                    // membership words of this sample: nwords rows of T thread-private words
                    int mine = 0;
                    for (int w = 0; w < nwords; ++w) {
#pragma unroll
                        for (int c = 0; c < T / 32; ++c) mine += __popc(hit_load(w, k, 32 * c + lane));
                    }
                    total = __reduce_add_sync(RRTK_FULL, mine);
                    if (total <= cap) {
                        // compaction: exclusive prefix of the per-lane counts, then every lane lists its members
                        int incl = mine;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const int t = __shfl_up_sync(RRTK_FULL, incl, o);
                            if (lane >= o) incl += t;
                        }
                        uint16_t *out = list + (incl - mine);
                        for (int w = 0; w < nwords; ++w) {
#pragma unroll
                            for (int c = 0; c < T / 32; ++c) {
                                uint32_t bits = hit_load(w, k, 32 * c + lane);
                                const int vtop = (32 * w + 31) * T + 32 * c + lane;      // bit b of the word <-> row 32 w + 31 - b
                                while (bits) {
                                    const int b = 31 - __clz(bits);
                                    bits ^= 1u << b;
                                    *out++ = (uint16_t)(vtop - b * T);
                                }
                            }
                        }
                        __syncwarp();
                    }
                }
                const int hit = walk_finish(gg, TY, wk, lane);
                my_checks += 1; my_cells += cells_tested(hit);
                if (hit < 0) {
                    flags |= 4;
                    c0 = reach_cost(cnear, bd);
                    if (KIND != RRTK_STANDARD) {
                        ring = total;
                        if (total <= cap) {
                            // choose-parent (rrt.py:510-521), cheapest first: up to three candidates per lane have their costs
                            // loaded and evaluated together; the cheapest live one of the warp is walked, and the first
                            // free one is the minimum over (cost, index) of everything that beats the nearest vertex.
                            // (the list is in lane order, not index order: every tie is resolved on the vertex index)
                            for (int base = 0; base < total; base += 96) {
                                int cv[3];
                                uint32_t cp[3];
                                unsigned long long ck[3];                     // cost bits; ~0 = not a candidate
                                double ccv[3];
                                const int left = total - base;                // slots u with 32 u >= left are empty for every lane
#pragma unroll
                                for (int u = 0; u < 3; ++u) {
                                    ck[u] = ~0ull; cv[u] = 0; cp[u] = 0u; ccv[u] = CUDART_INF;
                                    if (32 * u < left) {
                                        const int idx = base + 32 * u + lane;
                                        const bool has = idx < total;
                                        cv[u] = has ? (int)list[idx] : 0;
                                        cp[u] = s_pts[tree_slot<T>(cv[u])];
                                        if (has) ccv[u] = cost[cv[u]];
                                    }
                                }
#pragma unroll
                                for (int u = 0; u < 3; ++u) {
                                    if (32 * u < left) {
                                        const double cn = reach_cost(ccv[u], dist2(cp[u], x, y));
                                        const bool live = cn < c0 && (cn < wc || (cn == wc && cv[u] < wv));
                                        if (live) ck[u] = (unsigned long long)__double_as_longlong(cn);   // positive doubles order like their bits
                                    }
                                }
                                for (;;) {
                                    // this lane's cheapest live candidate, lowest vertex index among equal costs
                                    unsigned long long bk = ck[0];
                                    int bu = 0, bvx = cv[0];
                                    if (ck[1] < bk || (ck[1] == bk && cv[1] < bvx)) { bk = ck[1]; bu = 1; bvx = cv[1]; }
                                    if (ck[2] < bk || (ck[2] == bk && cv[2] < bvx)) { bk = ck[2]; bu = 2; bvx = cv[2]; }
                                    const uint32_t hi = (uint32_t)(bk >> 32);
                                    const uint32_t mhi = warp_min_u32(hi);
                                    if (mhi == 0xffffffffu) break;                    // nothing left that beats the incumbent
                                    const uint32_t lo = (hi == mhi) ? (uint32_t)bk : 0xffffffffu;
                                    const uint32_t mlo = warp_min_u32(lo);
                                    const uint32_t vv = (hi == mhi && lo == mlo) ? (uint32_t)bvx : 0xffffffffu;
                                    const uint32_t mv = warp_min_u32(vv);
                                    const int src = __ffs(__ballot_sync(RRTK_FULL, vv == mv)) - 1;
                                    const uint32_t bpx = bu == 0 ? cp[0] : bu == 1 ? cp[1] : cp[2];
                                    const uint32_t pp = __shfl_sync(RRTK_FULL, bpx, src);
                                    const int h = WALK(px(pp), py(pp), x, y);
                                    my_checks += 1; my_cells += cells_tested(h);
                                    if (h < 0) { wc = __hiloint2double((int)mhi, (int)mlo); wv = (int)mv; break; }
                                    if (lane == src) {
                                        if (bu == 0) ck[0] = ~0ull; else if (bu == 1) ck[1] = ~0ull; else ck[2] = ~0ull;
                                    }
                                }
                            }
                        } else {
                            // very large radius sets: test every vertex directly, 32 per step; while one beats the
                            // incumbent, walk the cheapest
                            auto consider = [&](bool has, int v, uint32_t p, double cn) {
                                bool live = has && cn < c0;
                                for (;;) {
                                    const bool cand = live && (cn < wc || (cn == wc && v < wv));
                                    if (!__any_sync(RRTK_FULL, cand)) break;
                                    const uint32_t hi = cand ? (uint32_t)__double2hiint(cn) : 0xffffffffu;
                                    const uint32_t mhi = warp_min_u32(hi);
                                    const uint32_t lo = (cand && hi == mhi) ? (uint32_t)__double2loint(cn) : 0xffffffffu;
                                    const uint32_t mlo = warp_min_u32(lo);
                                    const uint32_t vv = (cand && hi == mhi && lo == mlo) ? (uint32_t)v : 0xffffffffu;
                                    const uint32_t mv = warp_min_u32(vv);
                                    const int src = __ffs(__ballot_sync(RRTK_FULL, vv == mv && mv != 0xffffffffu)) - 1;
                                    const uint32_t pp = __shfl_sync(RRTK_FULL, p, src);
                                    const int h = WALK(px(pp), py(pp), x, y);
                                    my_checks += 1; my_cells += cells_tested(h);
                                    if (h < 0) { wc = __hiloint2double((int)mhi, (int)mlo); wv = (int)mv; }
                                    else if (lane == src) live = false;
                                }
                            };
                            for (int base = 0; base < j; base += 32) {
                                const int v = base + lane;
                                const uint32_t p = s_pts[tree_slot<T>(v < j ? v : 0)];
                                const uint32_t dd = dist2(p, x, y);
                                const bool has = v < j && dd < r2x;
                                double cn = CUDART_INF;
                                if (has) cn = reach_cost(cost[v], dd);
                                consider(has, v, p, cn);
                            }
                        }
                    }
                }
            }
            if (lane == 0) {
                SampleRec r;
                r.pnew = pack_xy(x, y); r.bd = bd; r.vnear = vnear; r.flags = flags; r.bv = wv; r.ring = ring;
                r.c0 = c0; r.bc = wc; r.ell = ellipse_mode ? s_qc[k] : 0.0;
                s_rec[k] = r;
            }
            {
                int nk = 0;
                if (lane == 0) nk = atomicAdd(&s_next, 1);
                k = __shfl_sync(RRTK_FULL, nk, 0);
            }
        }
        PHASE_T(t_1b);
        __syncthreads();                                                   // ---- barrier: K results visible
        PHASE_T(t_2);

        // ---- commit phase: warp 0 replays the results in sample order; lane m holds the m-th vertex
        //      accepted in this round ----------------------------------------------------------------
        if (warp == cw) {
            uint32_t newp = 0;
            double newc = 0.0;
            int nnew = 0, consumed = 0, jc = j;
            bool hs = have_sol, finished = false, cut = false;
            int vs = vsol;
            double cs = csol;
            long long fs = first_sol;
            // Lane k replays sample k.  What a sample has to be checked against -- the vertices accepted earlier in the same round --
            // is settled one earlier sample per step: at step kk sample kk is final (every sample before it has had its say),
            // so its point, verdict and cost are broadcast and the later lanes test themselves against it: same cell -> the
            // later sample is a duplicate; strictly nearer than its recorded nearest vertex -> the round ends before it; inside
            // its radius -> one more radius-set member, and a candidate parent if it is cheaper than what the sample has (those
            // few edges are walked one after the other, by the whole warp).  Candidates meet a sample in index order and replace
            // its parent only when strictly cheaper, which is the reference's choose-parent order (rrt.py:510-521).  The in-order
            // loop below (one sample at a time) remains for the rounds in which the tree may fill up, and under -DRRTK_SEQ_COMMIT.
            bool fast = false;
#ifndef RRTK_SEQ_COMMIT
            if (j + kact <= n) {
                const SampleRec r = s_rec[min(lane, K - 1)];
                const bool in = lane < kact;
                bool a = in && !(r.flags & 2) && (r.flags & 4);              // accepted unless the round interferes
                double bc = r.bc;
                int bv = r.bv;
                const int x = px(r.pnew), y = py(r.pnew);
                int extra = 0, stop = kact, nacc = 0;                        // samples [stop, kact) are left for the next round
                unsigned addm = __ballot_sync(RRTK_FULL, a);                 // who adds a vertex, as far as settled (bit kk is final at step kk)
                for (int kk = 0; kk < stop; ++kk) {
                    if (!((addm >> kk) & 1u)) continue;                      // sample kk adds no vertex
                    const uint32_t pk = __shfl_sync(RRTK_FULL, r.pnew, kk);
                    const uint32_t du = dist2(pk, x, y);
                    const bool later = in && lane > kk && lane < stop;
                    bool special = false;                                     // INFORMED: the vertex lies in the goal region
                    if (KIND == RRTK_INFORMED) special = __dsqrt_rn((double)dist2(pk, gx, gy)) < P.r_goal;     // rrt.py:744-745
                    // the common step: nobody later in the round is touched by this vertex (one ballot, nothing else to exchange)
                    if (!special && !__any_sync(RRTK_FULL, later && (du < r.bd || (a && (du == 0 || du < r2x))))) { ++nacc; continue; }
                    const double myc = (bv != 0x7fffffff) ? bc : r.c0;       // final for lane kk
                    const double ck = __shfl_sync(RRTK_FULL, myc, kk);
                    if (special) {
                        const bool changed = !hs || ck < cs;
                        if (!hs) fs = it0 + kk;
                        if (changed) { cs = ck; vs = j + nacc; }
                        hs = true;
                        if (changed) { stop = kk + 1; ++nacc; break; }         // later samples of the round used the old sampler state
                    }
                    const unsigned cutm = __ballot_sync(RRTK_FULL, later && du != 0 && du < r.bd);
                    if (cutm) stop = min(stop, __ffs(cutm) - 1);             // it would be their nearest vertex: redo from there
                    const bool still = later && lane < stop;
                    if (still && du == 0 && a) {                              // now in `sampled` (rrt.py:426/508/708)
                        a = false;
                    }
                    addm = __ballot_sync(RRTK_FULL, a);
                    const bool inr = KIND != RRTK_STANDARD && still && a && du < r2x;
                    if (__any_sync(RRTK_FULL, inr)) {
                        double cn = CUDART_INF;
                        if (inr) { ++extra; cn = reach_cost(ck, du); }
                        unsigned wm = __ballot_sync(RRTK_FULL, inr && cn < r.c0 && cn < bc);    // higher index: loses cost ties
                        while (wm) {
                            const int dst = __ffs(wm) - 1;
                            wm &= wm - 1;
                            const uint32_t pq = __shfl_sync(RRTK_FULL, r.pnew, dst);
                            const int h = WALK(px(pk), py(pk), px(pq), py(pq));
                            my_checks += 1; my_cells += cells_tested(h);
                            if (h < 0 && lane == dst) { bc = cn; bv = j + nacc; }
                        }
                    }
                    ++nacc;
                }
                const bool cons = lane < stop;
                const bool acc = a && cons;
                const unsigned accm = __ballot_sync(RRTK_FULL, acc);
                const int myj = j + __popc(accm & ((1u << lane) - 1u));      // the tree size when this sample is reached
                if (acc) {                                                    // rrt.py:524-529
                    const bool hasbv = bv != 0x7fffffff;
                    s_pts[tree_slot<T>(myj)] = r.pnew; cost[myj] = hasbv ? bc : r.c0; parent[myj] = hasbv ? bv : r.vnear;
                }
                if (KIND == RRTK_INFORMED && ellipse_mode) {
                    if (cons) ell_c[myj] = r.ell;                            // rrt.py:701
                    ell_iters += stop;
                }
                consumed = stop;
                jc = j + __popc(accm);
                nn_pairs += __reduce_add_sync(RRTK_FULL, cons ? myj : 0);
                ring_members += __reduce_add_sync(RRTK_FULL, acc ? r.ring + extra : 0);
                accepted += __popc(accm);
                fast = true;
            }
#endif
            for (int k = 0; k < kact && !fast; ++k) {
                const SampleRec r = s_rec[k];
                if (KIND != RRTK_INFORMED && jc == n) { finished = true; break; }
                const int x = px(r.pnew), y = py(r.pnew);
                bool reject = (r.flags & 2) || jc == n || !(r.flags & 4);
                double bc = r.bc;
                int bv = r.bv;
                // vertices accepted earlier in this round are not in the scan this sample was compared with
                const bool mine = lane < nnew;
                const uint32_t du = mine ? dist2(newp, x, y) : 0xffffffffu;
                if (__any_sync(RRTK_FULL, mine && du != 0 && du < r.bd)) { cut = true; break; }   // it would be the nearest vertex: redo
                if (__any_sync(RRTK_FULL, mine && du == 0)) reject = true;             // now in `sampled` (rrt.py:426/508/708)
                int ringm = r.ring;
                if (KIND != RRTK_STANDARD && !reject) {
                    const bool inr = mine && du < r2x;
                    const unsigned inm = __ballot_sync(RRTK_FULL, inr);
                    ringm += __popc(inm);
                    if (inm) {
                        double cn = CUDART_INF;
                        if (inr) cn = reach_cost(newc, du);
                        bool live = inr && cn < r.c0 && cn < bc;              // higher index: loses cost ties
                        for (;;) {                                            // cheapest first; equal cost -> lower lane
                            if (!__any_sync(RRTK_FULL, live)) break;
                            const uint32_t hi = live ? (uint32_t)__double2hiint(cn) : 0xffffffffu;
                            const uint32_t mhi = warp_min_u32(hi);
                            const uint32_t lo = (live && hi == mhi) ? (uint32_t)__double2loint(cn) : 0xffffffffu;
                            const uint32_t mlo = warp_min_u32(lo);
                            const int src = __ffs(__ballot_sync(RRTK_FULL, live && hi == mhi && lo == mlo)) - 1;
                            const uint32_t pp = __shfl_sync(RRTK_FULL, newp, src);
                            const int h = WALK(px(pp), py(pp), x, y);
                            my_checks += 1; my_cells += cells_tested(h);
                            if (h < 0) { bc = __hiloint2double((int)mhi, (int)mlo); bv = j + src; break; }
                            if (lane == src) live = false;
                        }
                    }
                }
                ++consumed;
                nn_pairs += jc;
                if (KIND == RRTK_INFORMED && ellipse_mode) {
                    if (lane == 0) ell_c[jc] = r.ell;                          // rrt.py:701
                    ++ell_iters;
                }
                if (reject) continue;
                ring_members += ringm;
                const int vbest = (bv != 0x7fffffff) ? bv : r.vnear;
                const double cbest = (bv != 0x7fffffff) ? bc : r.c0;
                if (lane == 0) { s_pts[tree_slot<T>(jc)] = r.pnew; cost[jc] = cbest; parent[jc] = vbest; }   // rrt.py:524-529
                if (lane == nnew) { newp = r.pnew; newc = cbest; }
                ++nnew;
                ++accepted;
                bool changed = false;
                if (KIND == RRTK_INFORMED) {
                    const uint32_t dg = dist2(r.pnew, gx, gy);
                    if (__dsqrt_rn((double)dg) < P.r_goal) {                   // rrt.py:744-745
                        changed = !hs || cbest < cs;
                        if (!hs) fs = it0 + k;
                        if (changed) { cs = cbest; vs = jc; }
                        hs = true;
                    }
                }
                ++jc;
                if (changed) break;                                            // later samples of the round used the old sampler state
            }
            if (it0 + consumed >= n) finished = true;
            // stage the next round's samples
            const int itn = it0 + consumed;
            __syncwarp();                                                      // lane 0's tree writes -> all lanes
            const int kwant_next = consumed < kact ? max(min(K, 1 + (jc >> 3)), max(1, kact >> 1)) : min(K, 2 * kact);
            const int kact_next = min(min(K, n - itn), kwant_next);          // the next round's kact (same formula as above)
            if (lane == 0) s_next = NW;
            if (KIND == RRTK_INFORMED && hs && balls != nullptr) {
                if (lane < K) {
                    short2 qn = make_short2(0, 0);
                    if (itn + lane < n) {
                        const double c = reach_cost(cs, dist2(s_pts[tree_slot<T>(vs)], gx, gy));   // rrt.py:698-699
                        int ex, ey;
                        ellipse_sample(P.W, P.H, dsc->rot, sx, sy, gx, gy, c, balls[itn + lane], ex, ey);
                        qn = make_short2((short)ex, (short)ey);
                        s_qc[lane] = c;
                    }
                    s_q[lane] = qn;
                    s_qk[lane] = scan_consts(qn, lane < kact_next);
                }
            } else {
                const int src = min(consumed + lane, 31);
                const int ax_ = __shfl_sync(RRTK_FULL, (int)ahead.x, src), ay_ = __shfl_sync(RRTK_FULL, (int)ahead.y, src);
                if (lane < K) {
                    const short2 qn = make_short2((short)ax_, (short)ay_);
                    s_q[lane] = qn;
                    s_qk[lane] = scan_consts(qn, lane < kact_next);
                }
            }
            if (lane == 0) {
                RoundSummary s;
                s.j = jc; s.consumed = consumed; s.flags = (hs ? 1 : 0) | (finished ? 2 : 0);
                s.vsol = vs; s.csol = cs; s.first_sol = fs;
                s.kwant = kwant_next; s.pad = 0;
                s_sum = s;
            }
            (void)cut;
        }
        __syncthreads();                                                   // ---- barrier: tree updated
        PHASE_T(t_3);
        PHASE_ADD(clk_scan, t_0, t_1); PHASE_ADD(clk_owner, t_1, t_2); PHASE_ADD(clk_commit, t_2, t_3); PHASE_ADD(clk_ownwork, t_1, t_1b);
#ifdef RRTK_PHASE_CLOCKS
        ++rounds;
#endif
        {
            const RoundSummary s = s_sum;
#ifndef RRTK_FIXED_COMMIT
            cw = (cw + 1 == NW) ? 0 : cw + 1;
#endif
            j = s.j;
            it0 += s.consumed;
            kwant = s.kwant;
            have_sol = s.flags & 1;
            vsol = s.vsol; csol = s.csol; first_sol = s.first_sol;
            if (s.flags & 2) break;
        }
    }

    // ---- goal connection: rrt.py:284-332, ascending (cost, index), filled vertices only ------
    if (tid == 0) { s_goalc = 0x7ff0000000000000ull; s_goalv = 0x7fffffff; }
    __syncthreads();
    for (int base = warp * 32; base < j; base += NW * 32) {
        const int v = base + lane;
        const bool valid = v < j;
        const uint32_t p = s_pts[tree_slot<T>(valid ? v : 0)];
        double cg = CUDART_INF;
        if (valid) cg = reach_cost(cost[v], dist2(p, gx, gy));
        unsigned m = __ballot_sync(RRTK_FULL, valid && cg < __longlong_as_double(*(volatile unsigned long long *)&s_goalc));
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const double cv = __shfl_sync(RRTK_FULL, cg, l);
            const uint32_t pp = __shfl_sync(RRTK_FULL, p, l);
            if (cv < __longlong_as_double(*(volatile unsigned long long *)&s_goalc)) {
                const int h = WALK(px(pp), py(pp), gx, gy);
                my_checks += 1; my_cells += cells_tested(h);
                if (h < 0 && lane == 0) atomicMin(&s_goalc, (unsigned long long)__double_as_longlong(cv));
            }
        }
    }
    __syncthreads();
    const unsigned long long cstar_bits = s_goalc;
    const bool reachable = cstar_bits != 0x7ff0000000000000ull;
    if (reachable) {   // lowest index among vertices with exactly the minimum cost and a free walk
        for (int base = warp * 32; base < j; base += NW * 32) {
            const int v = base + lane;
            const bool valid = v < j;
            const uint32_t p = s_pts[tree_slot<T>(valid ? v : 0)];
            double cg = CUDART_INF;
            if (valid) cg = reach_cost(cost[v], dist2(p, gx, gy));
            unsigned m = __ballot_sync(RRTK_FULL, valid && (unsigned long long)__double_as_longlong(cg) == cstar_bits);
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                const uint32_t pp = __shfl_sync(RRTK_FULL, p, l);
                const int h = WALK(px(pp), py(pp), gx, gy);
                my_checks += 1; my_cells += cells_tested(h);
                if (h < 0 && lane == 0) atomicMin(&s_goalv, base + l);
            }
        }
    }
    if (lane == 0) {
        atomicAdd(&s_checks, (unsigned long long)my_checks);
        atomicAdd(&s_cells, (unsigned long long)my_cells);
    }
    __syncthreads();

    // ---- outputs -------------------------------------------------------------------------------
    const int vparent = s_goalv;
    const bool found = reachable && vparent != 0x7fffffff;
    const int top = found ? j + 1 : j;     // rows holding real vertices
    short2 *opts = P.pts + (size_t)plan * (n + 1);
    for (int v = tid; v <= n; v += T) {
        short2 o = make_short2(-32768, -32768);
        if (v < j) {
            const uint32_t p = s_pts[tree_slot<T>(v)];
            o = make_short2((short)px(p), (short)py(p));
        } else if (v == j && found) {
            o = make_short2((short)gx, (short)gy);
        }
        opts[v] = o;
        if (v >= top) { cost[v] = CUDART_INF; parent[v] = -1; }
    }
    if (lane == 0) {      // every warp has committed some rounds: add the counters up
        atomicAdd(&s_cnt[0], (unsigned long long)ell_iters); atomicAdd(&s_cnt[1], (unsigned long long)nn_pairs);
        atomicAdd(&s_cnt[2], (unsigned long long)ring_members); atomicAdd(&s_cnt[3], (unsigned long long)accepted);
    }
    __syncthreads();
    ell_iters = (long long)s_cnt[0]; nn_pairs = (long long)s_cnt[1]; ring_members = (long long)s_cnt[2]; accepted = (long long)s_cnt[3];
    if (tid == 0) {
        if (found) { cost[j] = __longlong_as_double((long long)cstar_bits); parent[j] = vparent; }
        long long *st = P.stats + (size_t)plan * RRTK_STAT_COUNT;
        st[RRTK_STAT_J] = j;
        st[RRTK_STAT_VGOAL] = found ? j : 0;
        st[RRTK_STAT_FOUND] = found ? 1 : 0;
        st[RRTK_STAT_CHECKS] = (long long)s_checks;
        st[RRTK_STAT_CELLS] = (long long)s_cells;
        st[RRTK_STAT_FIRST_SOL_ITER] = first_sol;
        st[RRTK_STAT_ELL_ITERS] = ell_iters;
        st[RRTK_STAT_NN_PAIRS] = nn_pairs;
        st[RRTK_STAT_RING_MEMBERS] = ring_members;
        st[RRTK_STAT_ACCEPTED] = accepted;
        st[RRTK_STAT_RESERVED0] = 0;
        st[RRTK_STAT_RESERVED1] = 0;
#ifdef RRTK_PHASE_CLOCKS
        st[RRTK_STAT_RESERVED0] = clk_scan;
        st[RRTK_STAT_RESERVED1] = clk_owner;
        st[RRTK_STAT_ELL_ITERS] = clk_commit;
        st[RRTK_STAT_FIRST_SOL_ITER] = clk_ownwork;
        st[RRTK_STAT_RING_MEMBERS] = rounds;
#endif
    }
#undef WALK
}

}  // namespace rrtk
