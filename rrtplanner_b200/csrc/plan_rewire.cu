// K8: planners the reference advertises but does not contain -- RRT* whose rewire step fires (the reference's
// predicate rrt.py:532-536 never does) and the Dubins-vehicle RRT / RRT* (README.md:12,18-19).  Specification and
// bit-exact oracle: oracle/rewire_oracle.c (parity UNPINNED: there is no reference code for these; with the Euclidean
// model and rewire off this kernel reproduces the pinned reference trees, tests/test_gpu_rewire.py).
//
// One thread block per plan, one sample per round (a rewire changes costs the next sample's choose-parent reads, so
// the K-samples-per-round replay of plan_scan.cuh does not apply).  Per round:
//   A  scan      each warp owns a contiguous slice of the tree: nearest vertex (lowest index on ties), duplicate test,
//                membership of the rewire radius as one ballot word per 32 vertices
//   B  gate ||   the LAST warp measures and tests the gate edge nearest -> sample; meanwhile the other warps (named
//      lists     barrier 1 among themselves) build the ascending radius list, bound the new vertex's cost from below to
//                drop hopeless rewire candidates, and measure one edge per thread (Dubins: a lookup in the memo of the
//                primitive when the batch has one, else the shortest of six words)
//   C  rank      candidates (Euclidean prefilter and cost test of the specification) ranked by (cost, vertex)
//   D  choose    warps test the candidates' edges in rank order; the lowest free rank is the parent
//   E  insert    vertex j; rewire candidates flagged against the new vertex's cost
//   F  test      warps test the rewire edges sample -> member
//   G  apply     warp 0, ascending vertex order, re-testing against costs already lowered this round; the rewired
//                subtree's costs are recomputed breadth-first over child lists kept in shared memory
// The goal connection evaluates every vertex, prunes with a shared 64-bit minimum and breaks ties by index.
//
// Informed sampling (cfg.informed, the rule of rrt.py:690-701,744-745 on top of this loop): accepted vertices within r_goal
// of the goal join a list; while it is non-empty the (x, y) of a round is the ellipse point for c = cost of the list's
// cheapest vertex + its distance to the goal.  A rewire can lower that cost, so warp 0 re-reads the list at the end of every
// accepted round (one sample per round is exactly what this needs); rejected rounds change nothing and reuse c.
#include <math_constants.h>
#include <cstdio>

#include "dubins.cuh"
#include "plan_common.cuh"      // ellipse_sample

#ifndef RRTK_K8_BLOCK_THREADS
#define RRTK_K8_BLOCK_THREADS 768        // resident threads per SM the register allocation is bounded for
#endif

namespace rrtk {

// Dubins model on heading-layer grids (rrtk_plan2_batch_layers): a pose tests the layer grid of its own heading.  Internal: the
// public rrtk_model values are EUCLID and DUBINS.
constexpr int kModelDubinsLayers = 2;

enum { S2_J = 0, S2_VGOAL, S2_FOUND, S2_CHECKS, S2_ACCEPTED, S2_REWIRES, S2_PROPAGATED, S2_RING, S2_LEN_EVALS, S2_OVERFLOW, S2_ELL_ITERS, S2_FIRST_SOL };

struct Plan2Params {
    const uint32_t *bits;
    size_t words_per_grid;
    int W, H, TY;
    const rrtk_plan_desc *plans;
    int n;
    int star, rewire, NH;
    uint32_t r2_excl;
    double rho, ds;
    const short2 *samples;
    const uint8_t *heads;
    short2 *pts;
    uint8_t *head;
    double *cost;
    double *elen;
    int *parent;
    long long *stats;
    double *gcost;          // scratch: (n + 1) doubles per plan
    uint16_t *queue;        // scratch: (n + 1) vertex ids per plan
    uint16_t *sol;          // scratch: (n + 1) vertex ids per plan: the solution vertices of an informed plan, in the order they joined
    int informed;
    double r_goal;
    const double2 *balls;   // informed: n unit-disc draws per plan (NULL = probe: stop at the first solution vertex)
    double *ell_c;          // informed, optional: (n + 1) per plan, the budget the last ellipse sample drawn at that j used
    int ring_cap;
    // optional memo of the Dubins primitive (rrtk_dubins_table_build): shortest path for every displacement in
    // [-tR, tR]^2 and every heading pair, entry ((dx + tR) * (2 tR + 1) + dy + tR) * NH * NH + h0 * NH + h1
    const double *tlen;     // length
    const double *ttpq;     // (t, p, q)
    const uint8_t *tword;   // word
    int tR;
    int nlayers;            // kModelDubinsLayers: heading-layer grids per world, words_per_grid apart
};

__host__ __device__ __forceinline__ size_t dubins_table_entries(int R, int NH) { return (size_t)(2 * R + 1) * (2 * R + 1) * NH * NH; }
__device__ __forceinline__ size_t dubins_table_index(int dx, int dy, int h0, int h1, int R, int NH)
{
    return ((size_t)((dx + R) * (2 * R + 1) + dy + R) * NH + h0) * NH + h1;
}

constexpr uint16_t kNil = 0xffffu;

template <int MODEL>
struct Edge {
    // length of a -> b (Dubins: w.word and w.len are set; t, p, q only when the path was computed, see path())
    static __device__ __forceinline__ double length(const Plan2Params &P, const double2 *tab, uint32_t pa, int ha, uint32_t pb, int hb,
                                                    DubinsPath &w)
    {
        if (MODEL == RRTK_MODEL_EUCLID) {
            w.word = 0;
            return __dsqrt_rn((double)dist2(pa, px(pb), py(pb)));
        }
        const int dx = px(pb) - px(pa), dy = py(pb) - py(pa);
        if (P.tlen && abs(dx) <= P.tR && abs(dy) <= P.tR) {           // memoised: one L2-resident load instead of ~1.5 k FP64 operations
            const size_t i = dubins_table_index(dx, dy, ha, hb, P.tR, P.NH);
            w.word = (int)__ldg(P.tword + i);
            w.len = __ldg(P.tlen + i);
            w.t = w.p = w.q = CUDART_NAN;
            return w.len;
        }
        DubinsPath tmp;                           // only this copy has its address taken: w itself can stay in registers
        dubins_shortest(dx, dy, ha, hb, P.NH, P.rho, tab, tmp);
        w = tmp;
        return w.len;
    }
    // (t, p, q) of the word length() chose for the same pair (same bits either way: the table was filled by dubins_shortest)
    static __device__ __forceinline__ void path(const Plan2Params &P, const double2 *tab, uint32_t pa, int ha, uint32_t pb, int hb, int word,
                                                DubinsPath &w)
    {
        if (MODEL == RRTK_MODEL_EUCLID) { w.word = 0; return; }
        const int dx = px(pb) - px(pa), dy = py(pb) - py(pa);
        if (P.tlen && abs(dx) <= P.tR && abs(dy) <= P.tR) {
            const size_t i = dubins_table_index(dx, dy, ha, hb, P.tR, P.NH);
            w.word = word;
            w.len = __ldg(P.tlen + i);
            w.t = __ldg(P.ttpq + 3 * i); w.p = __ldg(P.ttpq + 3 * i + 1); w.q = __ldg(P.ttpq + 3 * i + 2);
            return;
        }
        DubinsPath tmp;
        dubins_rebuild(dx, dy, ha, hb, P.NH, P.rho, tab, word, tmp);
        w = tmp;
    }
    // warp-cooperative: is a -> b free (w = the path of path() for the same pair)
    static __device__ __forceinline__ bool is_free(const Plan2Params &P, const uint32_t *bits, uint32_t pa, int ha, uint32_t pb, int hb,
                                                   const DubinsPath &w, int lane)
    {
        if (MODEL == RRTK_MODEL_EUCLID)
            return warp_first_hit(GlobalGrid{bits}, P.TY, px(pa), py(pa), px(pb), py(pb), lane) < 0;
        if (MODEL == kModelDubinsLayers)
            return dubins_free_warp_layers(bits, P.words_per_grid, P.nlayers, P.W, P.H, P.TY, px(pa), py(pa), ha, px(pb), py(pb), hb, P.NH,
                                           P.rho, P.ds, w, lane);
        return dubins_free_warp(bits, P.W, P.H, P.TY, px(pa), py(pa), ha, px(pb), py(pb), P.NH, P.rho, P.ds, w, lane);
    }
};

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(RRTK_FULL, v, o);
        v = other < v ? other : v;
    }
    return v;
}

// INF: the informed sampling rule, compiled in only where it is asked for (the plain planners keep their registers)
template <int MODEL, int T, bool INF>
__global__ void __launch_bounds__(T, RRTK_K8_BLOCK_THREADS / T) plan_rewire_kernel(Plan2Params P)
{
    constexpr int NW = T / 32;
    constexpr bool DUB = MODEL != RRTK_MODEL_EUCLID;
    constexpr int KS = 1024 / T;                 // radius-set slots per thread (the list holds at most 1024)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = P.n, cap = P.ring_cap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int plan = blockIdx.x;

    // ---- shared-memory carve-up -------------------------------------------------------------------
    unsigned char *sp = smem_raw;
    double *valL1 = reinterpret_cast<double *>(sp); sp += sizeof(double) * cap;      // length member -> sample, per radius-set slot
    double *valL2 = reinterpret_cast<double *>(sp); sp += sizeof(double) * cap;      // length sample -> member
    double2 *tab = reinterpret_cast<double2 *>(sp); sp += sizeof(double2) * 256;     // (sin, cos) per heading
    uint32_t *spts = reinterpret_cast<uint32_t *>(sp); sp += sizeof(uint32_t) * (size_t)((n + 2) & ~1);
    uint32_t *mask = reinterpret_cast<uint32_t *>(sp); sp += sizeof(uint32_t) * (size_t)(((n + 1 + 31) / 32 + 1) & ~1);
    uint16_t *first = reinterpret_cast<uint16_t *>(sp); sp += sizeof(uint16_t) * (size_t)((n + 4) & ~3);
    uint16_t *next = reinterpret_cast<uint16_t *>(sp); sp += sizeof(uint16_t) * (size_t)((n + 4) & ~3);
    uint16_t *ring = reinterpret_cast<uint16_t *>(sp); sp += sizeof(uint16_t) * (size_t)cap;
    uint8_t *flag = reinterpret_cast<uint8_t *>(sp); sp += (size_t)cap;
    uint8_t *word1 = reinterpret_cast<uint8_t *>(sp); sp += (size_t)cap;             // Dubins word of the two edges per slot
    uint8_t *word2 = reinterpret_cast<uint8_t *>(sp); sp += (size_t)cap;
    uint16_t *tasks2 = reinterpret_cast<uint16_t *>(sp); sp += sizeof(uint16_t) * (size_t)cap;    // slots whose edge sample -> member is wanted
    uint8_t *shead = reinterpret_cast<uint8_t *>(sp);

    __shared__ unsigned long long s_wmin[NW];
    __shared__ int s_wcnt[NW];
    __shared__ int s_wdup[NW];
    __shared__ unsigned long long s_wlb[NW];
    __shared__ int s_ntask2;
    __shared__ unsigned long long s_best;       // goal connection: bit pattern of the cheapest free cost
    __shared__ int s_bestslot;
    __shared__ int s_bestrank, s_ncand;         // choose-parent: lowest free rank, number of ranked candidates
    __shared__ int s_accept, s_tail;
    __shared__ double s_c0, s_l0;
    __shared__ long long s_stat[10];
    __shared__ int s_nsol, s_first;             // informed: solution vertices so far, iteration that accepted the first one
    __shared__ double s_cb;                     // informed: budget c of the ellipse the next sample is drawn from (s_nsol > 0)

    const rrtk_plan_desc pd = P.plans[plan];
    const uint32_t *bits = P.bits + (size_t)pd.world * (MODEL == kModelDubinsLayers ? P.nlayers : 1) * P.words_per_grid;
    const short2 *samples = P.samples + (size_t)plan * n;
    const uint8_t *heads = P.heads ? P.heads + (size_t)plan * n : nullptr;
    short2 *o_pts = P.pts + (size_t)plan * (n + 1);
    uint8_t *o_head = P.head + (size_t)plan * (n + 1);
    double *cost = P.cost + (size_t)plan * (n + 1);
    double *elen = P.elen + (size_t)plan * (n + 1);
    int *parent = P.parent + (size_t)plan * (n + 1);
    double *gcost = P.gcost + (size_t)plan * (n + 1);
    uint16_t *queue = P.queue + (size_t)plan * (n + 1);
    uint16_t *sol = P.sol + (size_t)plan * (n + 1);
    const double2 *balls = (INF && P.balls) ? P.balls + (size_t)plan * n : nullptr;
    double *ell_c = (INF && P.ell_c) ? P.ell_c + (size_t)plan * (n + 1) : nullptr;
    const double rot[4] = {INF ? pd.rot[0] : 0.0, INF ? pd.rot[1] : 0.0, INF ? pd.rot[2] : 0.0, INF ? pd.rot[3] : 0.0};

    // ---- initialise ---------------------------------------------------------------------------------
    for (int v = tid; v <= n; v += T) {
        spts[v] = RRTK_FAR_VERTEX; shead[v] = 255; first[v] = kNil; next[v] = kNil;
        o_pts[v] = make_short2(-32768, -32768); o_head[v] = 255;
        cost[v] = CUDART_INF; elen[v] = CUDART_INF; parent[v] = -1;
        if (INF && ell_c) ell_c[v] = CUDART_NAN;
    }
    if (DUB) {
        const double dth = DM_TWO_PI / (double)P.NH;
        for (int h = tid; h < P.NH; h += T) {
            double s, c;
            dm_sincos((double)h * dth, s, c);
            tab[h] = make_double2(s, c);
        }
    }
    if (tid < 10) s_stat[tid] = 0;
    if (tid == 0) { s_nsol = 0; s_first = -1; s_cb = 0.0; }
    __syncthreads();
    const int start_h = DUB ? pd.reserved[0] : 0;
    const int goal_h = DUB ? pd.reserved[1] : 0;
    if (tid == 0) {
        spts[0] = pack_xy(pd.start_x, pd.start_y); shead[0] = (uint8_t)start_h;
        o_pts[0] = make_short2((short)pd.start_x, (short)pd.start_y); o_head[0] = (uint8_t)start_h;
        cost[0] = 0.0; elen[0] = 0.0;
    }
    __syncthreads();

    int j = 1;
    long long my_checks = 0, my_lens = 0;      // per-thread counters, reduced at the end
    long long ell_iters = 0;                   // informed: rounds whose sample came from the ellipse (the same in every thread)
    // -DRRTK_K8_CLOCKS (experiment builds): cycles thread 0 spends up to the barrier that ends each phase, printed for plan 0
#ifdef RRTK_K8_CLOCKS
    long long clk_acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, clk_last = clock64(), clk_rounds = 0;
    long long clk_sub[4] = {0, 0, 0, 0}, clk_t0 = 0;
#define K8_SUB0() do { if (tid == 0) clk_t0 = clock64(); } while (0)
#define K8_SUB(i) do { if (tid == 0) { const long long now_ = clock64(); clk_sub[i] += now_ - clk_t0; clk_t0 = now_; } } while (0)
#define K8_CLK(i) do { if (tid == 0) { const long long now_ = clock64(); clk_acc[i] += now_ - clk_last; clk_last = now_; } } while (0)
#else
#define K8_CLK(i) do { } while (0)
#define K8_SUB0() do { } while (0)
#define K8_SUB(i) do { } while (0)
#endif
    const bool both = P.rewire != 0;           // edge lengths in both directions per member
    // Dubins: a length costs ~1.5 k instructions, so phase B2 first drops the members no new vertex could improve;
    // Euclid: a length is one square root, so all of them are simply measured
    const bool prune = both && DUB;

    for (int it = 0; it < n; ++it) {
        const short2 sm = samples[it];
        int qx = sm.x, qy = sm.y;
        if (INF && s_nsol > 0) {                 // uniform: the list and the budget only change before a round's last barrier
            if (!balls) break;                    // probe run
            const double c = s_cb;
            ellipse_sample(P.W, P.H, rot, pd.start_x, pd.start_y, pd.goal_x, pd.goal_y, c, balls[it], qx, qy);   // rrt.py:699-700
            if (tid == 0 && ell_c) ell_c[j] = c;                                                                     // rrt.py:701
            ++ell_iters;
        }
        const int qh = (DUB && heads) ? heads[it] : 0;
        const uint32_t pnew = pack_xy(qx, qy);

        // ---- A: scan ---------------------------------------------------------------------------------
        const int chunk = (((j + NW - 1) / NW) + 31) & ~31;
        const int v0 = warp * chunk, v1 = min(j, v0 + chunk);
        {
            uint32_t bd = 0xffffffffu;
            int bv = 0, cnt = 0;
            bool dup = false;
            for (int base = v0; base < v1; base += 32) {
                const int v = base + lane;
                const bool in = v < v1;
                const uint32_t d2 = in ? dist2(spts[v], qx, qy) : 0xffffffffu;
                if (d2 < bd) { bd = d2; bv = v; }
                dup |= in && d2 == 0u && v >= 1;
                const unsigned m = __ballot_sync(RRTK_FULL, in && d2 < P.r2_excl);
                if (lane == 0) mask[base >> 5] = m;
                cnt += __popc(m);
            }
            const unsigned long long key = warp_min_u64(((unsigned long long)bd << 32) | (unsigned)bv);
            const bool anydup = __any_sync(RRTK_FULL, dup);
            if (lane == 0) { s_wmin[warp] = key; s_wcnt[warp] = cnt; s_wdup[warp] = anydup; }
        }
        __syncthreads();
        K8_CLK(0);

        // ---- B: the last warp tests the gate edge nearest -> sample (a path lookup, then up to ~90 sampled cells: the longest
        //         single job of a round) while the other warps build the radius list and measure its edges; the workers
        //         synchronise among themselves on named barrier 1, everybody meets again at the block barrier below ------
        unsigned long long nk = s_wmin[0];
        int m_total = 0, my_off = 0, dup_any = 0, last_off = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            nk = s_wmin[w] < nk ? s_wmin[w] : nk;
            if (w < warp) my_off += s_wcnt[w];
            if (w < NW - 1) last_off += s_wcnt[w];
            m_total += s_wcnt[w];
            dup_any |= s_wdup[w];
        }
        const int vnear = (int)(nk & 0xffffffffu);
        const bool overflow = P.star && m_total > cap;
        const int m = (P.star && !overflow) ? m_total : 0;
        if (warp == NW - 1) {
            // ---- gate warp ---------------------------------------------------------------------------------------
            const uint32_t pn = spts[vnear];
            const int hn = shead[vnear];
            DubinsPath w0;
            const double l0 = Edge<MODEL>::length(P, tab, pn, hn, pnew, qh, w0);
            if (DUB && w0.t != w0.t)      // memoised length: fetch the path's (t, p, q)
                Edge<MODEL>::path(P, tab, pn, hn, pnew, qh, w0.word, w0);
            w0.len = l0;
            const bool ok = Edge<MODEL>::is_free(P, bits, pn, hn, pnew, qh, w0, lane);
            if (lane == 0) {
                ++my_checks; ++my_lens;
                s_accept = ok && !dup_any && j != n && !overflow;
                if (overflow) s_stat[S2_OVERFLOW] = 1;
                s_c0 = __dadd_rn(cost[vnear], l0); s_l0 = l0;
                s_bestrank = 0x7fffffff; s_ncand = 0;
            }
        } else {
            // ---- worker warps: B1 ascending radius list; lower bound on the new vertex's cost ---------------------
            constexpr int TW = T - 32;                            // worker threads
            if (m) {
                // own slice of the tree, and warp 0 also takes the gate warp's slice
                for (int part = 0; part < (warp == 0 ? 2 : 1); ++part) {
                    const int c0v = part ? (NW - 1) * chunk : v0, c1v = part ? min(j, c0v + chunk) : v1;
                    int off = part ? last_off : my_off;
                    for (int base = c0v; base < c1v; base += 32) {
                        const unsigned mk = mask[base >> 5];
                        if ((mk >> lane) & 1u) ring[off + __popc(mk & ((1u << lane) - 1u))] = (uint16_t)(base + lane);
                        off += __popc(mk);
                    }
                }
            }
            if (tid == 0) s_ntask2 = 0;
            asm volatile("bar.sync 1, %0;" ::"r"(TW) : "memory");
            // ---- B2: which members need the edge sample -> member: only those a vertex of cost >= lb could improve ---
            if (prune && m) {
                // lower bound on the new vertex's cost, min over the members of cost + straight-line distance, taken over the
                // dense list (in the sparse ballot loop above it ran with one or two active lanes per step)
                unsigned long long lbk = 0xffffffffffffffffull;
                for (int base = warp * 32; base < m; base += TW) {
                    const int i = base + lane;
                    if (i < m) {
                        const int vn = ring[i];
                        const double c = __dadd_rn(cost[vn], __dsqrt_rn((double)dist2(spts[vn], qx, qy)));
                        const unsigned long long k = (unsigned long long)__double_as_longlong(c);
                        lbk = k < lbk ? k : lbk;
                    }
                }
                lbk = warp_min_u64(lbk);
                if (lane == 0) s_wlb[warp] = lbk;
                asm volatile("bar.sync 1, %0;" ::"r"(TW) : "memory");
                lbk = (unsigned long long)__double_as_longlong(__dadd_rn(cost[vnear], __dsqrt_rn((double)(uint32_t)(nk >> 32))));
#pragma unroll
                for (int w = 0; w < NW - 1; ++w) lbk = s_wlb[w] < lbk ? s_wlb[w] : lbk;
                // every edge is at least as long as the straight line up to rounding (and the 1e-9 snap of mod2pi): 1e-6 cells of slack
                const double lb = __dsub_rn(__longlong_as_double((long long)lbk), 1e-6);
                for (int base = warp * 32; base < m; base += TW) {
                    const int i = base + lane;
                    bool want = false;
                    if (i < m) {
                        const int vn = ring[i];
                        want = __dadd_rn(lb, __dsqrt_rn((double)dist2(spts[vn], qx, qy))) < cost[vn];
                        word2[i] = 0xfe;                              // "not measured": phase E must never need it
                    }
                    const unsigned bal = __ballot_sync(RRTK_FULL, want);
                    int at = 0;
                    if (lane == 0 && bal) at = atomicAdd(&s_ntask2, __popc(bal));
                    at = __shfl_sync(RRTK_FULL, at, 0);
                    if (want) tasks2[at + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)i;
                }
                asm volatile("bar.sync 1, %0;" ::"r"(TW) : "memory");
            }
            // ---- B3: edge lengths, one task per worker thread: member -> sample for every member, sample -> member
            //          where B2 asked for it (Euclid: everywhere) ------------------------------------------------------
            const int ntask = m + (prune ? (m ? s_ntask2 : 0) : (both ? m : 0));
            for (int tsk = tid; tsk < ntask; tsk += TW) {
                const bool back = tsk >= m;                          // sample -> member
                const int slot = back ? (prune ? (int)tasks2[tsk - m] : tsk - m) : tsk;
                const int vn = ring[slot];
                const uint32_t pv = spts[vn];
                const int hv = shead[vn];
                DubinsPath w;
                const double l = Edge<MODEL>::length(P, tab, back ? pnew : pv, back ? qh : hv, back ? pv : pnew, back ? hv : qh, w);
                ++my_lens;
                if (back) { valL2[slot] = l; word2[slot] = (uint8_t)w.word; }
                else { valL1[slot] = l; word1[slot] = (uint8_t)w.word; }
            }
        }
        __syncthreads();
        K8_CLK(3);
        if (!s_accept) continue;                 // uniform: every thread reads the same shared flag
        const double c0 = s_c0;

        // ---- C: parent candidates (prefilter and cost test of the specification); a candidate's slot of valL1 now holds
        //         its cost through that edge, the edge length stays in a register of the thread that owns the slot --------
        double myL[KS];
#pragma unroll
        for (int k = 0; k < KS; ++k) {
            const int i = tid + k * T;
            myL[k] = 0.0;
            if (i < m) {
                const int vn = ring[i];
                uint8_t f = 0;
                if (vn != vnear) {
                    const double cv = cost[vn];
                    const double D = __dsqrt_rn((double)dist2(spts[vn], qx, qy));
                    const double L = valL1[i];
                    const double cn = __dadd_rn(cv, L);
                    if (__dadd_rn(cv, D) < c0 && cn < c0) { f = 1; myL[k] = L; valL1[i] = cn; }
                }
                flag[i] = f;
            }
        }
        __syncthreads();
        K8_CLK(4);
        // ---- C2: rank the candidates by (cost, vertex) -- the order the specification breaks ties in -- so that the edge
        //          tests below run cheapest first and the first free one in that order is the parent ----------------------
        for (int i = tid; i < m; i += T) {
            if (!flag[i]) continue;
            const double cn = valL1[i];
            int rank = 0;
            for (int t = 0; t < m; ++t) {
                if (!flag[t]) continue;
                const double ct = valL1[t];
                rank += (ct < cn || (ct == cn && t < i)) ? 1 : 0;
            }
            tasks2[rank] = (uint16_t)i;              // tasks2 is free again: rank -> slot
            atomicAdd(&s_ncand, 1);
        }
        __syncthreads();
        K8_CLK(5);

        // ---- D: choose the parent: warps test the candidates' edges in rank order, the lowest free rank wins -----------
        for (int r = warp; r < s_ncand; r += NW) {
            if (r > s_bestrank) break;                // a cheaper free edge is known
            const int i = tasks2[r];
            const int vn = ring[i];
            const uint32_t pv = spts[vn];
            DubinsPath w;
            w.word = 0;
            Edge<MODEL>::path(P, tab, pv, shead[vn], pnew, qh, word1[i], w);
            const bool ok = Edge<MODEL>::is_free(P, bits, pv, shead[vn], pnew, qh, w, lane);
            if (lane == 0) {
                ++my_checks;
                if (ok) atomicMin(&s_bestrank, r);
            }
        }
        __syncthreads();
        K8_CLK(6);
        // ---- E: insert vertex j, rewire candidates ---------------------------------------------------------
        int vbest = vnear, wslot = -1;
        double cbest = c0;
        if (s_bestrank != 0x7fffffff) { wslot = tasks2[s_bestrank]; vbest = ring[wslot]; cbest = valL1[wslot]; }
        if (wslot >= 0 && tid == (wslot % T)) {       // the owner of the winning slot still holds the edge length
            double lb = 0.0;
#pragma unroll
            for (int k = 0; k < KS; ++k) lb = (wslot / T == k) ? myL[k] : lb;
            elen[j] = lb;
        }
        if (tid == 0) {
            spts[j] = pnew; shead[j] = (uint8_t)qh;
            o_pts[j] = make_short2((short)qx, (short)qy); o_head[j] = (uint8_t)qh;
            cost[j] = cbest; parent[j] = vbest;
            if (wslot < 0) elen[j] = s_l0;
            next[j] = first[vbest]; first[vbest] = (uint16_t)j;
            s_stat[S2_ACCEPTED] += 1; s_stat[S2_RING] += m;
            if (INF && __dsqrt_rn((double)dist2(pnew, pd.goal_x, pd.goal_y)) < P.r_goal) {      // rrt.py:744-745
                if (s_nsol == 0) s_first = it;
                sol[s_nsol] = (uint16_t)j;
                s_nsol = s_nsol + 1;
            }
        }
        if (both) {
            for (int i = tid; i < m; i += T) {
                const int vn = ring[i];
                uint8_t f = 0;
                if (vn != vbest) {
                    const double cv = cost[vn];
                    const double D = __dsqrt_rn((double)dist2(spts[vn], qx, qy));
                    if (__dadd_rn(cbest, D) < cv) {
                        if (prune && word2[i] == 0xfe) s_stat[S2_OVERFLOW] = 2;   // the lower bound of B2 was not one: report, never hide
                        else if (__dadd_rn(cbest, valL2[i]) < cv) f = 1;
                    }
                }
                flag[i] = f;
            }
            __syncthreads();
        K8_CLK(7);
            // ---- F: test the rewire edges sample -> member -------------------------------------------------
            for (int i = warp; i < m; i += NW) {
                if (!flag[i]) continue;
                const int vn = ring[i];
                const uint32_t pv = spts[vn];
                DubinsPath w;
                w.word = 0;
                Edge<MODEL>::path(P, tab, pnew, qh, pv, shead[vn], word2[i], w);
                const bool ok = Edge<MODEL>::is_free(P, bits, pnew, qh, pv, shead[vn], w, lane);
                __syncwarp();                        // every lane has read flag[i] before lane 0 rewrites it
                if (lane == 0) { ++my_checks; flag[i] = ok ? 2 : 0; }
            }
            __syncthreads();
        K8_CLK(8);
            // ---- G: apply in ascending vertex order ----------------------------------------------------------
            if (warp == 0) {
                for (int base = 0; base < m; base += 32) {
                    const int i = base + lane;
                    unsigned todo = __ballot_sync(RRTK_FULL, i < m && flag[i] == 2);
                    while (todo) {
                        const int b = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const int slot = base + b;
                        const int vn = ring[slot];
                        const double lr = valL2[slot];
                        const double cm = __dadd_rn(cbest, lr);
                        const double cv = cost[vn];              // may have been lowered by an earlier rewire of this round
                        const double D = __dsqrt_rn((double)dist2(spts[vn], qx, qy));
                        if (!(__dadd_rn(cbest, D) < cv && cm < cv)) continue;       // warp-uniform
                        if (lane == 0) {
                            const int op = parent[vn];
                            if (first[op] == vn) first[op] = next[vn];
                            else { int c = first[op]; while (next[c] != vn) c = next[c]; next[c] = next[vn]; }
                            next[vn] = first[j]; first[j] = (uint16_t)vn;
                            parent[vn] = j; elen[vn] = lr; cost[vn] = cm;
                            queue[0] = (uint16_t)vn;
                            s_tail = 1;
                            s_stat[S2_REWIRES] += 1;
                        }
                        __syncwarp();
                        int qhd = 0, qtl = 1;
                        while (qhd < qtl) {                       // breadth-first: a level's costs are final before its children read them
                            const int take = min(32, qtl - qhd);
                            if (lane < take) {
                                const int u = queue[qhd + lane];
                                const double cu = cost[u];
                                for (int c = first[u]; c != kNil; c = next[c]) {
                                    cost[c] = __dadd_rn(cu, elen[c]);
                                    queue[atomicAdd(&s_tail, 1)] = (uint16_t)c;
                                }
                            }
                            qhd += take;
                            __syncwarp();
                            qtl = s_tail;
                            __syncwarp();
                        }
                        if (lane == 0) s_stat[S2_PROPAGATED] += qtl - 1;
                        __syncwarp();
                    }
                }
            }
        }
        if (INF && warp == 0) {
            // least_cost over the solution vertices (rrt.py:627-633: first minimum in list order) with the costs as they stand after
            // this round's rewires, + that vertex's distance to the goal (rrt.py:697-698): the budget of the next ellipse
            __syncwarp();
            const int ns = s_nsol;
            if (ns > 0) {
                double bc = CUDART_INF;
                int bk = 0x7fffffff;
                for (int k = lane; k < ns; k += 32) {
                    const double c = cost[sol[k]];
                    if (c < bc) { bc = c; bk = k; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double oc = __shfl_xor_sync(RRTK_FULL, bc, o);
                    const int ok = __shfl_xor_sync(RRTK_FULL, bk, o);
                    if (oc < bc || (oc == bc && ok < bk)) { bc = oc; bk = ok; }
                }
                if (lane == 0) s_cb = __dadd_rn(bc, __dsqrt_rn((double)dist2(spts[sol[bk]], pd.goal_x, pd.goal_y)));
            }
        }
        ++j;
        __syncthreads();
        K8_CLK(9);
    }

#ifdef RRTK_K8_CLOCKS
    if (tid == 0 && plan == 0)
        printf("K8 clocks plan0 j=%d: A %lld B1 %lld B2 %lld B3 %lld C %lld D %lld Dres %lld E %lld F %lld G %lld\n", j, clk_acc[0], clk_acc[1],
               clk_acc[2], clk_acc[3], clk_acc[4], clk_acc[5], clk_acc[6], clk_acc[7], clk_acc[8], clk_acc[9]);
    if (tid == 0 && plan == 0) printf("K8 B3 split: tasks %lld path %lld gate-test %lld\n", clk_sub[0], clk_sub[1], clk_sub[2]);
#endif
    // ---- goal connection (rrt.py:284-332 with this model's edges) ----------------------------------------
    const uint32_t pgoal = pack_xy(pd.goal_x, pd.goal_y);
    if (tid == 0) { s_best = 0xffffffffffffffffull; s_bestslot = 0x7fffffff; }
    for (int v = tid; v < j; v += T) {
        DubinsPath w;
        const double lg = Edge<MODEL>::length(P, tab, spts[v], shead[v], pgoal, goal_h, w);
        ++my_lens;
        gcost[v] = __dadd_rn(cost[v], lg);
        first[v] = (uint16_t)(w.word & 0xff);          // the child lists are no longer needed: keep the word per vertex here
    }
    __syncthreads();
    // every vertex whose cost is not already beaten is tested; the shared minimum only prunes
    for (int v = warp; v < j; v += NW) {
        const double cg = gcost[v];
        if ((unsigned long long)__double_as_longlong(cg) > s_best) continue;        // a cheaper free edge is known
        DubinsPath w;
        w.word = 0;
        Edge<MODEL>::path(P, tab, spts[v], shead[v], pgoal, goal_h, (int)(int8_t)first[v], w);
        const bool ok = Edge<MODEL>::is_free(P, bits, spts[v], shead[v], pgoal, goal_h, w, lane);
        if (lane == 0) {
            ++my_checks;
            if (ok) atomicMin(&s_best, (unsigned long long)__double_as_longlong(cg));
            queue[v] = ok ? 1 : 0;
        }
    }
    __syncthreads();
    const unsigned long long gbest = s_best;
    if (gbest != 0xffffffffffffffffull) {
        for (int v = tid; v < j; v += T) {
            const unsigned long long b = (unsigned long long)__double_as_longlong(gcost[v]);
            // a vertex with cost == gbest was never pruned (pruning needs cost > best >= gbest), so queue[v] is its verdict
            if (b == gbest && queue[v] == 1) atomicMin(&s_bestslot, v);
        }
    }
    __syncthreads();
    // reduce the per-thread counters
    for (int o = 16; o > 0; o >>= 1) {
        my_checks += __shfl_xor_sync(RRTK_FULL, my_checks, o);
        my_lens += __shfl_xor_sync(RRTK_FULL, my_lens, o);
    }
    if (lane == 0) {
        atomicAdd(reinterpret_cast<unsigned long long *>(&s_stat[S2_CHECKS]), (unsigned long long)my_checks);
        atomicAdd(reinterpret_cast<unsigned long long *>(&s_stat[S2_LEN_EVALS]), (unsigned long long)my_lens);
    }
    __syncthreads();
    if (tid == 0) {
        int vgoal = 0, found = 0;
        if (gbest != 0xffffffffffffffffull) {
            const int v = s_bestslot;
            DubinsPath w;
            const double lg = Edge<MODEL>::length(P, tab, spts[v], shead[v], pgoal, goal_h, w);
            vgoal = j; found = 1;
            o_pts[j] = make_short2((short)pd.goal_x, (short)pd.goal_y); o_head[j] = (uint8_t)goal_h;
            cost[j] = gcost[v]; elen[j] = lg; parent[j] = v;
        }
        long long *st = P.stats + (size_t)plan * RRTK_STAT_COUNT;
        for (int k = 0; k < RRTK_STAT_COUNT; ++k) st[k] = k < 10 ? s_stat[k] : 0;
        st[S2_J] = j; st[S2_VGOAL] = vgoal; st[S2_FOUND] = found;
        st[S2_ELL_ITERS] = ell_iters; st[S2_FIRST_SOL] = s_first;
    }
}

// ---- launch -----------------------------------------------------------------------------------------------
static size_t plan2_smem(int n, int cap)
{
    size_t b = 0;
    b += sizeof(double) * 2 * (size_t)cap;
    b += sizeof(double2) * 256;
    b += sizeof(uint32_t) * (size_t)((n + 2) & ~1);
    b += sizeof(uint32_t) * (size_t)(((n + 1 + 31) / 32 + 1) & ~1);
    b += sizeof(uint16_t) * 2 * (size_t)((n + 4) & ~3);
    b += sizeof(uint16_t) * (size_t)cap;
    b += (size_t)cap * 5;
    b += (size_t)(n + 1);
    return (b + 15) & ~(size_t)15;
}

static int plan2_ring_cap(int n)
{
    int cap = (n + 1 + 31) & ~31;
    return cap < 1024 ? cap : 1024;
}

size_t plan2_scratch_bytes(int nplans, int n)
{
    return (size_t)nplans * (n + 1) * (sizeof(double) + 2 * sizeof(uint16_t)) + 16;
}

template <int MODEL, int T, bool INF>
static int plan2_launch_ti(const Plan2Params &P, int nplans, size_t smem, cudaStream_t st)
{
    RRTK_CUDA(cudaFuncSetAttribute(plan_rewire_kernel<MODEL, T, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    plan_rewire_kernel<MODEL, T, INF><<<nplans, T, smem, st>>>(P);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

template <int MODEL, int T>
static int plan2_launch_t(const Plan2Params &P, int nplans, size_t smem, cudaStream_t st)
{
    return P.informed ? plan2_launch_ti<MODEL, T, true>(P, nplans, smem, st) : plan2_launch_ti<MODEL, T, false>(P, nplans, smem, st);
}

int plan2_footprint(int n, int threads, int optin, int sm_smem, int *smem_bytes, int *blocks_per_sm)
{
    const size_t smem = plan2_smem(n, plan2_ring_cap(n));
    if (smem + 1024 > (size_t)optin) return RRTK_ERR_CAPACITY;
    const int T = threads > 0 ? threads : 256;
    int b = (int)((size_t)sm_smem / (smem + 1024 + 512));
    if (b > 2048 / T) b = 2048 / T;
    if (smem_bytes) *smem_bytes = (int)smem;
    if (blocks_per_sm) *blocks_per_sm = b < 1 ? 1 : b;
    return RRTK_OK;
}

// nlayers > 0: DUBINS on nlayers heading-layer grids per world (rrtk_plan2_batch_layers); 0: one grid per world
int plan2_launch(const rrtk_plan2_cfg &cfg, const uint32_t *d_bits, int W, int H, int nlayers, const rrtk_plan_desc *d_plans, int nplans,
                 int n, const int16_t *d_samples, const uint8_t *d_heads, int16_t *d_pts, uint8_t *d_head, double *d_cost, double *d_elen,
                 int32_t *d_parent, int64_t *d_stats, void *d_scratch, int threads, int optin, cudaStream_t st)
{
    Plan2Params P;
    P.bits = d_bits;
    P.words_per_grid = grid_words(W, H);
    P.W = W; P.H = H; P.TY = tiles_y(H);
    P.plans = d_plans;
    P.n = n;
    P.star = cfg.star != 0; P.rewire = cfg.star != 0 && cfg.rewire != 0; P.NH = cfg.nheadings;
    const double lim = ceil(cfg.r_rewire * cfg.r_rewire);
    P.r2_excl = !P.star ? 0u : (lim >= 1073741824.0 ? 1073741824u : (lim <= 0.0 ? 0u : (uint32_t)lim));
    P.rho = cfg.rho; P.ds = cfg.ds;
    P.samples = reinterpret_cast<const short2 *>(d_samples);
    P.heads = d_heads;
    P.pts = reinterpret_cast<short2 *>(d_pts);
    P.head = d_head;
    P.cost = d_cost; P.elen = d_elen; P.parent = d_parent;
    P.stats = reinterpret_cast<long long *>(d_stats);
    uintptr_t s = (reinterpret_cast<uintptr_t>(d_scratch) + 15) & ~(uintptr_t)15;
    P.gcost = reinterpret_cast<double *>(s);
    P.queue = reinterpret_cast<uint16_t *>(P.gcost + (size_t)nplans * (n + 1));
    P.sol = P.queue + (size_t)nplans * (n + 1);
    P.informed = cfg.informed != 0;
    P.r_goal = cfg.r_goal;
    P.balls = reinterpret_cast<const double2 *>(cfg.balls);
    P.ell_c = cfg.ell_c;
    P.tlen = nullptr; P.ttpq = nullptr; P.tword = nullptr; P.tR = 0;
    if (cfg.model == RRTK_MODEL_DUBINS && cfg.dubins_table && cfg.table_radius > 0) {
        const size_t N = dubins_table_entries(cfg.table_radius, cfg.nheadings);
        P.tlen = reinterpret_cast<const double *>(cfg.dubins_table);
        P.ttpq = P.tlen + N;
        P.tword = reinterpret_cast<const uint8_t *>(P.ttpq + 3 * N);
        P.tR = cfg.table_radius;
    }
    P.nlayers = nlayers;
    P.ring_cap = plan2_ring_cap(n);
    const size_t smem = plan2_smem(n, P.ring_cap);
    if (smem + 1024 > (size_t)optin) {
        set_error("plan with n=%d needs %zu bytes of shared memory (limit %d)", n, smem, optin);
        return RRTK_ERR_CAPACITY;
    }
    const int T = threads > 0 ? threads : 256;
    if (T != 128 && T != 256) {
        set_error("rrtk_plan2_batch: threads must be 0, 128 or 256");
        return RRTK_ERR_INVALID;
    }
    if (nlayers > 0)
        return T == 128 ? plan2_launch_t<kModelDubinsLayers, 128>(P, nplans, smem, st) : plan2_launch_t<kModelDubinsLayers, 256>(P, nplans, smem, st);
    if (cfg.model == RRTK_MODEL_EUCLID)
        return T == 128 ? plan2_launch_t<RRTK_MODEL_EUCLID, 128>(P, nplans, smem, st) : plan2_launch_t<RRTK_MODEL_EUCLID, 256>(P, nplans, smem, st);
    return T == 128 ? plan2_launch_t<RRTK_MODEL_DUBINS, 128>(P, nplans, smem, st) : plan2_launch_t<RRTK_MODEL_DUBINS, 256>(P, nplans, smem, st);
}

// ---- Dubins primitive, batched (README.md:12 "Dubins Primitive Module") --------------------------------------
__global__ void dubins_paths_kernel(const int *q, long long nq, int NH, double rho, int *word, double *tpq, double *len)
{
    __shared__ double2 tab[256];
    const double dth = DM_TWO_PI / (double)NH;
    for (int h = threadIdx.x; h < NH; h += blockDim.x) {
        double s, c;
        dm_sincos((double)h * dth, s, c);
        tab[h] = make_double2(s, c);
    }
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const int *e = q + 6 * i;
    DubinsPath w;
    dubins_shortest(e[3] - e[0], e[4] - e[1], e[2], e[5], NH, rho, tab, w);
    if (word) word[i] = w.word;
    if (tpq) { tpq[3 * i] = w.t; tpq[3 * i + 1] = w.p; tpq[3 * i + 2] = w.q; }
    if (len) len[i] = w.len;
}

// one warp per query: sampled collision test, and optionally the sampled poses (cap per query).  LAYERS: each world has nlayers
// heading-layer grids (rrtk_dubins_collision_layers).
template <bool LAYERS>
__global__ void dubins_walk_kernel(const uint32_t *bits, size_t words_per_grid, int W, int H, int nlayers, const int *q, const int *world,
                                   long long nq, int NH, double rho, double ds, uint8_t *free_out, int cap, double *xyth, int *count)
{
    __shared__ double2 tab[256];
    const double dth = DM_TWO_PI / (double)NH;
    for (int h = threadIdx.x; h < NH; h += blockDim.x) {
        double s, c;
        dm_sincos((double)h * dth, s, c);
        tab[h] = make_double2(s, c);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= nq) return;
    const int *e = q + 6 * i;
    DubinsPath w;
    dubins_shortest(e[3] - e[0], e[4] - e[1], e[2], e[5], NH, rho, tab, w);
    if (free_out) {
        const uint32_t *g = bits + (size_t)(world ? world[i] : 0) * (LAYERS ? nlayers : 1) * words_per_grid;
        const bool ok = LAYERS ? dubins_free_warp_layers(g, words_per_grid, nlayers, W, H, tiles_y(H), e[0], e[1], e[2], e[3], e[4], e[5], NH,
                                                         rho, ds, w, lane)
                               : dubins_free_warp(g, W, H, tiles_y(H), e[0], e[1], e[2], e[3], e[4], NH, rho, ds, w, lane);
        if (lane == 0) free_out[i] = ok ? 1 : 0;
    }
    if (xyth) {
        const DubinsTrack tr = dubins_track(e[0], e[1], e[2], NH, rho, w);
        const long long ns = (long long)floor(w.len / ds);
        double *o = xyth + (size_t)i * cap * 3;
        for (long long k = lane; k <= ns && k < cap; k += 32) {
            const Pose a = dubins_point(tr, (double)k * ds);
            o[3 * k] = a.x; o[3 * k + 1] = a.y; o[3 * k + 2] = a.th;
        }
        if (lane == 0) count[i] = (int)(ns + 1);
    }
}

// memo of the primitive: one thread per (displacement, heading pair)
__global__ void dubins_table_kernel(int R, int NH, double rho, double *tlen, double *ttpq, uint8_t *tword)
{
    __shared__ double2 tab[256];
    const double dth = DM_TWO_PI / (double)NH;
    for (int h = threadIdx.x; h < NH; h += blockDim.x) {
        double s, c;
        dm_sincos((double)h * dth, s, c);
        tab[h] = make_double2(s, c);
    }
    __syncthreads();
    const size_t N = dubins_table_entries(R, NH);
    const int side = 2 * R + 1;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (size_t)gridDim.x * blockDim.x) {
        const int h1 = (int)(i % NH), h0 = (int)((i / NH) % NH);
        const size_t cell = i / ((size_t)NH * NH);
        const int dy = (int)(cell % side) - R, dx = (int)(cell / side) - R;
        DubinsPath w;
        dubins_shortest(dx, dy, h0, h1, NH, rho, tab, w);
        tlen[i] = w.len; tword[i] = (uint8_t)w.word;
        ttpq[3 * i] = w.t; ttpq[3 * i + 1] = w.p; ttpq[3 * i + 2] = w.q;
    }
}

size_t dubins_table_bytes(int R, int NH) { return dubins_table_entries(R, NH) * (4 * sizeof(double) + 1) + 16; }

int dubins_table_launch(int R, int NH, double rho, void *d_table, int sm_count, cudaStream_t st)
{
    const size_t N = dubins_table_entries(R, NH);
    double *tlen = reinterpret_cast<double *>(d_table);
    double *ttpq = tlen + N;
    uint8_t *tword = reinterpret_cast<uint8_t *>(ttpq + 3 * N);
    size_t blocks = (N + 127) / 128;
    const size_t cap = (size_t)(sm_count > 0 ? sm_count : 148) * 64;
    dubins_table_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 128, 0, st>>>(R, NH, rho, tlen, ttpq, tword);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

int dubins_paths_launch(const int32_t *d_q, int64_t nq, int NH, double rho, int32_t *d_word, double *d_tpq, double *d_len, cudaStream_t st)
{
    dubins_paths_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, st>>>(d_q, nq, NH, rho, d_word, d_tpq, d_len);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

// nlayers > 0: the worlds of d_bits are heading-layer grids, nlayers per world (rrtk_dubins_collision_layers)
int dubins_walk_launch(const uint32_t *d_bits, int W, int H, int nlayers, const int32_t *d_q, const int32_t *d_world, int64_t nq, int NH,
                       double rho, double ds, uint8_t *d_free, int cap, double *d_xyth, int32_t *d_count, cudaStream_t st)
{
    const unsigned blocks = (unsigned)((nq + 3) / 4);
    if (nlayers > 0)
        dubins_walk_kernel<true><<<blocks, 128, 0, st>>>(d_bits, grid_words(W, H), W, H, nlayers, d_q, d_world, nq, NH, rho, ds, d_free, cap,
                                                         d_xyth, d_count);
    else
        dubins_walk_kernel<false><<<blocks, 128, 0, st>>>(d_bits, grid_words(W, H), W, H, 0, d_q, d_world, nq, NH, rho, ds, d_free, cap,
                                                          d_xyth, d_count);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

}  // namespace rrtk
