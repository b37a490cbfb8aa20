// Sample streams: RRT.sample_all_free (rrt.py:231-240) with the reference's random generator.
//
// The reference draws free[rand_gen.choice(nfree)] with rand_gen = np.random.default_rng(seed)
// (rrt.py:85), i.e. numpy's PCG64 (128-bit LCG, XSL-RR 64-bit output, stepped before output)
// feeding Lemire's bounded 32-bit rejection method from buffered 32-bit halves (low half first).
// numpy is not part of /root/reference; the algorithm is restated from numpy's published source
// (numpy/random/src/pcg64/pcg64.h, numpy/random/src/distributions/distributions.c, numpy 1.21 ..
// 2.3 identical here) and pinned by tests against default_rng(seed).integers(0, nfree, n) and
// against tests/golden/sampler_seed12345.npz (drawn by the reference's own sampler).
//
// rank -> cell: free = argwhere(og == 0) (rrt.py:64) lists free cells row-major, so rank k lies in
// the row x with rowcum[x] <= k < rowcum[x+1] and is the (k - rowcum[x])-th clear bit of that row.
#include "common.cuh"

namespace rrtk {

struct Pcg64 {
    unsigned long long hi, lo, inc_hi, inc_lo;
    bool has32;
    uint32_t buf32;

    __device__ __forceinline__ void step()
    {
        // state = state * 0x2360ED051FC65DA44385DF649FCCF645 + inc  (mod 2^128)
        const unsigned long long mh = 0x2360ED051FC65DA4ull, ml = 0x4385DF649FCCF645ull;
        const unsigned long long l = lo * ml;
        const unsigned long long h = __umul64hi(lo, ml) + hi * ml + lo * mh;
        const unsigned long long nl = l + inc_lo;
        hi = h + inc_hi + (nl < l ? 1ull : 0ull);
        lo = nl;
    }
    __device__ __forceinline__ unsigned long long next64()
    {
        step();
        const unsigned long long x = hi ^ lo;
        const unsigned r = (unsigned)(hi >> 58);
        return (x >> r) | (x << ((64 - r) & 63));
    }
    __device__ __forceinline__ uint32_t next32()
    {
        if (has32) { has32 = false; return buf32; }
        const unsigned long long v = next64();
        has32 = true;
        buf32 = (uint32_t)(v >> 32);
        return (uint32_t)v;
    }
    // Generator.integers(0, bound) for 0 < bound <= 2^32 - 1  (Lemire, 32-bit)
    __device__ __forceinline__ uint32_t bounded(uint32_t bound)
    {
        const uint32_t rng = bound - 1;
        if (rng == 0) return 0;
        unsigned long long m = (unsigned long long)next32() * bound;
        uint32_t left = (uint32_t)m;
        if (left < bound) {
            const uint32_t thr = (0xffffffffu - rng) % bound;
            while (left < thr) {
                m = (unsigned long long)next32() * bound;
                left = (uint32_t)m;
            }
        }
        return (uint32_t)(m >> 32);
    }
    // Generator.integers(0, bound) for any bound >= 1 (a weighted stream's total): 32-bit Lemire below 2^32, the raw
    // buffered 32-bit half at exactly 2^32, 64-bit Lemire on next64 above (which leaves the buffered half alone)
    __device__ __forceinline__ unsigned long long bounded(unsigned long long bound)
    {
        if (bound < 0x100000000ull) return bounded((uint32_t)bound);
        if (bound == 0x100000000ull) return next32();
        unsigned long long v = next64();
        unsigned long long left = v * bound;
        if (left < bound) {
            const unsigned long long thr = (0ull - bound) % bound;
            while (left < thr) {
                v = next64();
                left = v * bound;
            }
        }
        return __umul64hi(v, bound);
    }
};

// rowcum may live in shared memory (the parallel kernel stages it) or in global memory
__device__ __forceinline__ short2 rank_to_cell(const uint32_t *__restrict__ g, const int *rowcum, int W, int TY, int k)
{
    int lo = 0, hi = W;                    // largest x with rowcum[x] <= k
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (rowcum[mid] <= k) lo = mid; else hi = mid;
    }
    int rem = k - rowcum[lo];
    int y = 0;
    const uint32_t *row = g + word_index(lo, 0, TY);        // word of tile (lo >> 5, ty) is row[ty << 5]
    for (int t0 = 0; t0 < TY; t0 += 4) {                    // four independent loads in flight per step
        uint32_t fr[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) fr[u] = (t0 + u < TY) ? ~__ldg(row + ((t0 + u) << 5)) : 0u;
        bool done = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = __popc(fr[u]);
            if (!done && rem < c) { y = ((t0 + u) << 5) + __fns(fr[u], 0, rem + 1); done = true; }
            if (!done) rem -= c;
        }
        if (done) break;
    }
    return make_short2((short)lo, (short)y);
}

// ---- the generator in parallel ----------------------------------------------------------------------------------
// PCG64 is a 128-bit LCG, so the state k steps ahead is state * A^k + inc * (A^k - 1) / (A - 1), computable in
// O(log k) (O'Neill's pcg_advance_lcg_128, restated): every thread jumps to its own slice of the raw 64-bit output
// sequence.  Lemire's rejection loop then simply drops the raw 32-bit values whose low product half falls below the
// threshold, i.e. the bounded draws are a stream COMPACTION of the raw values -- one block scan.
struct U128 { unsigned long long hi, lo; };
__device__ __forceinline__ U128 mul128(U128 a, U128 b)
{
    U128 r;
    r.lo = a.lo * b.lo;
    r.hi = __umul64hi(a.lo, b.lo) + a.hi * b.lo + a.lo * b.hi;
    return r;
}
__device__ __forceinline__ U128 add128(U128 a, U128 b)
{
    U128 r;
    r.lo = a.lo + b.lo;
    r.hi = a.hi + b.hi + (r.lo < a.lo ? 1ull : 0ull);
    return r;
}
// delta steps of the LCG as one affine map: state -> state * mult + plus
struct PcgAffine { U128 mult, plus; };
__device__ __forceinline__ PcgAffine pcg_affine(unsigned long long inc_hi, unsigned long long inc_lo, unsigned long long delta)
{
    U128 cur_mult = {0x2360ED051FC65DA4ull, 0x4385DF649FCCF645ull}, cur_plus = {inc_hi, inc_lo};
    U128 acc_mult = {0ull, 1ull}, acc_plus = {0ull, 0ull};
    while (delta) {
        if (delta & 1ull) {
            acc_mult = mul128(acc_mult, cur_mult);
            acc_plus = add128(mul128(acc_plus, cur_mult), cur_plus);
        }
        cur_plus = mul128(add128(cur_mult, U128{0ull, 1ull}), cur_plus);
        cur_mult = mul128(cur_mult, cur_mult);
        delta >>= 1;
    }
    return PcgAffine{acc_mult, acc_plus};
}
__device__ __forceinline__ void pcg_apply(Pcg64 &g, const PcgAffine &a)
{
    const U128 st = add128(mul128(a.mult, U128{g.hi, g.lo}), a.plus);
    g.hi = st.hi; g.lo = st.lo;
}
__device__ __forceinline__ void pcg_jump(Pcg64 &g, unsigned long long delta) { pcg_apply(g, pcg_affine(g.inc_hi, g.inc_lo, delta)); }

#ifndef RRTK_SAMPLE_THREADS
#define RRTK_SAMPLE_THREADS 256
#endif
constexpr int kSampleThreads = RRTK_SAMPLE_THREADS;
constexpr int kRawSlack = 62;          // raw 32-bit values generated beyond n; more rejections than that -> sequential path

// 32-bit words of the raw window of the parallel sampler: n + kRawSlack raw 32-bit values for 32-bit ranks; for 64-bit ranks
// also n + kRawSlack / 2 raw next64 outputs (64-bit Lemire), i.e. 2 n + kRawSlack words.  Plus 4 words of slack.
__host__ __device__ __forceinline__ int raw_window_words(int n, int rank_words) { return n * rank_words + kRawSlack + 4; }   // n <= 65534

// ---- the select step: where a bounded draw lands ------------------------------------------------------------------
// A sampler draws n ranks from integers(0, bound) and maps each rank to a cell.  The generator, the rejection compaction
// and the sequential fallback below are shared; the select policy supplies the bound of a world, what the parallel kernel
// stages in shared memory for it, and the rank -> cell map.
//   bound_t / rank_t   integer types of the bound and of a rank
//   stage_words(W)     32-bit words of shared memory the parallel kernel stages per plan
//   bound(world, W)    the plan's bound (a bound <= 1 draws 0 without touching the generator, as numpy does)
//   stage(world, W, s, tid)          fill the staged words (block-wide; read after the kernel's barriers)
//   unstaged(world, W)               the same words in global memory, for the sequential kernel (which stages nothing)
//   cell(world, W, H, s, k)          rank k -> cell; s = the staged words or their global copy

// Uniform: free[integers(0, nfree)], rank = index into the row-major list of free cells (rowcum + bit grid).
struct UniformSelect {
    using bound_t = uint32_t;
    using rank_t = uint32_t;
    const uint32_t *bits;
    const int *rowcum;
    static size_t stage_words(int W) { return (size_t)W + 1; }
    __device__ __forceinline__ uint32_t bound(int world, int W) const { return (uint32_t)__ldg(rowcum + (size_t)world * (W + 1) + W); }
    __device__ __forceinline__ void stage(int world, int W, uint32_t *s, int tid) const
    {
        const int *rc = rowcum + (size_t)world * (W + 1);
        for (int x = tid; x <= W; x += kSampleThreads) s[x] = (uint32_t)__ldg(rc + x);
    }
    __device__ __forceinline__ const uint32_t *unstaged(int world, int W) const
    {
        return reinterpret_cast<const uint32_t *>(rowcum + (size_t)world * (W + 1));
    }
    __device__ __forceinline__ short2 cell(int world, int W, int H, const uint32_t *s, uint32_t k) const
    {
        return rank_to_cell(bits + (size_t)world * grid_words(W, H), reinterpret_cast<const int *>(s), W, tiles_y(H), (int)k);
    }
};

// Weighted: the effective weight of a cell is its uint8 weight where the grid is free, else 0; rank k of integers(0, T),
// T = the world's total, lands on the cell whose exclusive prefix of effective weights (row-major) is <= k < prefix + weight
// (np.searchsorted(cumsum, k, side="right")).  The index (rrtk_weight_index) holds, after the nworlds totals, per world
// the W + 1 int64 prefixes of the row totals and per row the uint32 prefix at each 32-cell chunk (one bit-grid word).
struct WeightIndex {
    long long *tot;                    // nworlds totals T
    long long *rows;                   // world w: rows + w * (W + 1), rows[x] = weight of rows < x
    uint32_t *chunks;                  // world w, row x: chunks + (w * W + x) * TY, entry t = weight of cells y < 32 t of the row
    __host__ __device__ WeightIndex(void *base, int nworlds, int W, int H)
    {
        tot = reinterpret_cast<long long *>(base);
        rows = tot + nworlds;
        chunks = reinterpret_cast<uint32_t *>(rows + (size_t)nworlds * (W + 1));
        (void)H;
    }
    static size_t bytes(int nworlds, int W, int H)
    {
        return 8 * ((size_t)nworlds + (size_t)nworlds * (W + 1)) + 4 * (size_t)nworlds * W * tiles_y(H);
    }
};

struct WeightedSelect {
    using bound_t = unsigned long long;
    using rank_t = unsigned long long;
    const uint32_t *bits;
    const uint8_t *weights;
    const long long *tot, *rows;
    const uint32_t *chunks;
    static size_t stage_words(int) { return 0; }
    __device__ __forceinline__ unsigned long long bound(int world, int) const { return (unsigned long long)__ldg(tot + world); }
    __device__ __forceinline__ void stage(int, int, uint32_t *, int) const {}
    __device__ __forceinline__ const uint32_t *unstaged(int, int) const { return nullptr; }
    __device__ __forceinline__ short2 cell(int world, int W, int H, const uint32_t *, unsigned long long k) const
    {
        const int TY = tiles_y(H);
        const long long *rp = rows + (size_t)world * (W + 1);
        int lo = 0, hi = W;                                   // largest x with rp[x] <= k (rp[W] = T > k)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((unsigned long long)__ldg(rp + mid) <= k) lo = mid; else hi = mid;
        }
        uint32_t rem = (uint32_t)(k - (unsigned long long)__ldg(rp + lo));
        const uint32_t *cp = chunks + ((size_t)world * W + lo) * TY;
        int a = 0, b = TY;                                    // largest chunk t with cp[t] <= rem
        while (b - a > 1) {
            const int mid = (a + b) >> 1;
            if (__ldg(cp + mid) <= rem) a = mid; else b = mid;
        }
        rem -= __ldg(cp + a);
        const uint32_t occ = __ldg(bits + (size_t)world * grid_words(W, H) + word_index(lo, a << 5, TY));
        const uint8_t *wr = weights + ((size_t)world * W + lo) * H;
        int y = a << 5;
        const int last = min(H, y + 32) - 1;
        for (; y < last; ++y) {                               // at most 32 masked bytes; the last one takes what is left
            const uint32_t e = ((occ >> (y & 31)) & 1u) ? 0u : (uint32_t)__ldg(wr + y);
            if (rem < e) break;
            rem -= e;
        }
        return make_short2((short)lo, (short)y);
    }
};

// Lemire's 32-bit threshold (2^32 - bound) mod bound; for bound = 2^32 it is 0 and the rank is the raw value itself
__device__ __forceinline__ uint32_t lemire32_threshold(uint32_t bound) { return (0xffffffffu - (bound - 1u)) % bound; }
__device__ __forceinline__ uint32_t lemire32_threshold(unsigned long long bound) { return (uint32_t)((0x100000000ull - bound) % bound); }
__device__ __forceinline__ bool needs_next64(uint32_t) { return false; }
__device__ __forceinline__ bool needs_next64(unsigned long long bound) { return bound > 0x100000000ull; }

// 64-bit outputs k0 .. k1-1 of the generator, each thread its own slice [tid * per, ...) reached by jump-ahead
template <class Store>
__device__ __forceinline__ void raw_slices(const Pcg64 &g0, int n64, int tid, Store store)
{
    const int per = (n64 + kSampleThreads - 1) / kSampleThreads;      // outputs per thread
    Pcg64 g = g0;
    const int k0 = tid * per;
    if (k0 < n64) {
        pcg_jump(g, (unsigned long long)k0);
        const int k1 = min(n64, k0 + per);
        for (int k = k0; k < k1; ++k) store(k, g.next64());
    }
}

// Lemire's rejection loop as a block compaction of the raw values s_raw[0 .. total): thread t owns raw indices
// [t * span, (t + 1) * span); accept(raw, rank) says whether a raw value is kept and gives its rank.  Writes the first n ranks
// and returns (block-uniformly) the raw values they used up, or -1 when the window held fewer than n accepted values.
template <class Raw, class Rank, class Accept>
__device__ __forceinline__ int compact_ranks(const Raw *s_raw, int total, int n, Rank *s_rank, Accept accept, int *s_warp, int *s_consumed,
                                             int tid)
{
    const int lane = tid & 31, warp = tid >> 5;
    const int span = (total + kSampleThreads - 1) / kSampleThreads;
    const int r0 = tid * span, r1 = min(total, r0 + span);
    Rank rank;
    int acc = 0;
    for (int r = r0; r < r1; ++r) acc += accept(s_raw[r], rank) ? 1 : 0;
    int incl = acc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(RRTK_FULL, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    if (tid == 0) *s_consumed = -1;
    __syncthreads();
    int before = incl - acc;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    for (int r = r0; r < r1; ++r) {
        if (accept(s_raw[r], rank)) {
            if (before < n) s_rank[before] = rank;
            if (before == n - 1) *s_consumed = r + 1;
            ++before;
        }
    }
    __syncthreads();
    return *s_consumed;
}

__device__ __forceinline__ void store_state(unsigned long long *state_out, int plan, const Pcg64 &g)
{
    state_out[4 * plan] = g.hi; state_out[4 * plan + 1] = g.lo; state_out[4 * plan + 2] = g.inc_hi; state_out[4 * plan + 3] = g.inc_lo;
}

// one block per plan: the generator's raw outputs in parallel slices, Lemire's rejection as a compaction, then
// ranks -> cells in parallel.  The sequential generator remains as the fallback for a stream with more than kRawSlack
// rejections (probability ~ (n * bound / 2^32)^62 / 62!).  state_out / carry (optional) receive the generator after the
// n draws; state_out may alias state.
template <class Sel>
__global__ void __launch_bounds__(kSampleThreads)
sample_stream_kernel(Sel sel, int W, int H, const rrtk_plan_desc *__restrict__ plans, const unsigned long long *__restrict__ state, int n,
                     short2 *__restrict__ samples, unsigned long long *__restrict__ state_out, uint32_t *__restrict__ carry)
{
    using Bound = typename Sel::bound_t;
    using Rank = typename Sel::rank_t;
    extern __shared__ uint32_t s_mem[];
    constexpr int kRankWords = (int)(sizeof(Rank) / 4);
    Rank *s_rank = reinterpret_cast<Rank *>(s_mem);                     // n bounded draws
    uint32_t *s_raw = s_mem + kRankWords * n;                           // raw values in the order numpy hands them out
    uint32_t *s_stage = s_mem + kRankWords * n + raw_window_words(n, kRankWords);   // what the select step stages for this plan's world
    __shared__ int s_warp[kSampleThreads / 32];
    __shared__ int s_consumed;                   // raw values used up by the n draws (-1: not enough generated)
    const int plan = blockIdx.x, tid = threadIdx.x;
    const int world = plans[plan].world;
    const Bound bound = sel.bound(world, W);
    sel.stage(world, W, s_stage, tid);           // visible after the barriers below
    Pcg64 g0;
    g0.hi = state[4 * plan]; g0.lo = state[4 * plan + 1];
    g0.inc_hi = state[4 * plan + 2]; g0.inc_lo = state[4 * plan + 3];
    g0.has32 = false; g0.buf32 = 0;
    if (carry) { g0.has32 = carry[2 * plan] != 0; g0.buf32 = carry[2 * plan + 1]; }   // numpy's has_uint32 / uinteger
    const int off = g0.has32 ? 1 : 0;
    if (bound <= 1u) {                           // numpy returns the single value without touching the generator
        for (int i = tid; i < n; i += kSampleThreads) s_rank[i] = 0;
        if (tid == 0 && state_out) store_state(state_out, plan, g0);
        __syncthreads();
    } else if (needs_next64(bound)) {            // 64-bit Lemire: one raw next64 per candidate, the buffered half untouched
        unsigned long long *s_raw64 = reinterpret_cast<unsigned long long *>(s_raw);
        const int nraw = n + kRawSlack / 2;
        raw_slices(g0, nraw, tid, [&](int k, unsigned long long v) { s_raw64[k] = v; });
        __syncthreads();
        const unsigned long long thr = (0ull - (unsigned long long)bound) % (unsigned long long)bound;
        const int consumed = compact_ranks(s_raw64, nraw, n, s_rank, [&](unsigned long long v, Rank &rank) {
            rank = (Rank)__umul64hi(v, (unsigned long long)bound);
            return v * (unsigned long long)bound >= thr;
        }, s_warp, &s_consumed, tid);
        if (consumed < 0) {
            if (tid == 0) {
                Pcg64 g = g0;
                for (int i = 0; i < n; ++i) s_rank[i] = (Rank)g.bounded(bound);
                if (state_out) store_state(state_out, plan, g);
            }
        } else if (tid == 0 && state_out) {
            Pcg64 g = g0;
            pcg_jump(g, (unsigned long long)consumed);
            store_state(state_out, plan, g);
        }
        __syncthreads();
    } else {
        const int nraw = n + kRawSlack;                                   // raw values wanted: indices 0 .. nraw-1
        const int n64 = (nraw - off + 1) >> 1;                            // 64-bit outputs that cover them
        raw_slices(g0, n64, tid, [&](int k, unsigned long long v) {
            s_raw[off + 2 * k] = (uint32_t)v;
            s_raw[off + 2 * k + 1] = (uint32_t)(v >> 32);
        });
        if (tid == 0 && off) s_raw[0] = g0.buf32;
        __syncthreads();
        const uint32_t thr = lemire32_threshold(bound);
        const int consumed = compact_ranks(s_raw, off + 2 * n64, n, s_rank, [&](uint32_t v, Rank &rank) {
            const unsigned long long m = (unsigned long long)v * bound;
            rank = (Rank)(m >> 32);
            return (uint32_t)m >= thr;
        }, s_warp, &s_consumed, tid);
        if (consumed < 0) {                      // not enough accepted values in the window: the plain sequential generator
            if (tid == 0) {
                Pcg64 g = g0;
                for (int i = 0; i < n; ++i) s_rank[i] = g.bounded(bound);
                if (state_out) store_state(state_out, plan, g);
                if (carry) { carry[2 * plan] = g.has32 ? 1u : 0u; carry[2 * plan + 1] = g.buf32; }
            }
        } else if (tid == 0 && (state_out || carry)) {
            // the generator as the next plan() of the same planner object finds it (rrt.py:85: one rand_gen per object)
            const int used = consumed - off;                              // raw values taken from fresh 64-bit outputs
            const int out64 = (used + 1) >> 1;
            Pcg64 g = g0;
            pcg_jump(g, (unsigned long long)out64);
            if (state_out) store_state(state_out, plan, g);
            if (carry) {
                const bool half = used > 0 ? (used & 1) != 0 : g0.has32 && consumed == 0;
                carry[2 * plan] = half ? 1u : 0u;
                carry[2 * plan + 1] = half ? s_raw[consumed] : (used > 0 ? s_raw[consumed - 1] : g0.buf32);
            }
        }
        __syncthreads();
    }
    short2 *out = samples + (size_t)plan * n;
    for (int i = tid; i < n; i += kSampleThreads) out[i] = sel.cell(world, W, H, s_stage, s_rank[i]);
}

// n too large for the raw window in shared memory: thread 0 runs the generator sequentially
template <class Sel>
__global__ void sample_stream_seq_kernel(Sel sel, int W, int H, const rrtk_plan_desc *__restrict__ plans,
                                         const unsigned long long *__restrict__ state, int n, short2 *__restrict__ samples,
                                         unsigned long long *__restrict__ state_out, uint32_t *__restrict__ carry)
{
    using Rank = typename Sel::rank_t;
    extern __shared__ uint32_t s_mem[];
    Rank *s_rank = reinterpret_cast<Rank *>(s_mem);
    const int plan = blockIdx.x;
    const int world = plans[plan].world;
    const typename Sel::bound_t bound = sel.bound(world, W);
    if (threadIdx.x == 0) {
        Pcg64 g;
        g.hi = state[4 * plan]; g.lo = state[4 * plan + 1];
        g.inc_hi = state[4 * plan + 2]; g.inc_lo = state[4 * plan + 3];
        g.has32 = false; g.buf32 = 0;
        if (carry) { g.has32 = carry[2 * plan] != 0; g.buf32 = carry[2 * plan + 1]; }
        for (int i = 0; i < n; ++i) s_rank[i] = bound ? g.bounded(bound) : 0;
        if (state_out) store_state(state_out, plan, g);
        if (carry) { carry[2 * plan] = g.has32 ? 1u : 0u; carry[2 * plan + 1] = g.buf32; }
    }
    __syncthreads();
    short2 *out = samples + (size_t)plan * n;
    const uint32_t *rows = sel.unstaged(world, W);
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = sel.cell(world, W, H, rows, s_rank[i]);
}

template <class Sel>
static int sample_launch(const Sel &sel, int W, int H, const rrtk_plan_desc *d_plans, int nplans, const uint64_t *d_state, int n,
                         int16_t *d_samples, int optin, cudaStream_t st, uint64_t *d_state_out, uint32_t *d_carry)
{
    if (nplans == 0 || n == 0) return RRTK_OK;
    const size_t rank_words = sizeof(typename Sel::rank_t) / 4;
    const size_t smem = (n * rank_words + (size_t)raw_window_words(n, (int)rank_words) + Sel::stage_words(W)) * 4;   // draws + raw values + staged words
    const size_t smem_seq = (size_t)n * rank_words * 4;
    const unsigned long long *st64 = reinterpret_cast<const unsigned long long *>(d_state);
    unsigned long long *out64 = reinterpret_cast<unsigned long long *>(d_state_out);
    short2 *out = reinterpret_cast<short2 *>(d_samples);
    if (smem <= (size_t)optin) {
        RRTK_CUDA(cudaFuncSetAttribute(sample_stream_kernel<Sel>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        sample_stream_kernel<Sel><<<nplans, kSampleThreads, smem, st>>>(sel, W, H, d_plans, st64, n, out, out64, d_carry);
    } else if (smem_seq <= (size_t)optin) {
        RRTK_CUDA(cudaFuncSetAttribute(sample_stream_seq_kernel<Sel>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_seq));
        sample_stream_seq_kernel<Sel><<<nplans, 128, smem_seq, st>>>(sel, W, H, d_plans, st64, n, out, out64, d_carry);
    } else {
        set_error("sample stream of n=%d does not fit shared memory", n);
        return RRTK_ERR_CAPACITY;
    }
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

int sample_streams_launch(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H, const rrtk_plan_desc *d_plans,
                          int nplans, const uint64_t *d_state, int n, int16_t *d_samples, int optin, cudaStream_t st,
                          uint64_t *d_state_out, uint32_t *d_carry)
{
    return sample_launch(UniformSelect{d_bits, d_rowcum}, W, H, d_plans, nplans, d_state, n, d_samples, optin, st, d_state_out, d_carry);
}

// ---- weighted sampling: the index and the stream ------------------------------------------------------------------
size_t weight_index_bytes(int nworlds, int W, int H) { return WeightIndex::bytes(nworlds, W, H); }

// one warp per (world, row): lane t sums the effective weights of chunk t (+32, ...) -- the grid word is the mask -- then a
// warp scan writes the chunk prefixes and the row total (into rows[x + 1], made a prefix by weight_rows_kernel)
constexpr int kIndexWarps = 8;
__global__ void __launch_bounds__(kIndexWarps * 32)
weight_chunks_kernel(const uint32_t *__restrict__ bits, const uint8_t *__restrict__ weights, int nworlds, int W, int H, bool words4,
                     WeightIndex ix)
{
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * kIndexWarps + (threadIdx.x >> 5);
    if (r >= (long long)nworlds * W) return;
    const int world = (int)(r / W), x = (int)(r % W);
    const int TY = tiles_y(H);
    const uint32_t *g = bits + (size_t)world * grid_words(W, H);
    const uint8_t *wr = weights + (size_t)r * H;
    uint32_t *cp = ix.chunks + (size_t)r * TY;
    uint32_t carry = 0;
    for (int t0 = 0; t0 < TY; t0 += 32) {
        const int t = t0 + lane;
        uint32_t sum = 0;
        if (t < TY) {
            const uint32_t occ = __ldg(g + word_index(x, t << 5, TY));
            const int y0 = t << 5, len = min(32, H - y0);
            if (words4) {                         // every row starts 4-byte aligned: four cells per load
                const uint32_t *w4 = reinterpret_cast<const uint32_t *>(wr + y0);
                for (int j = 0; j < (len >> 2); ++j) {
                    const uint32_t v = __ldg(w4 + j), m = occ >> (4 * j);
#pragma unroll
                    for (int b = 0; b < 4; ++b) sum += ((m >> b) & 1u) ? 0u : ((v >> (8 * b)) & 0xffu);
                }
            } else {
                for (int j = 0; j < len; ++j) sum += ((occ >> j) & 1u) ? 0u : (uint32_t)__ldg(wr + y0 + j);
            }
        }
        uint32_t incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(RRTK_FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (t < TY) cp[t] = carry + incl - sum;
        carry += __shfl_sync(RRTK_FULL, incl, 31);
    }
    if (lane == 0) ix.rows[(size_t)world * (W + 1) + x + 1] = carry;
}

// one block per world: rows[0] = 0 and the row totals in rows[1 .. W] become inclusive prefixes; tot[world] = rows[W]
constexpr int kRowThreads = 1024;
__global__ void __launch_bounds__(kRowThreads) weight_rows_kernel(int W, WeightIndex ix)
{
    __shared__ long long s_warp[kRowThreads / 32];
    const int world = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long *rp = ix.rows + (size_t)world * (W + 1);
    const int per = (W + kRowThreads - 1) / kRowThreads;
    const int x0 = 1 + tid * per, x1 = min(W + 1, x0 + per);
    long long acc = 0;
    for (int x = x0; x < x1; ++x) acc += rp[x];
    long long incl = acc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long v = __shfl_up_sync(RRTK_FULL, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    long long run = incl - acc;
    for (int w = 0; w < warp; ++w) run += s_warp[w];
    for (int x = x0; x < x1; ++x) { run += rp[x]; rp[x] = run; }
    if (tid == 0) rp[0] = 0;
    if (x0 <= W && W < x1) ix.tot[world] = run;
    if (W == 0 && tid == 0) ix.tot[world] = 0;
}

int weight_index_launch(const uint32_t *d_bits, const uint8_t *d_weights, int nworlds, int W, int H, void *d_index, cudaStream_t st)
{
    if (nworlds == 0) return RRTK_OK;
    WeightIndex ix(d_index, nworlds, W, H);
    const long long warps = (long long)nworlds * W;
    // the weights may start anywhere (a view into a caller's buffer): whole words only when the base and every row are aligned
    const bool words4 = (H & 3) == 0 && (reinterpret_cast<uintptr_t>(d_weights) & 3) == 0;
    weight_chunks_kernel<<<(unsigned)((warps + kIndexWarps - 1) / kIndexWarps), kIndexWarps * 32, 0, st>>>(d_bits, d_weights, nworlds, W, H,
                                                                                                          words4, ix);
    RRTK_CUDA(cudaGetLastError());
    weight_rows_kernel<<<nworlds, kRowThreads, 0, st>>>(W, ix);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

int weighted_streams_launch(const uint32_t *d_bits, const uint8_t *d_weights, const void *d_index, int nworlds, int W, int H,
                            const rrtk_plan_desc *d_plans, int nplans, uint64_t *d_state, uint32_t *d_carry, int n, int16_t *d_samples,
                            int optin, cudaStream_t st)
{
    WeightIndex ix(const_cast<void *>(d_index), nworlds, W, H);
    const WeightedSelect sel{d_bits, d_weights, ix.tot, ix.rows, ix.chunks};
    return sample_launch(sel, W, H, d_plans, nplans, d_state, n, d_samples, optin, st, d_carry ? d_state : nullptr, d_carry);
}

// ---- the ellipse-phase unit-disc stream of RRTStarInformed.plan (rrt.py:579-587, 694-701) -------------------------
// The reference draws from ONE generator: free[choice(nfree)] in every iteration up to and including the first solution
// vertex f (rrt.py:240), then unitball() = two uniform(0, 1) draws per iteration (rrt.py:582-583).  Given f from a probe
// launch, plan p's generator is replayed past its m = f + 1 bounded draws (m = n when f < 0) by thread 0 -- rejections
// are rare, so that is about m / 2 PCG steps -- and the ellipse phase, a fixed two 64-bit outputs per row, is split over
// the block: thread t writes rows f+1+t, f+1+t+T, ... (coalesced), jumping 2T - 2 steps between its rows.
//   uniform(0, 1) = (next64 >> 11) * 2^-53 (numpy's next_double: no use of the buffered 32-bit half)
//   ball = (sqrt(u1) cos(a), sqrt(u1) sin(a)),  a = 6.283185307179586 * u2  (Python's 2 * np.pi * u)
// sqrt and the products are correctly rounded; cos / sin are CUDA's (<= 2 ulp), so a ball may differ from numpy's in its
// last bits.  Rows <= f (every row when f < 0) are 0.0, as RRTStarInformed.plan hands them to the plan kernel.
constexpr int kBallThreads = 256;

__global__ void __launch_bounds__(kBallThreads)
ball_stream_kernel(const int *__restrict__ rowcum, int W, const rrtk_plan_desc *__restrict__ plans, int n,
                   const unsigned long long *state, const uint32_t *carry, const long long *__restrict__ first, int first_stride,
                   double2 *__restrict__ balls, unsigned long long *state_out, uint32_t *carry_out)
{
    __shared__ unsigned long long s_st[4];       // generator after the bounded draws
    __shared__ int s_first;
    const int plan = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        // only this thread reads the plan's inputs before the barrier, so state_out / carry_out may alias state / carry
        Pcg64 g;
        g.hi = state[4 * plan]; g.lo = state[4 * plan + 1];
        g.inc_hi = state[4 * plan + 2]; g.inc_lo = state[4 * plan + 3];
        g.has32 = false; g.buf32 = 0;
        if (carry) { g.has32 = carry[2 * plan] != 0; g.buf32 = carry[2 * plan + 1]; }
        long long f = first[(size_t)plan * first_stride];
        if (f < 0 || f >= n) f = -1;             // f = n - 1 and "none" consume the same draws and write the same rows
        const int fi = (int)f;
        const uint32_t nfree = (uint32_t)__ldg(rowcum + (size_t)plans[plan].world * (W + 1) + W);
        if (nfree > 1u) {                        // numpy returns the single value without touching the generator
            const int m = fi < 0 ? n : fi + 1;
            for (int i = 0; i < m; ++i) g.bounded(nfree);
        }
        s_st[0] = g.hi; s_st[1] = g.lo; s_st[2] = g.inc_hi; s_st[3] = g.inc_lo;
        s_first = fi;
        if (carry_out) { carry_out[2 * plan] = g.has32 ? 1u : 0u; carry_out[2 * plan + 1] = g.buf32; }
        if (state_out) {                         // the generator as the planner object holds it after plan()
            if (fi >= 0) pcg_jump(g, 2ull * (unsigned long long)(n - 1 - fi));
            state_out[4 * plan] = g.hi; state_out[4 * plan + 1] = g.lo; state_out[4 * plan + 2] = g.inc_hi; state_out[4 * plan + 3] = g.inc_lo;
        }
    }
    __syncthreads();
    const int fi = s_first;
    const int r0 = fi < 0 ? n : fi + 1;          // first ellipse-phase row
    double2 *out = balls + (size_t)plan * n;
    for (int i = tid; i < r0; i += kBallThreads) out[i] = make_double2(0.0, 0.0);
    if (r0 >= n) return;
    Pcg64 g;
    g.hi = s_st[0]; g.lo = s_st[1]; g.inc_hi = s_st[2]; g.inc_lo = s_st[3];
    g.has32 = false; g.buf32 = 0;
    pcg_jump(g, 2ull * (unsigned long long)tid);
    const PcgAffine skip = pcg_affine(g.inc_hi, g.inc_lo, 2ull * kBallThreads - 2ull);
    for (int i = r0 + tid; i < n; i += kBallThreads) {
        const double u1 = __dmul_rn((double)(g.next64() >> 11), 1.0 / 9007199254740992.0);
        const double u2 = __dmul_rn((double)(g.next64() >> 11), 1.0 / 9007199254740992.0);
        const double a = __dmul_rn(6.283185307179586, u2);
        double s, c;
        sincos(a, &s, &c);
        const double r = __dsqrt_rn(u1);
        out[i] = make_double2(__dmul_rn(r, c), __dmul_rn(r, s));
        pcg_apply(g, skip);
    }
}

int ball_streams_launch(const int32_t *d_rowcum, int W, const rrtk_plan_desc *d_plans, int nplans, int n, const uint64_t *d_state,
                        const uint32_t *d_carry, const int64_t *d_first, int first_stride, double *d_balls, uint64_t *d_state_out,
                        uint32_t *d_carry_out, cudaStream_t st)
{
    if (nplans == 0) return RRTK_OK;
    ball_stream_kernel<<<nplans, kBallThreads, 0, st>>>(d_rowcum, W, d_plans, n, reinterpret_cast<const unsigned long long *>(d_state), d_carry,
                                                        reinterpret_cast<const long long *>(d_first), first_stride,
                                                        reinterpret_cast<double2 *>(d_balls),
                                                        reinterpret_cast<unsigned long long *>(d_state_out), d_carry_out);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

}  // namespace rrtk
