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

// one block per plan: the generator's raw outputs in parallel slices, Lemire's rejection as a compaction, then
// ranks -> cells in parallel.  The sequential generator remains as the fallback for a stream with more than kRawSlack
// rejections (probability ~ (n * nfree / 2^32)^62 / 62!).
__global__ void __launch_bounds__(kSampleThreads)
sample_stream_kernel(const uint32_t *__restrict__ bits, const int *__restrict__ rowcum, int W, int H,
                     const rrtk_plan_desc *__restrict__ plans, const unsigned long long *__restrict__ state, int n,
                     short2 *__restrict__ samples, unsigned long long *__restrict__ state_out, uint32_t *__restrict__ carry)
{
    extern __shared__ uint32_t s_mem[];
    uint32_t *s_rank = s_mem;                    // n bounded draws
    uint32_t *s_raw = s_mem + n;                 // raw 32-bit values in the order numpy's next_uint32 hands them out
    int *s_rowcum = reinterpret_cast<int *>(s_mem + 2 * n + kRawSlack + 4);      // W + 1 row offsets of this plan's world
    __shared__ int s_warp[kSampleThreads / 32];
    __shared__ int s_consumed;                   // raw values used up by the n draws (-1: not enough generated)
    const int plan = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int world = plans[plan].world;
    const int *rc = rowcum + (size_t)world * (W + 1);
    const uint32_t nfree = (uint32_t)__ldg(rc + W);
    for (int x = tid; x <= W; x += kSampleThreads) s_rowcum[x] = __ldg(rc + x);    // visible after the barriers below
    Pcg64 g0;
    g0.hi = state[4 * plan]; g0.lo = state[4 * plan + 1];
    g0.inc_hi = state[4 * plan + 2]; g0.inc_lo = state[4 * plan + 3];
    g0.has32 = false; g0.buf32 = 0;
    if (carry) { g0.has32 = carry[2 * plan] != 0; g0.buf32 = carry[2 * plan + 1]; }   // numpy's has_uint32 / uinteger
    const int off = g0.has32 ? 1 : 0;
    if (nfree <= 1u) {                           // numpy returns the single value without touching the generator
        for (int i = tid; i < n; i += kSampleThreads) s_rank[i] = 0;
        if (tid == 0) {
            if (state_out) { state_out[4 * plan] = g0.hi; state_out[4 * plan + 1] = g0.lo; state_out[4 * plan + 2] = g0.inc_hi; state_out[4 * plan + 3] = g0.inc_lo; }
        }
        __syncthreads();
    } else {
        const int nraw = n + kRawSlack;                                   // raw values wanted: indices 0 .. nraw-1
        const int n64 = (nraw - off + 1) >> 1;                            // 64-bit outputs that cover them
        const int per = (n64 + kSampleThreads - 1) / kSampleThreads;      // outputs per thread
        {
            Pcg64 g = g0;
            const int k0 = tid * per;
            if (k0 < n64) {
                pcg_jump(g, (unsigned long long)k0);
                const int k1 = min(n64, k0 + per);
                for (int k = k0; k < k1; ++k) {
                    const unsigned long long v = g.next64();
                    s_raw[off + 2 * k] = (uint32_t)v;
                    s_raw[off + 2 * k + 1] = (uint32_t)(v >> 32);
                }
            }
            if (tid == 0 && off) s_raw[0] = g0.buf32;
        }
        __syncthreads();
        // compaction: thread t owns raw indices [t * span, (t + 1) * span)
        const int total = off + 2 * n64;                                  // raw values available (>= nraw)
        const int span = (total + kSampleThreads - 1) / kSampleThreads;
        const uint32_t thr = (0xffffffffu - (nfree - 1u)) % nfree;        // Lemire's threshold
        const int r0 = tid * span, r1 = min(total, r0 + span);
        int acc = 0;
        for (int r = r0; r < r1; ++r) acc += ((uint32_t)((unsigned long long)s_raw[r] * nfree) >= thr) ? 1 : 0;
        int incl = acc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(RRTK_FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        if (tid == 0) s_consumed = -1;
        __syncthreads();
        int before = incl - acc;
        for (int w = 0; w < warp; ++w) before += s_warp[w];
        for (int r = r0; r < r1; ++r) {
            const unsigned long long m = (unsigned long long)s_raw[r] * nfree;
            if ((uint32_t)m >= thr) {
                if (before < n) s_rank[before] = (uint32_t)(m >> 32);
                if (before == n - 1) s_consumed = r + 1;
                ++before;
            }
        }
        __syncthreads();
        if (s_consumed < 0) {                    // not enough accepted values in the window: the plain sequential generator
            if (tid == 0) {
                Pcg64 g = g0;
                for (int i = 0; i < n; ++i) s_rank[i] = g.bounded(nfree);
                if (state_out) { state_out[4 * plan] = g.hi; state_out[4 * plan + 1] = g.lo; state_out[4 * plan + 2] = g.inc_hi; state_out[4 * plan + 3] = g.inc_lo; }
                if (carry) { carry[2 * plan] = g.has32 ? 1u : 0u; carry[2 * plan + 1] = g.buf32; }
            }
        } else if (tid == 0 && (state_out || carry)) {
            // the generator as the next plan() of the same planner object finds it (rrt.py:85: one rand_gen per object)
            const int used = s_consumed - off;                            // raw values taken from fresh 64-bit outputs
            const int out64 = (used + 1) >> 1;
            Pcg64 g = g0;
            pcg_jump(g, (unsigned long long)out64);
            if (state_out) { state_out[4 * plan] = g.hi; state_out[4 * plan + 1] = g.lo; state_out[4 * plan + 2] = g.inc_hi; state_out[4 * plan + 3] = g.inc_lo; }
            if (carry) {
                const bool half = used > 0 ? (used & 1) != 0 : g0.has32 && s_consumed == 0;
                carry[2 * plan] = half ? 1u : 0u;
                carry[2 * plan + 1] = half ? s_raw[s_consumed] : (used > 0 ? s_raw[s_consumed - 1] : g0.buf32);
            }
        }
        __syncthreads();
    }
    const uint32_t *g = bits + (size_t)world * grid_words(W, H);
    const int TY = tiles_y(H);
    short2 *out = samples + (size_t)plan * n;
    for (int i = tid; i < n; i += kSampleThreads) out[i] = rank_to_cell(g, s_rowcum, W, TY, (int)s_rank[i]);
}

// n too large for the raw window in shared memory: thread 0 runs the generator sequentially
__global__ void sample_stream_seq_kernel(const uint32_t *__restrict__ bits, const int *__restrict__ rowcum, int W, int H,
                                         const rrtk_plan_desc *__restrict__ plans, const unsigned long long *__restrict__ state, int n,
                                         short2 *__restrict__ samples, unsigned long long *__restrict__ state_out, uint32_t *__restrict__ carry)
{
    extern __shared__ uint32_t s_rank[];
    const int plan = blockIdx.x;
    const int world = plans[plan].world;
    const int *rc = rowcum + (size_t)world * (W + 1);
    const uint32_t nfree = (uint32_t)__ldg(rc + W);
    if (threadIdx.x == 0) {
        Pcg64 g;
        g.hi = state[4 * plan]; g.lo = state[4 * plan + 1];
        g.inc_hi = state[4 * plan + 2]; g.inc_lo = state[4 * plan + 3];
        g.has32 = false; g.buf32 = 0;
        if (carry) { g.has32 = carry[2 * plan] != 0; g.buf32 = carry[2 * plan + 1]; }
        for (int i = 0; i < n; ++i) s_rank[i] = nfree ? g.bounded(nfree) : 0;
        if (state_out) {
            state_out[4 * plan] = g.hi; state_out[4 * plan + 1] = g.lo;
            state_out[4 * plan + 2] = g.inc_hi; state_out[4 * plan + 3] = g.inc_lo;
        }
        if (carry) { carry[2 * plan] = g.has32 ? 1u : 0u; carry[2 * plan + 1] = g.buf32; }
    }
    __syncthreads();
    const uint32_t *g = bits + (size_t)world * grid_words(W, H);
    const int TY = tiles_y(H);
    short2 *out = samples + (size_t)plan * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = rank_to_cell(g, rc, W, TY, (int)s_rank[i]);
}

int sample_streams_launch(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H, const rrtk_plan_desc *d_plans,
                          int nplans, const uint64_t *d_state, int n, int16_t *d_samples, int optin, cudaStream_t st,
                          uint64_t *d_state_out, uint32_t *d_carry)
{
    if (nplans == 0 || n == 0) return RRTK_OK;
    const size_t smem = ((size_t)2 * n + kRawSlack + 4 + W + 1) * 4;      // bounded draws + raw 32-bit values + row offsets
    const size_t smem_seq = (size_t)n * 4;
    const unsigned long long *st64 = reinterpret_cast<const unsigned long long *>(d_state);
    if (smem <= (size_t)optin) {
        RRTK_CUDA(cudaFuncSetAttribute(sample_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        sample_stream_kernel<<<nplans, kSampleThreads, smem, st>>>(d_bits, d_rowcum, W, H, d_plans, st64, n, reinterpret_cast<short2 *>(d_samples),
                                                                  reinterpret_cast<unsigned long long *>(d_state_out), d_carry);
    } else if (smem_seq <= (size_t)optin) {
        RRTK_CUDA(cudaFuncSetAttribute(sample_stream_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_seq));
        sample_stream_seq_kernel<<<nplans, 128, smem_seq, st>>>(d_bits, d_rowcum, W, H, d_plans, st64, n, reinterpret_cast<short2 *>(d_samples),
                                                               reinterpret_cast<unsigned long long *>(d_state_out), d_carry);
    } else {
        set_error("sample stream of n=%d does not fit shared memory", n);
        return RRTK_ERR_CAPACITY;
    }
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
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
