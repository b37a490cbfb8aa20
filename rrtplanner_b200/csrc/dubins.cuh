// Dubins primitive on the device ("Dubins Primitive Module", README.md:12 of the reference -- advertised there, absent
// from its tree; the specification is oracle/rewire_oracle.c and every function here must agree with it bit for bit).
//
// All arithmetic is IEEE-754 double add / sub / mul / div / sqrt / floor in the order the specification fixes; the
// library is compiled with --fmad=false so nothing is contracted.  atan2 / sin / cos are the specification's own
// polynomials (dm_*), not CUDA's libm, because last-ulp differences would change strict cost comparisons and hence trees.
#pragma once
#include <math_constants.h>

#include "common.cuh"

#ifndef RRTK_DM_INLINE
#define RRTK_DM_INLINE __noinline__
#endif

namespace rrtk {

#define DM_PI 3.14159265358979323846
#define DM_TWO_PI 6.28318530717958647692
#define DM_INV_TWO_PI 0.15915494309189533577
#define DM_HALF_PI 1.57079632679489661923
#define DM_QUARTER_PI 0.78539816339744830962
#define DM_TWO_OVER_PI 0.63661977236758134308
#define DM_TAN_PI_8 0.41421356237309504880

// atan(z), |z| <= tan(pi/8): z * sum_{k<16} (-1)^k z^(2k) / (2k+1) as E(s^2) + s * O(s^2), s = z^2 (two Horner chains)
__device__ __forceinline__ double dm_atan_small(double z)
{
    const double s = z * z, s2 = s * s;
    double e = 1.0 / 29.0, o = -1.0 / 31.0;
    e = e * s2 + 1.0 / 25.0;  o = o * s2 - 1.0 / 27.0;
    e = e * s2 + 1.0 / 21.0;  o = o * s2 - 1.0 / 23.0;
    e = e * s2 + 1.0 / 17.0;  o = o * s2 - 1.0 / 19.0;
    e = e * s2 + 1.0 / 13.0;  o = o * s2 - 1.0 / 15.0;
    e = e * s2 + 1.0 / 9.0;   o = o * s2 - 1.0 / 11.0;
    e = e * s2 + 1.0 / 5.0;   o = o * s2 - 1.0 / 7.0;
    e = e * s2 + 1.0;         o = o * s2 - 1.0 / 3.0;
    return z * (e + s * o);
}

__device__ RRTK_DM_INLINE double dm_atan2(double y, double x)
{
    if (x == 0.0 && y == 0.0) return 0.0;
    const double ax = fabs(x), ay = fabs(y);
    const bool swap = ay > ax;
    const double num = swap ? ax : ay, den = swap ? ay : ax;
    const bool hi = num > DM_TAN_PI_8 * den;
    const double zn = hi ? num - den : num, zd = hi ? num + den : den;
    double r = dm_atan_small(zn / zd);
    if (hi) r = DM_QUARTER_PI + r;
    if (swap) r = DM_HALF_PI - r;
    if (x < 0.0) r = DM_PI - r;
    if (y < 0.0) r = -r;
    return r;
}

// quadrant k = floor(a * 2/pi + 1/2), r = a - k * pi/2, Taylor polynomials on |r| <= pi/4
// (sin, cos) returned by value: a non-inlined function hands 16 bytes back in registers, while reference outputs would
// go through local memory (which misses the small L1 left beside the plan blocks' shared memory)
__device__ RRTK_DM_INLINE double2 dm_sincos2(double a)
{
    double sn, cs;
    const double kf = floor(a * DM_TWO_OVER_PI + 0.5);
    const double r = a - kf * DM_HALF_PI;
    const double s = r * r;
    double ps = -1.0 / 1307674368000.0;
    ps = ps * s + 1.0 / 6227020800.0;
    ps = ps * s - 1.0 / 39916800.0;
    ps = ps * s + 1.0 / 362880.0;
    ps = ps * s - 1.0 / 5040.0;
    ps = ps * s + 1.0 / 120.0;
    ps = ps * s - 1.0 / 6.0;
    ps = ps * s + 1.0;
    ps = ps * r;
    double pc = 1.0 / 20922789888000.0;
    pc = pc * s - 1.0 / 87178291200.0;
    pc = pc * s + 1.0 / 479001600.0;
    pc = pc * s - 1.0 / 3628800.0;
    pc = pc * s + 1.0 / 40320.0;
    pc = pc * s - 1.0 / 720.0;
    pc = pc * s + 1.0 / 24.0;
    pc = pc * s - 1.0 / 2.0;
    pc = pc * s + 1.0;
    const long long k = (long long)kf;
    switch ((int)(k & 3)) {
        case 0: sn = ps; cs = pc; break;
        case 1: sn = pc; cs = -ps; break;
        case 2: sn = -ps; cs = -pc; break;
        default: sn = -pc; cs = ps; break;
    }
    return make_double2(sn, cs);
}
__device__ __forceinline__ void dm_sincos(double a, double &sn, double &cs)
{
    const double2 r = dm_sincos2(a);
    sn = r.x; cs = r.y;
}

// angle into [0, 2 pi); a result within 1e-9 of a full turn (an exact 0 that rounded below) snaps to 0
__device__ __forceinline__ double dm_mod2pi(double x)
{
    const double r = x - DM_TWO_PI * floor(x * DM_INV_TWO_PI);
    return (r < 0.0 || r > DM_TWO_PI - 1e-9) ? 0.0 : r;
}
__device__ __forceinline__ double dm_acos(double v) { return dm_atan2(sqrt(1.0 - v * v), v); }

struct DubinsPath {
    int word;               // 0..5 = LSL RSR LSR RSL RLR LRL, -1 none
    double t, p, q, len;    // normalised segment lengths, total length in cells
};

struct DubinsIn { double d, dd, alpha, beta, sa, ca, sb, cb, cab; };

// tab[h] = (sin, cos) of heading h, i.e. dm_sincos(h * 2 pi / NH) -- the same values the specification recomputes
__device__ __forceinline__ void dubins_setup(int dx, int dy, int h0, int h1, int NH, double rho, const double2 *tab, DubinsIn &g)
{
    const double dth = DM_TWO_PI / (double)NH;
    const double th0 = (double)h0 * dth, th1 = (double)h1 * dth;
    const double2 a0 = tab[h0], a1 = tab[h1];
    int hd = (h0 - h1) % NH;
    if (hd < 0) hd += NH;
    const double D = sqrt((double)((long long)dx * dx + (long long)dy * dy));
    g.d = D * (1.0 / rho);
    g.dd = g.d * g.d;
    double cphi = 1.0, sphi = 0.0;
    if (D > 0.0) { const double inv = 1.0 / D; cphi = (double)dx * inv; sphi = (double)dy * inv; }
    const double phi = dm_atan2((double)dy, (double)dx);
    g.alpha = dm_mod2pi(th0 - phi);
    g.beta = dm_mod2pi(th1 - phi);
    g.sa = a0.x * cphi - a0.y * sphi; g.ca = a0.y * cphi + a0.x * sphi;
    g.sb = a1.x * cphi - a1.y * sphi; g.cb = a1.y * cphi + a1.x * sphi;
    g.cab = tab[hd].y;
}

__device__ __forceinline__ bool dubins_word(const DubinsIn &g, int w, double &t, double &p, double &q)
{
    const double d = g.d, dd = g.dd, alpha = g.alpha, beta = g.beta;
    const double sa = g.sa, ca = g.ca, sb = g.sb, cb = g.cb, cab = g.cab;
    double tmp, psq;
    switch (w) {
        case 0:
            psq = 2.0 + dd - 2.0 * cab + 2.0 * d * (sa - sb);
            if (psq < 0.0) return false;
            tmp = dm_atan2(cb - ca, d + sa - sb);
            t = dm_mod2pi(tmp - alpha); p = sqrt(psq); q = dm_mod2pi(beta - tmp);
            return true;
        case 1:
            psq = 2.0 + dd - 2.0 * cab + 2.0 * d * (sb - sa);
            if (psq < 0.0) return false;
            tmp = dm_atan2(ca - cb, d - sa + sb);
            t = dm_mod2pi(alpha - tmp); p = sqrt(psq); q = dm_mod2pi(tmp - beta);
            return true;
        case 2:
            psq = dd - 2.0 + 2.0 * cab + 2.0 * d * (sa + sb);
            if (psq < 0.0) return false;
            p = sqrt(psq);
            tmp = dm_atan2(-ca - cb, d + sa + sb) - dm_atan2(-2.0, p);
            t = dm_mod2pi(tmp - alpha); q = dm_mod2pi(tmp - dm_mod2pi(beta));
            return true;
        case 3:
            psq = dd - 2.0 + 2.0 * cab - 2.0 * d * (sa + sb);
            if (psq < 0.0) return false;
            p = sqrt(psq);
            tmp = dm_atan2(ca + cb, d - sa - sb) - dm_atan2(2.0, p);
            t = dm_mod2pi(alpha - tmp); q = dm_mod2pi(beta - tmp);
            return true;
        case 4:
            tmp = (6.0 - dd + 2.0 * cab + 2.0 * d * (sa - sb)) * 0.125;
            if (fabs(tmp) > 1.0) return false;
            p = dm_mod2pi(DM_TWO_PI - dm_acos(tmp));
            t = dm_mod2pi(alpha - dm_atan2(ca - cb, d - sa + sb) + p * 0.5);
            q = dm_mod2pi(alpha - beta - t + p);
            return true;
        default:
            tmp = (6.0 - dd + 2.0 * cab + 2.0 * d * (sb - sa)) * 0.125;
            if (fabs(tmp) > 1.0) return false;
            p = dm_mod2pi(DM_TWO_PI - dm_acos(tmp));
            t = dm_mod2pi(p * 0.5 - alpha + dm_atan2(cb - ca, d + sa - sb));
            q = dm_mod2pi(dm_mod2pi(beta) - alpha - t + p);
            return true;
    }
}

// shortest word from (0, 0, h0) to (dx, dy, h1); ties to the first word in the order above.  Same operations per word as
// dubins_word (so the same bits); the two angles that LSL / LRL and RSR / RLR share are evaluated once.
__device__ __noinline__ void dubins_shortest(int dx, int dy, int h0, int h1, int NH, double rho, const double2 *tab, DubinsPath &out)
{
    DubinsIn g;
    dubins_setup(dx, dy, h0, h1, NH, rho, tab, g);
    const double d = g.d, dd = g.dd, alpha = g.alpha, beta = g.beta;
    const double sa = g.sa, ca = g.ca, sb = g.sb, cb = g.cb, cab = g.cab;
    out.word = -1; out.len = CUDART_INF; out.t = out.p = out.q = 0.0;
    const double a_lsl = dm_atan2(cb - ca, d + sa - sb);
    const double a_rsr = dm_atan2(ca - cb, d - sa + sb);
    double t, p, q, tmp, psq, len;
#define RRTK_DUBINS_TAKE(W)                                                                  \
    len = ((t + p) + q) * rho;                                                              \
    if (len < out.len) { out.len = len; out.word = (W); out.t = t; out.p = p; out.q = q; }
    psq = 2.0 + dd - 2.0 * cab + 2.0 * d * (sa - sb);
    if (!(psq < 0.0)) {
        t = dm_mod2pi(a_lsl - alpha); p = sqrt(psq); q = dm_mod2pi(beta - a_lsl);
        RRTK_DUBINS_TAKE(0)
    }
    psq = 2.0 + dd - 2.0 * cab + 2.0 * d * (sb - sa);
    if (!(psq < 0.0)) {
        t = dm_mod2pi(alpha - a_rsr); p = sqrt(psq); q = dm_mod2pi(a_rsr - beta);
        RRTK_DUBINS_TAKE(1)
    }
    psq = dd - 2.0 + 2.0 * cab + 2.0 * d * (sa + sb);
    if (!(psq < 0.0)) {
        p = sqrt(psq);
        tmp = dm_atan2(-ca - cb, d + sa + sb) - dm_atan2(-2.0, p);
        t = dm_mod2pi(tmp - alpha); q = dm_mod2pi(tmp - dm_mod2pi(beta));
        RRTK_DUBINS_TAKE(2)
    }
    psq = dd - 2.0 + 2.0 * cab - 2.0 * d * (sa + sb);
    if (!(psq < 0.0)) {
        p = sqrt(psq);
        tmp = dm_atan2(ca + cb, d - sa - sb) - dm_atan2(2.0, p);
        t = dm_mod2pi(alpha - tmp); q = dm_mod2pi(beta - tmp);
        RRTK_DUBINS_TAKE(3)
    }
    tmp = (6.0 - dd + 2.0 * cab + 2.0 * d * (sa - sb)) * 0.125;
    if (!(fabs(tmp) > 1.0)) {
        p = dm_mod2pi(DM_TWO_PI - dm_acos(tmp));
        t = dm_mod2pi(alpha - a_rsr + p * 0.5);
        q = dm_mod2pi(alpha - beta - t + p);
        RRTK_DUBINS_TAKE(4)
    }
    tmp = (6.0 - dd + 2.0 * cab + 2.0 * d * (sb - sa)) * 0.125;
    if (!(fabs(tmp) > 1.0)) {
        p = dm_mod2pi(DM_TWO_PI - dm_acos(tmp));
        t = dm_mod2pi(p * 0.5 - alpha + a_lsl);
        q = dm_mod2pi(dm_mod2pi(beta) - alpha - t + p);
        RRTK_DUBINS_TAKE(5)
    }
#undef RRTK_DUBINS_TAKE
}

// (t, p, q, len) of one given word (the one dubins_shortest chose for the same arguments: identical operations, identical bits)
__device__ __noinline__ void dubins_rebuild(int dx, int dy, int h0, int h1, int NH, double rho, const double2 *tab, int word, DubinsPath &out)
{
    DubinsIn g;
    dubins_setup(dx, dy, h0, h1, NH, rho, tab, g);
    out.word = word;
    out.t = out.p = out.q = 0.0;
    out.len = CUDART_INF;
    double t, p, q;
    if (word >= 0 && dubins_word(g, word, t, p, q)) { out.t = t; out.p = p; out.q = q; out.len = ((t + p) + q) * rho; }
    else out.word = -1;
}

// segment kinds of word w (0 left arc, 1 straight, 2 right arc) for LSL RSR LSR RSL RLR LRL: three 2-bit fields per word,
// six words packed in one constant (a lookup array would live in local memory)
__device__ __forceinline__ int dubins_seg(int word, int i)
{
    constexpr unsigned long long kCodes = (4ull << 0) | (38ull << 6) | (36ull << 12) | (6ull << 18) | (34ull << 24) | (8ull << 30);
    return (int)((kCodes >> (6 * word + 2 * i)) & 3ull);
}

struct Pose { double x, y, th; };

// one segment from pose a, whose heading's (sin, cos) = (sa, ca) the caller already has; returns the end pose and,
// through (se, ce), the (sin, cos) of its heading.  Same operations as the specification's advance().
__device__ __forceinline__ Pose dubins_advance(Pose a, double sa, double ca, int kind, double len, double rho, double &se, double &ce)
{
    if (kind == 1) {
        a.x = a.x + rho * len * ca;
        a.y = a.y + rho * len * sa;
        se = sa; ce = ca;
    } else if (kind == 0) {
        dm_sincos(a.th + len, se, ce);
        a.x = a.x + rho * (se - sa);
        a.y = a.y + rho * (ca - ce);
        a.th = a.th + len;
    } else {
        dm_sincos(a.th - len, se, ce);
        a.x = a.x + rho * (sa - se);
        a.y = a.y + rho * (ce - ca);
        a.th = a.th - len;
    }
    return a;
}

// the path cut at its two junctions: q0 start, q1 after the first segment, q2 after the second, each with the
// (sin, cos) of its heading (the specification recomputes them per point; the values are the same)
struct DubinsTrack {
    Pose q0, q1, q2;
    double s0, c0, s1, c1, s2, c2;
    int k0, k1, k2;
    double t, p, rho, inv_rho;
};

__device__ __forceinline__ DubinsTrack dubins_track(int x0, int y0, int h0, int NH, double rho, const DubinsPath &w)
{
    DubinsTrack tr;
    tr.k0 = dubins_seg(w.word, 0); tr.k1 = dubins_seg(w.word, 1); tr.k2 = dubins_seg(w.word, 2);
    tr.t = w.t; tr.p = w.p; tr.rho = rho; tr.inv_rho = 1.0 / rho;
    tr.q0.x = (double)x0; tr.q0.y = (double)y0; tr.q0.th = (double)h0 * (DM_TWO_PI / (double)NH);
    dm_sincos(tr.q0.th, tr.s0, tr.c0);
    tr.q1 = dubins_advance(tr.q0, tr.s0, tr.c0, tr.k0, w.t, rho, tr.s1, tr.c1);
    tr.q2 = dubins_advance(tr.q1, tr.s1, tr.c1, tr.k1, w.p, rho, tr.s2, tr.c2);
    return tr;
}

// pose at arc length s (cells) from the start
__device__ __forceinline__ Pose dubins_point(const DubinsTrack &tr, double s)
{
    const double u = s * tr.inv_rho;
    double se, ce;
    if (u < tr.t) return dubins_advance(tr.q0, tr.s0, tr.c0, tr.k0, u, tr.rho, se, ce);
    const double u2 = u - tr.t;
    if (u2 < tr.p) return dubins_advance(tr.q1, tr.s1, tr.c1, tr.k1, u2, tr.rho, se, ce);
    return dubins_advance(tr.q2, tr.s2, tr.c2, tr.k2, u2 - tr.p, tr.rho, se, ce);
}

__device__ __forceinline__ bool cell_blocked(const uint32_t *bits, int W, int H, int TY, double x, double y)
{
    const double fx = floor(x + 0.5), fy = floor(y + 0.5);
    if (!(fx >= 0.0 && fx < (double)W && fy >= 0.0 && fy < (double)H)) return true;
    const int cx = (int)fx, cy = (int)fy;
    return (__ldg(bits + word_index(cx, cy, TY)) >> (cy & 31)) & 1u;
}

// Heading layer of a pose with angle th on L layer grids (include/rrtk.h, rrtk_plan2_batch_layers): floor(th * (L / 2 pi) + 1/2)
// mod L, non-negative.  The same double operations as the specification (oracle/body_oracle.c, body_layer).
__device__ __forceinline__ int body_layer(double th, int L)
{
    const double f = floor(__dadd_rn(__dmul_rn(th, (double)L / DM_TWO_PI), 0.5));
    const int l = (int)((long long)f % L);
    return l < 0 ? l + L : l;
}

// warp-cooperative sampled collision test of the path w from (x0, y0, h0) to cell (x1, y1): points at arc length
// k * ds, k = 0 .. floor(len / ds), one per lane, two rounds of 32 in flight together (their grid reads overlap),
// plus the target cell.  All lanes must pass the same path.
// LAYERS: bits is the first of L heading-layer grids lstride words apart; a pose tests the layer of its own angle, the target
// cell the layer of heading h1 (the angle dubins_track gives a vertex heading).  Otherwise h1, lstride and L are not read.
#ifndef RRTK_FREE_INLINE
#define RRTK_FREE_INLINE __forceinline__
#endif
// Inlined by default; as a real call (-DRRTK_FREE_INLINE=__noinline__, measured: -4 %) it would have the register budget to
// itself but pays for saving the plan loop's state around every test.
template <bool LAYERS>
__device__ RRTK_FREE_INLINE bool dubins_free_path_t(const uint32_t *bits, int W, int H, int TY, int x0, int y0, int h0, int x1, int y1,
                                                   int h1, int NH, double rho, double ds, int word, double t, double p, double len,
                                                   int lane, size_t lstride, int L)
{
    if (word < 0) return false;
    DubinsPath w;
    w.word = word; w.t = t; w.p = p; w.q = 0.0; w.len = len;
    const DubinsTrack tr = dubins_track(x0, y0, h0, NH, rho, w);
    const long long ns = (long long)floor(len / ds);
    for (long long base = 0; base <= ns; base += 64) {
        const long long ka = base + lane, kb = base + 32 + lane;
        bool hit = false;
        if (ka <= ns) {
            const Pose a = dubins_point(tr, (double)ka * ds);
            hit = cell_blocked(LAYERS ? bits + (size_t)body_layer(a.th, L) * lstride : bits, W, H, TY, a.x, a.y);
        }
        if (kb <= ns) {
            const Pose b = dubins_point(tr, (double)kb * ds);
            hit |= cell_blocked(LAYERS ? bits + (size_t)body_layer(b.th, L) * lstride : bits, W, H, TY, b.x, b.y);
        }
        if (__any_sync(RRTK_FULL, hit)) return false;
    }
    const uint32_t *g1 = LAYERS ? bits + (size_t)body_layer((double)h1 * (DM_TWO_PI / (double)NH), L) * lstride : bits;
    return !((__ldg(g1 + word_index(x1, y1, TY)) >> (y1 & 31)) & 1u);
}

__device__ RRTK_FREE_INLINE bool dubins_free_path(const uint32_t *bits, int W, int H, int TY, int x0, int y0, int h0, int x1, int y1,
                                                 int NH, double rho, double ds, int word, double t, double p, double len, int lane)
{
    return dubins_free_path_t<false>(bits, W, H, TY, x0, y0, h0, x1, y1, 0, NH, rho, ds, word, t, p, len, lane, 0, 1);
}

__device__ __forceinline__ bool dubins_free_warp(const uint32_t *bits, int W, int H, int TY, int x0, int y0, int h0, int x1, int y1,
                                                 int NH, double rho, double ds, const DubinsPath &w, int lane)
{
    return dubins_free_path(bits, W, H, TY, x0, y0, h0, x1, y1, NH, rho, ds, w.word, w.t, w.p, w.len, lane);
}

// dubins_free_warp on L heading-layer grids lstride words apart; h1 = the heading index of the target vertex
__device__ __forceinline__ bool dubins_free_warp_layers(const uint32_t *bits, size_t lstride, int L, int W, int H, int TY, int x0, int y0,
                                                        int h0, int x1, int y1, int h1, int NH, double rho, double ds, const DubinsPath &w,
                                                        int lane)
{
    return dubins_free_path_t<true>(bits, W, H, TY, x0, y0, h0, x1, y1, h1, NH, rho, ds, w.word, w.t, w.p, w.len, lane, lstride, L);
}

}  // namespace rrtk
