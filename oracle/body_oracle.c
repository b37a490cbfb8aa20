/*
 * CPU specification of the Dubins planners for a body with a heading -- TEST INFRASTRUCTURE ONLY (loaded by tests through
 * oracle/body_oracle.py; never linked into the product).  The device path it specifies is rrtk_plan2_batch_layers /
 * rrtk_dubins_collision_layers (csrc/plan_rewire.cu, csrc/dubins.cuh), tested against it bit for bit.
 *
 * It is one translation unit with oracle/rewire_oracle.c (included below, unchanged): the Dubins primitive, the sampled
 * points of a path, the cell rounding, the informed ellipse point and the candidate order are that file's, so only the grid a
 * test reads differs.  Build with -ffp-contract=off, as that file.
 *
 *   og        L heading-layer grids, W x H uint8 cells each (non-zero = blocked), layer-major
 *   layer     of an angle th:  l(th) = floor(th * ((double)L / DM_TWO_PI) + 0.5) mod L, non-negative
 *   free(a -> b), model DUBINS only: the points of the shortest path at arc length k * ds, k = 0 .. floor(len / ds), each with
 *             its own angle th, rounded to the nearest cell, test layer l(th) there (a point outside the grid blocks); b's own
 *             cell tests layer l(h_b * (DM_TWO_PI / NH))
 *   loop      the loop of rewire_oracle.c's header (nearest, choose parent, rewire, goal connection, informed sampling) with
 *             this free test.  With L = 1 every result equals orc2_plan / orc2_plan_informed on that grid (tested).
 */
#include "rewire_oracle.c"

static int body_layer(double th, int L)
{
    const double f = floor(th * ((double)L / DM_TWO_PI) + 0.5);
    const int l = (int)((long long)f % L);
    return l < 0 ? l + L : l;
}

/* 1 = the sampled path from (x0, y0, h0) to (x1, y1, h1) is free on the layer grids og */
static int free_layers(const uint8_t *og, int L, int W, int H, int x0, int y0, int h0, int x1, int y1, int h1, int NH, double rho,
                       double ds, const dubins_t *w)
{
    if (w->word < 0) return 0;
    const size_t cells = (size_t)W * H;
    const long long ns = (long long)floor(w->len / ds);
    for (long long k = 0; k <= ns; ++k) {
        double x, y, th;
        orc2_dubins_point(x0, y0, h0, NH, rho, w, (double)k * ds, &x, &y, &th);
        if (cell_blocked(og + (size_t)body_layer(th, L) * cells, W, H, x, y)) return 0;
    }
    return og[(size_t)body_layer((double)h1 * (DM_TWO_PI / (double)NH), L) * cells + (size_t)x1 * H + y1] == 0;
}

/* orc2_dubins_free_batch on L layer grids; q = (x0, y0, h0, x1, y1, h1) int32 */
void orc2_dubins_free_layers(const uint8_t *og, int L, int W, int H, const int32_t *q, long nq, int NH, double rho, double ds,
                             uint8_t *free_out)
{
    for (long i = 0; i < nq; ++i) {
        dubins_t w;
        const int32_t *e = q + 6 * i;
        orc2_dubins(e[3] - e[0], e[4] - e[1], e[2], e[5], NH, rho, &w);
        free_out[i] = (uint8_t)free_layers(og, L, W, H, e[0], e[1], e[2], e[3], e[4], e[5], NH, rho, ds, &w);
    }
}

typedef struct {
    int NH, W, H, L;
    double rho, ds;
    const uint8_t *og;
    int64_t *stats;
} body_world_t;

/* rewire_oracle.c's edge() for model DUBINS, with the layered free test */
static double edge_layers(const body_world_t *w, int ax, int ay, int ah, int bx, int by, int bh, int *is_free)
{
    w->stats[S2_LEN_EVALS]++;
    dubins_t d;
    orc2_dubins(bx - ax, by - ay, ah, bh, w->NH, w->rho, &d);
    if (is_free) { *is_free = free_layers(w->og, w->L, w->W, w->H, ax, ay, ah, bx, by, bh, w->NH, w->rho, w->ds, &d); w->stats[S2_CHECKS]++; }
    return d.len;
}

/* rewire_oracle.c's plan_core, model DUBINS, every edge through edge_layers */
static int plan_layers_core(int star, int rewire, const uint8_t *og, int L, int W, int H, int n, double r_rewire, int NH, double rho,
                            double ds, const int32_t *start, const int32_t *goal, const int32_t *samples, int32_t *pts, int32_t *head,
                            double *cost, double *elen, int32_t *parent, int64_t *stats, int informed, double r_goal, const double *rot,
                            const double *balls, double *ell_c)
{
    uint8_t *seen = calloc((size_t)W * H, 1);
    int32_t *ring = malloc(sizeof(int32_t) * (size_t)(n + 1));
    int32_t *first = malloc(sizeof(int32_t) * (size_t)(n + 1));
    int32_t *next = malloc(sizeof(int32_t) * (size_t)(n + 1));
    int32_t *queue = malloc(sizeof(int32_t) * (size_t)(n + 1));
    cand2_t *cands = malloc(sizeof(cand2_t) * (size_t)(n + 1));
    int32_t *vsoln = malloc(sizeof(int32_t) * (size_t)(n + 1));
    int nsol = 0;
    if (!seen || !ring || !first || !next || !queue || !cands || !vsoln) return -1;
    if (informed && ell_c) for (int i = 0; i <= n; ++i) ell_c[i] = NAN;
    for (int i = 0; i <= n; ++i) {
        pts[2 * i] = pts[2 * i + 1] = INT32_MIN; head[i] = -1;
        cost[i] = INFINITY; elen[i] = INFINITY; parent[i] = -1; first[i] = -1; next[i] = -1;
    }
    memset(stats, 0, sizeof(int64_t) * S2_COUNT);
    stats[S2_FIRST_SOL] = -1;
    body_world_t w = {NH, W, H, L, rho, ds, og, stats};
    pts[0] = start[0]; pts[1] = start[1]; head[0] = start[2]; cost[0] = 0.0; elen[0] = 0.0;
    int j = 1;
    const double rr = r_rewire * r_rewire;

    for (int i = 0; i < n; ++i) {
        int x = samples[3 * i], y = samples[3 * i + 1];
        const int h = samples[3 * i + 2];
        if (informed && nsol > 0) {
            if (!balls) break;                                       /* probe */
            int vb = vsoln[0];
            for (int k = 1; k < nsol; ++k) if (cost[vsoln[k]] < cost[vb]) vb = vsoln[k];
            const double c = cost[vb] + euclid(pts, vb, goal[0], goal[1]);
            ellipse_xy(W, H, rot, start, goal, c, balls + 2 * i, &x, &y);
            if (ell_c) ell_c[j] = c;
            stats[S2_ELL_ITERS]++;
        }
        int vnear = 0;
        int64_t bd = INT64_MAX;
        for (int v = 0; v < j; ++v) {
            int64_t dx = (int64_t)pts[2 * v] - x, dy = (int64_t)pts[2 * v + 1] - y;
            int64_t d = dx * dx + dy * dy;
            if (d < bd) { bd = d; vnear = v; }
        }
        int ok;
        const double l0 = edge_layers(&w, pts[2 * vnear], pts[2 * vnear + 1], head[vnear], x, y, h, &ok);
        if (!ok || seen[(size_t)x * H + y] || j == n) continue;
        seen[(size_t)x * H + y] = 1;
        const double c0 = cost[vnear] + l0;
        int vbest = vnear, m = 0;
        double cbest = c0, lbest = l0;
        if (star) {
            for (int v = 0; v < j; ++v) {
                int64_t dx = (int64_t)pts[2 * v] - x, dy = (int64_t)pts[2 * v + 1] - y;
                if ((double)(dx * dx + dy * dy) < rr) ring[m++] = v;
            }
            stats[S2_RING] += m;
            for (int k = 0; k < m; ++k) {
                const int vn = ring[k];
                if (vn == vnear) continue;
                if (!(cost[vn] + euclid(pts, vn, x, y) < c0)) continue;
                const double lc = edge_layers(&w, pts[2 * vn], pts[2 * vn + 1], head[vn], x, y, h, NULL);
                const double cn = cost[vn] + lc;
                if (cn < cbest) {
                    int fr;
                    edge_layers(&w, pts[2 * vn], pts[2 * vn + 1], head[vn], x, y, h, &fr);
                    if (fr) { vbest = vn; cbest = cn; lbest = lc; }
                }
            }
        }
        pts[2 * j] = x; pts[2 * j + 1] = y; head[j] = h; cost[j] = cbest; elen[j] = lbest; parent[j] = vbest;
        next[j] = first[vbest]; first[vbest] = j;
        if (star && rewire) {
            for (int k = 0; k < m; ++k) {
                const int vn = ring[k];
                if (vn == vbest) continue;
                if (!(cbest + euclid(pts, vn, x, y) < cost[vn])) continue;
                int fr;
                const double lr = edge_layers(&w, x, y, h, pts[2 * vn], pts[2 * vn + 1], head[vn], NULL);
                const double cm = cbest + lr;
                if (!(cm < cost[vn])) continue;
                edge_layers(&w, x, y, h, pts[2 * vn], pts[2 * vn + 1], head[vn], &fr);
                if (!fr) continue;
                const int op = parent[vn];
                if (first[op] == vn) first[op] = next[vn];
                else { int c = first[op]; while (next[c] != vn) c = next[c]; next[c] = next[vn]; }
                next[vn] = first[j]; first[j] = vn;
                parent[vn] = j; elen[vn] = lr; cost[vn] = cm;
                stats[S2_REWIRES]++;
                int qh = 0, qt = 0;
                queue[qt++] = vn;
                while (qh < qt) {
                    const int u = queue[qh++];
                    for (int c = first[u]; c >= 0; c = next[c]) { cost[c] = cost[u] + elen[c]; queue[qt++] = c; stats[S2_PROPAGATED]++; }
                }
            }
        }
        stats[S2_ACCEPTED]++;
        if (informed && euclid(pts, j, goal[0], goal[1]) < r_goal) {
            vsoln[nsol++] = j;
            if (nsol == 1) stats[S2_FIRST_SOL] = i;
        }
        ++j;
    }

    for (int v = 0; v < j; ++v) {
        cands[v].c = cost[v] + edge_layers(&w, pts[2 * v], pts[2 * v + 1], head[v], goal[0], goal[1], goal[2], NULL);
        cands[v].v = v;
    }
    qsort(cands, (size_t)j, sizeof(cand2_t), cand2_cmp);
    int vgoal = 0, found = 0;
    for (int k = 0; k < j; ++k) {
        const int v = cands[k].v;
        int fr;
        const double lg = edge_layers(&w, pts[2 * v], pts[2 * v + 1], head[v], goal[0], goal[1], goal[2], &fr);
        if (fr) {
            vgoal = j; found = 1;
            pts[2 * j] = goal[0]; pts[2 * j + 1] = goal[1]; head[j] = goal[2];
            cost[j] = cands[k].c; elen[j] = lg; parent[j] = v;
            break;
        }
    }
    stats[S2_J] = j; stats[S2_VGOAL] = vgoal; stats[S2_FOUND] = found;
    free(seen); free(ring); free(first); free(next); free(queue); free(cands); free(vsoln);
    return 0;
}

/* orc2_plan (model DUBINS) on L heading-layer grids */
int orc2_plan_layers(int star, int rewire, const uint8_t *og, int L, int W, int H, int n, double r_rewire, int NH, double rho, double ds,
                     const int32_t *start, const int32_t *goal, const int32_t *samples, int32_t *pts, int32_t *head, double *cost,
                     double *elen, int32_t *parent, int64_t *stats)
{
    return plan_layers_core(star, rewire, og, L, W, H, n, r_rewire, NH, rho, ds, start, goal, samples, pts, head, cost, elen, parent, stats,
                            0, 0.0, NULL, NULL, NULL);
}

/* orc2_plan_informed (model DUBINS) on L heading-layer grids */
int orc2_plan_informed_layers(int star, int rewire, const uint8_t *og, int L, int W, int H, int n, double r_rewire, int NH, double rho,
                              double ds, const int32_t *start, const int32_t *goal, const int32_t *samples, int32_t *pts, int32_t *head,
                              double *cost, double *elen, int32_t *parent, int64_t *stats, double r_goal, const double *rot,
                              const double *balls, double *ell_c)
{
    return plan_layers_core(star, rewire, og, L, W, H, n, r_rewire, NH, rho, ds, start, goal, samples, pts, head, cost, elen, parent, stats,
                            1, r_goal, rot, balls, ell_c);
}
